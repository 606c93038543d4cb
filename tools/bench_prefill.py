"""Parallel prefill of a generation state against sequential priming, on the GPU, one JSON line.

  python tools/bench_prefill.py [--passes 3] [--out FILE]

* B = 256, n in {128, 3200, 16000, 64000}, fp16 and fp32: `prefill(state, audio, enc)` against sequential priming
  (`generate(state=, prefix=audio)` with T = n, every sample forced through the step kernel), both from a reset state;
* B = 1184, n in {3200, 16000}: prefill alone.

Times are whole calls (CUDA events around the call; the Python layer's checks included), median and all passes.  Inputs
are seeded (the teacher.py configuration: 30 layers, sum(d) = 3069, pool stride 128); L2 is flushed (256 MiB write) before
every timed pass.  The card's name and power limit are read in the same run.  Needs a CUDA device: without one it fails."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = [128, 3200, 16000, 64000]


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return {"name": name, "power_limit": limit}
    except Exception as e:                      # the measurement still stands; say why the card is unnamed
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def _timed(torch, flush, fn, passes):
    """ms of `passes` runs of fn after one warm-up, L2 flushed before each."""
    fn()
    out = []
    for _ in range(passes):
        flush.fill_(1)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args(argv)
    sys.path.insert(0, ROOT)
    import torch
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("bench_prefill needs a CUDA device")
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    dil, P = synth.DEFAULT_DILATIONS, 128
    t = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=5, dilations=dil, skip_channels=128,
                                latent_channels=32, pool_stride=P)
    t.set_weights(synth.make_teacher_weights(dil))
    res = {"tool": "bench_prefill", "card": _card(), "config": {"layers": len(dil), "sum_d": sum(dil), "pool_stride": P},
           "passes": args.passes, "l2_flush": "256 MiB write before every timed pass", "B256": {}, "B1184": {}}

    def run(B, n, prec, sequential):
        enc = torch.from_numpy(synth.synthetic_encoding(B, n // P, seed=4321)).cuda()
        audio = torch.from_numpy(synth.synthetic_audio(B, n, seed=1234)).cuda()
        state = t.generation_state(B, prec)
        if sequential:
            u1, u2 = (torch.from_numpy(a).cuda() for a in synth.sampler_uniforms(B, n, seed=999))

            def fn():
                state.reset()
                t.generate(enc, u1=u1, u2=u2, precision=prec, state=state, prefix=audio)
        else:
            def fn():
                state.reset()
                t.prefill(state, audio, enc)
        ms = _timed(torch, flush, fn, args.passes)
        assert state.position() == n
        del state
        torch.cuda.empty_cache()
        return {"median_ms": statistics.median(ms), "ms": ms}

    for prec in ("fp16", "fp32"):
        for n in NS:
            pf, sq = run(256, n, prec, False), run(256, n, prec, True)
            res["B256"]["%s_n%d" % (prec, n)] = {"prefill": pf, "sequential": sq,
                                                 "speedup": sq["median_ms"] / pf["median_ms"]}
            print(prec, n, "prefill %.3f ms, sequential %.2f ms" % (pf["median_ms"], sq["median_ms"]), file=sys.stderr,
                  flush=True)
        for n in (3200, 16000):
            res["B1184"]["%s_n%d" % (prec, n)] = {"prefill": run(1184, n, prec, False)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
