"""Cost of chunked student synthesis (fp16 fused flow kernel) on the GPU, one JSON line.

  python tools/bench_student_stream.py [--passes 5] [--out FILE]

8 x 64000, 4 flows (the student.py configuration), noise injected: one `generate` call over the clip, then the same clip
in calls of S = 512, 2048, 4096 and 16000 samples through one synthesis state.  For each: the time of the whole clip,
the time per call and the useful samples/s (B * T over the clip's time), and the ratio to the one-call rate next to the
re-warm model (Heff + S) / S averaged over the calls (each call recomputes min(t0, H) = up to H = 3072 carried rows per
utterance and flow).  Inputs are seeded; L2 is flushed (256 MiB write) before every timed pass.  The card's name and
power limit are read in the same run.  Needs a CUDA device: without one it fails."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, T, P, H = 8, 64000, 128, 3072
CHUNKS = [512, 2048, 4096, 16000]


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit, clock = [s.strip() for s in out.split(",")[:3]]
        return {"name": name, "power_limit": limit, "max_sm_clock": clock}
    except Exception as e:                      # the measurement still stands; say why the card is unnamed
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def _timed(torch, flush, fn, passes):
    """ms of `passes` runs of fn after one warm-up, each after an L2 flush"""
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_student_stream needs a CUDA device")
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth
    torch.cuda.set_device(0)
    dil = synth.DEFAULT_DILATIONS
    s = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=None, num_flows=4, skip_channels=128,
                             latent_channels=32, pool_stride=P)
    s.set_weights(synth.make_student_weights(dil, num_flows=4))
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // P, seed=4321)).cuda()
    z = torch.from_numpy(synth.logistic_noise(B, T, seed=777)).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    line = {"tool": "bench_student_stream", "card": _card(), "shape": "%dx%d" % (B, T), "flows": 4, "precision": "fp16",
            "noise": "injected", "l2": "flushed before every timed pass (256 MiB write)", "passes": args.passes}

    def one():
        s.generate(None, z, enc, precision="fp16")
    ms1 = _timed(torch, flush, one, args.passes)
    one_ms = statistics.median(ms1)
    line["one_call"] = {"ms": ms1, "median_ms": one_ms, "samples_per_s": B * T / one_ms * 1e3}
    ref = s.generate(None, z, enc, precision="fp16")
    chunked = {}
    for S in CHUNKS:
        state = s.synthesis_state(B, "fp16")
        zs = [z[:, a:a + S].contiguous() for a in range(0, T, S)]
        es = [enc[:, a // P:(a + S) // P].contiguous() for a in range(0, T, S)]

        def run():
            state.reset()
            return [s.generate(None, zc, ec, state=state) for zc, ec in zip(zs, es)]
        same = torch.equal(torch.cat(run(), 1), ref)
        ms = _timed(torch, flush, run, args.passes)
        med = statistics.median(ms)
        sizes = [min(S, T - a) for a in range(0, T, S)]
        model = sum(min(a, H) + n for a, n in zip(range(0, T, S), sizes)) / T
        chunked[str(S)] = {"calls": len(sizes), "ms": ms, "median_ms": med, "ms_per_call": med / len(sizes),
                           "samples_per_s": B * T / med * 1e3, "cost_vs_one_call": med / one_ms,
                           "rewarm_model": model, "bit_identical_to_one_call": same}
    line["chunked"] = chunked
    line["time"] = time.strftime("%Y-%m-%dT%H:%M:%S")
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
