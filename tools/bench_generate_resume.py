"""Cost of resumable generation (fp16 tensor-core kernel) on the GPU, one JSON line.

  python tools/bench_generate_resume.py [--parent-root DIR] [--repeats 3] [--out FILE]

* one-shot per-step time (`generate` without a state, the k_ar_mma kernel and the whole call) at 256x16000 and
  1184x4000; with --parent-root (a built checkout of another revision) the two trees run in alternating worker
  processes, `--repeats` times each, so that their spread can be compared;
* the same 256x16000 generation in calls of 128, 1024 and 16000 samples through one state: per-step time including
  the per-call overhead (launches, noise transform, frame table);
* priming: a call whose samples are all forced (prefix = T) against an unprimed call of the same T.

Inputs are seeded; L2 is flushed (256 MiB write) before every timed pass.  The card's name and power limit are read in
the same run.  Needs a CUDA device: without one it fails."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(256, 16000), (1184, 4000)]
CHUNKS = [128, 1024, 16000]


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return {"name": name, "power_limit": limit}
    except Exception as e:                      # the measurement still stands; say why the card is unnamed
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def _teacher(srwn, synth, T):
    dil = synth.DEFAULT_DILATIONS
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=5, dilations=dil, skip_channels=128,
                                latent_channels=32, pool_stride=128)
    t.set_weights(synth.make_teacher_weights(dil))
    return t


def _timed(torch, flush, fn, passes):
    """[(call ms, k_ar_mma ms summed over the pass)] of `passes` runs of fn after one warm-up; fn returns kernel ms."""
    fn()
    out = []
    for _ in range(passes):
        flush.fill_(1)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        k = fn()
        b.record()
        torch.cuda.synchronize()
        out.append((a.elapsed_time(b), k))
    return out


def worker(root, passes, extra):
    sys.path.insert(0, root)
    import torch
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    res = {"one_shot": {}}
    for B, T in SHAPES:
        t = _teacher(srwn, synth, T)
        t._eng.set_profiling(True)
        enc = torch.from_numpy(synth.synthetic_encoding(B, T // 128, seed=4321)).cuda()
        u1, u2 = (torch.from_numpy(a).cuda() for a in synth.sampler_uniforms(B, T, seed=999))

        def one():
            t.generate(enc, u1=u1, u2=u2, precision="fp16")
            return t._eng.last_kernel_ms()[0]
        r = _timed(torch, flush, one, passes)
        res["one_shot"]["%dx%d" % (B, T)] = {"kernel_us_per_step": [1e3 * k / T for _, k in r],
                                             "call_us_per_step": [1e3 * c / T for c, _ in r]}
        if not extra or (B, T) != SHAPES[0]:
            continue
        chunked = {}
        for S in CHUNKS:
            state = t.generation_state(B, "fp16")

            def run_chunks():
                state.reset()
                k = 0.0
                for a in range(0, T, S):
                    b = min(a + S, T)
                    t.generate(enc[:, a // 128:b // 128], u1=u1[:, a:b], u2=u2[:, a:b], precision="fp16", state=state)
                    k += t._eng.last_kernel_ms()[0]
                return k
            r = _timed(torch, flush, run_chunks, passes)
            chunked[str(S)] = {"calls": -(-T // S), "kernel_us_per_step": [1e3 * k / T for _, k in r],
                               "call_us_per_step": [1e3 * c / T for c, _ in r]}
        res["chunked_256x16000"] = chunked
        Tp = 4096                                   # priming: every sample of the call forced, against free generation
        prefix = torch.from_numpy(synth.synthetic_audio(B, Tp, seed=1234)).cuda()
        e, v1, v2 = enc[:, :Tp // 128].contiguous(), u1[:, :Tp].contiguous(), u2[:, :Tp].contiguous()
        state = t.generation_state(B, "fp16")

        def primed():
            state.reset()
            t.generate(e, u1=v1, u2=v2, precision="fp16", state=state, prefix=prefix)
            return t._eng.last_kernel_ms()[0]

        def free():
            state.reset()
            t.generate(e, u1=v1, u2=v2, precision="fp16", state=state)
            return t._eng.last_kernel_ms()[0]
        rp, rf = _timed(torch, flush, primed, passes), _timed(torch, flush, free, passes)
        res["priming_256x4096"] = {"primed_kernel_us_per_sample": [1e3 * k / Tp for _, k in rp],
                                   "free_kernel_us_per_step": [1e3 * k / Tp for _, k in rf],
                                   "primed_call_us_per_sample": [1e3 * c / Tp for c, _ in rp],
                                   "free_call_us_per_step": [1e3 * c / Tp for c, _ in rf]}
    print("RESULT " + json.dumps(res), flush=True)


def _run_worker(root, passes, extra):
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", root, "--passes", str(passes)] + (["--extra"] if extra else [])
    out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout
    return json.loads([ln for ln in out.splitlines() if ln.startswith("RESULT ")][-1][7:])


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent-root", default=None, help="built checkout of the revision to compare with")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--passes", type=int, default=3, help="timed passes per worker and measurement")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--extra", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args.worker, args.passes, args.extra)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_generate_resume needs a CUDA device")
    line = {"tool": "bench_generate_resume", "card": _card(), "l2": "flushed before every timed pass (256 MiB write)",
            "passes_per_worker": args.passes, "runs": []}
    trees = [("this", ROOT)] + ([("parent", os.path.abspath(args.parent_root))] if args.parent_root else [])
    for i in range(args.repeats):                  # alternate the trees
        for name, root in trees:
            r = _run_worker(root, args.passes, extra=(name == "this" and i == 0))
            r["tree"], r["order"] = name, i
            line["runs"].append(r)
    summary = {}
    for name, _ in trees:
        for shape in ["%dx%d" % s for s in SHAPES]:
            ks = [min(r["one_shot"][shape]["kernel_us_per_step"]) for r in line["runs"] if r["tree"] == name]
            summary["%s_%s_kernel_us_per_step_min_of_runs" % (name, shape)] = ks
            summary["%s_%s_kernel_us_per_step_median" % (name, shape)] = statistics.median(ks)
    line["summary"] = summary
    line["time"] = time.strftime("%Y-%m-%dT%H:%M:%S")
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
