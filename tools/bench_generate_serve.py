"""Continuous batching against static batching (fp16 tensor-core generation) on the GPU, one JSON line.

  python tools/bench_generate_serve.py [--requests 4096] [--slots 1184] [--out FILE]

* workload: `--requests` requests with lengths uniform in [16000, 64000] samples, rounded to pool_stride (128), no prime,
  uniforms drawn on the device;
* static batching: the requests in arrival order in batches of `--slots`, each batch one `generate` call that runs to
  its longest request;
* continuous batching: `WaveNetAutoEncoder.generate_requests` with `--slots` slots, in calls of 1024 and 4096 samples;
* rates are useful samples per second (the samples returned to requests) over the wall time of the whole workload;
* splice cost: microseconds per `srwn_generate_state_splice` call moving 1, 64 and `--slots` rows between two states of
  `--slots` utterances at different positions, both precisions: CUDA events around `--splice-reps` back-to-back calls
  (host enqueue included where it is longer than the kernel), three passes.

Inputs are seeded; L2 is flushed (256 MiB write) before every timed pass.  The card's name and power limit are read in
the same run.  Needs a CUDA device: without one it fails."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_generate_resume import _card, _teacher  # noqa: E402

P = 128
CHUNKS = [1024, 4096]


def _workload(torch, synth, n, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    lengths = (np.rint(rng.uniform(16000, 64000, size=n) / P) * P).astype(np.int64)
    frames = lengths // P
    enc = torch.from_numpy(synth.synthetic_encoding(1, int(frames.sum()), seed=seed + 1)[0]).cuda()
    offs = np.concatenate([[0], np.cumsum(frames)])
    return [enc[offs[i]:offs[i + 1]] for i in range(n)], lengths


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--requests", type=int, default=4096)
    ap.add_argument("--slots", type=int, default=1184)
    ap.add_argument("--splice-reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_generate_serve needs a CUDA device")
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    t = _teacher(srwn, synth, 1024)
    S = args.slots
    encs, lengths = _workload(torch, synth, args.requests, seed=2024)
    useful = int(lengths.sum())
    line = {"tool": "bench_generate_serve", "card": _card(), "l2": "flushed before every timed pass (256 MiB write)",
            "precision": "fp16", "requests": args.requests, "slots": S, "lengths": "uniform in [16000, 64000], rounded to 128",
            "useful_samples": useful}

    def wall(fn):
        flush.fill_(1)
        torch.cuda.synchronize()
        a = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - a

    # warm-up of every shape family the timed passes use
    warm = [e[:8] for e in encs[:2 * S // 8]]
    for C in CHUNKS:
        for _ in t.generate_requests(warm, slots=S, chunk=C):
            pass
    t.generate(encs[0][None, :8].contiguous().repeat(S, 1, 1), precision="fp16")

    def static():
        for a in range(0, args.requests, S):
            batch = encs[a:a + S]
            F = max(e.shape[0] for e in batch)
            e = torch.zeros(len(batch), F, encs[0].shape[1], device="cuda")
            for i, x in enumerate(batch):
                e[i, :x.shape[0]] = x
            t.generate(e, precision="fp16")
    s_static = wall(static)
    res = {"static": {"seconds": s_static, "useful_samples_per_s": useful / s_static,
                      "steps": int(sum(max(lengths[a:a + S]) for a in range(0, args.requests, S)))}}
    for C in CHUNKS:
        got = [0]

        def serve():
            for i, x in t.generate_requests(encs, slots=S, chunk=C):
                got[0] += x.shape[0]
        s = wall(serve)
        assert got[0] == useful, (got[0], useful)
        res["continuous_chunk%d" % C] = {"seconds": s, "useful_samples_per_s": useful / s,
                                         "speedup_over_static": s_static / s}
    line["rates"] = res

    splice = {}
    for prec in ("fp32", "fp16"):
        dst, src = t.generation_state(S, prec), t.generation_state(S, prec)
        e = encs[0][None, :1].contiguous().repeat(S, 1, 1)
        t.generate(e, precision=prec, state=src)                    # src at t0 = 128, dst at 0: the queues rotate
        for n in (1, 64, S):
            rows = list(range(n))
            dst.splice(rows, src)
            us = []
            for _ in range(3):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.splice_reps):
                    dst.splice(rows, src)
                b.record()
                torch.cuda.synchronize()
                us.append(1e3 * a.elapsed_time(b) / args.splice_reps)
            splice["%s_rows%d" % (prec, n)] = {"us_per_call": us, "median": statistics.median(us)}
    line["splice_us_per_call"] = splice
    line["time"] = time.strftime("%Y-%m-%dT%H:%M:%S")
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
