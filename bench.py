#!/usr/bin/env python
"""Benchmark of the SR-WaveNet hot path on B200 (contract: see the task statement / DESIGN.md).

Workload (BASELINE.json configs[1]): teacher WaveNet teacher-forced log-likelihood, batch
32 x 64000 samples per GPU (weak scaling: every rank scores its own 32 utterances, no data-path
collective).  One step = one scoring pass over one batch.  `value` is timed with CUDA events on
inputs already resident in HBM; `e2e` goes through the Python API with pinned host buffers
(H2D of audio + encoding and D2H of the log-likelihood inside the timed region).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload ...] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, so that two builds run with
the same arguments, and therefore the same seeded inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_SAMPLE_TEACHER = 468576      # SURVEY.md 8(d): 30*14336 + 37888 + 128 + 480
FLOP_PER_SAMPLE_STUDENT = 740224      # 4*184576 + 1920
BYTES_PER_SAMPLE_LAYER_F32 = 1280     # fp32 per-layer kernel: h read+write (2*128 B) + skip RMW (2*512 B)
BYTES_PER_SAMPLE_AR = 7684            # SURVEY.md 8(d): fp32 queue pop+push (2*30*32*4 B) + 4 B sample
BYTES_PER_SAMPLE_AR_F16 = 3844        # same with 16-bit queue state (2*30*32*2 B) + 4 B sample
# distillation backward (fp32, layer at a time): per (sample, layer, flow) the gate kernel reads x_l and g and writes
# da (3 x 128 B), the conv kernel reads x_l, g, da and writes dx (4 x 128 B): 896 B; x 30 layers x 4 flows
BYTES_PER_SAMPLE_BWD = 4 * 30 * 896
BYTES_PER_SAMPLE_ENC_LAYER = 512      # encoder layer launch: 16-bit image of relu(h), 128 channels, read + write
FLOP_PER_SAMPLE_ENC = 2949632         # GEMMs the encoder executes: 33280 (nc_conv) + 30*65536 (K=2 convs) + 29*32768 (1x1 residuals)
METRIC = "audio samples/sec"
UNIT = "samples/s"
DUMP_LIMIT_BYTES = 64 * 10 ** 6       # all files of one --dump-outputs, headers included


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), tf=float(d["bf16_tflops"]),
                    tf_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, source="fallback")   # B200_PROFILING.md


class ClockSampler(object):
    """Samples the SM clock and the clock-event (throttle) reasons of this rank's GPU while the timed region runs:
    NVML in-process every 2 ms (the timed region of the short workloads lasts ~15 ms, less than one nvidia-smi start-up);
    `nvidia-smi -lms` is the fallback when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NVML_REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self._stop = None, None, threading.Event()
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        try:
            mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            self.rows.append((mhz, int(get(self.handle))))
        except Exception:
            pass

    def _loop_nvml(self):
        while not self._stop.is_set():
            self._sample_nvml()
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._loop_nvml, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.thread.join(timeout=1.0)
            sm = sorted(r[0] for r in self.rows)
            mask = 0
            for r in self.rows:
                mask |= r[1]
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max,
                    "reasons": sorted(name for bit, name in self.NVML_REASONS if mask & bit), "samples": len(sm),
                    "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def cpu_port_samples_per_s(B, T, repeats, warm=1):
    """Times oracle/torch_cpu.py (the stand-in for the reference's TF CPU path) on this host."""
    import torch
    from sr_wavenet_b200 import synth
    from oracle.torch_cpu import TeacherCPU
    torch.set_num_threads(os.cpu_count() or 1)
    dil = synth.DEFAULT_DILATIONS
    cpu = TeacherCPU(synth.make_teacher_weights(dil), dil, 128, 5)
    x, enc = synth.synthetic_audio(B, T), synth.synthetic_encoding(B, T // 128)
    for _ in range(warm):
        cpu.nll(x, enc)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        cpu.nll(x, enc)
        times.append(time.perf_counter() - t0)
    return B * T / min(times), B * T / (sum(times) / len(times)), torch.get_num_threads(), times


def quick_measure(srwn, synth, shard, workload, B, T, rank, steps=3, warmup=3):
    """A short device-timed run of another BASELINE configuration inside the same job (inputs resident in HBM, CUDA events
    per step, MAX over ranks, whole-job samples/s).  Used for the `also` block: the strong split of configs[1] / [3] and
    the distillation step of configs[4], whose all-reduce is bracketed with its own CUDA events."""
    import torch
    dil, P = synth.DEFAULT_DILATIONS, 128
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // P, seed=4321 + rank)).cuda()
    extra = {}
    if workload in ("student", "distill"):
        teacher = None
        if workload == "distill":
            teacher = srwn.WaveNetAutoEncoder(T, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=P)
            teacher.set_weights(synth.make_teacher_weights(dil))
            truth = torch.from_numpy(synth.synthetic_audio(B, T, seed=1234 + rank * B)).cuda()
        model = srwn.ParallelWaveNet(T, 0, dil, teacher, num_flows=4, skip_channels=128, latent_channels=32, pool_stride=P,
                                     alpha=0.25, beta=1.0, gamma=1.0, learning_rate=1e-4)
        model.set_weights(synth.make_student_weights(dil, 4))
        z = torch.from_numpy(synth.logistic_noise(B, T, seed=777 + rank)).cuda()
        if workload == "distill":
            if shard.is_distributed():
                model._coll_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            step = lambda: model.train_fast(None, z, truth, enc)
        else:
            step = lambda: model.generate(None, z, enc, precision="fp16")
    else:
        model = srwn.WaveNetAutoEncoder(T, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=P)
        model.set_weights(synth.make_teacher_weights(dil))
        if workload == "teacher_nll":
            x = torch.from_numpy(synth.synthetic_audio(B, T, seed=1234 + rank * B)).cuda()
            step = lambda: model.nll(x, enc, precision="fp16")
        else:
            u1, u2 = (torch.from_numpy(a).cuda() for a in synth.sampler_uniforms(B, T, seed=999 + rank))
            step = lambda: model.generate(enc, u1=u1, u2=u2, precision="fp16")
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    shard.barrier()
    ms, coll = [], []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
        if getattr(model, "_coll_events", None):
            coll.append(model._coll_events[0].elapsed_time(model._coll_events[1]))
    shard.barrier()
    total_max, coll_max = shard.reduce_scalars([sum(ms), sum(coll)], "max")
    units, = shard.reduce_scalars([float(B * T * steps)], "sum")
    out = {"batch_per_gpu": B, "samples_per_utterance": T, "ms_per_step": total_max / steps, "value": units / (total_max * 1e-3)}
    if coll:
        out["allreduce_us"] = 1e3 * coll_max / steps
    if workload in ("teacher_nll", "student"):
        out["partition_teams_x_ctas"] = list(model._eng.last_partition())
    del model
    torch.cuda.empty_cache()
    return out


def run_reference(args, rank, world):
    """--impl reference: the CPU port of the reference path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    B, T = 2, 64000
    best, mean, cores, times = cpu_port_samples_per_s(B, T, args.steps, warm=max(1, args.warmup))
    ms = 1e3 * sum(times) / len(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": mean, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "teacher WaveNet teacher-forced log-likelihood (BASELINE.json configs[1])",
                   "sample": "each step scores %d x %d samples on the host" % (B, T),
                   "note": "TensorFlow 1.x (the reference runtime) is not installable here; this is the "
                           "PyTorch-CPU fp32 port oracle/torch_cpu.py of the same graph"},
        "cpu_baseline": {"value": mean, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d steps of %d x %d samples, mean" % (args.steps, B, T)},
        "e2e": {"value": mean, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes name -> array (NumPy or torch) as out_dir/<name>.npy: float64 stays float64, everything else becomes
    float32.  Each array gets an equal share of ``limit``; one larger than its share is replaced by a sample of its
    flattened elements, drawn with a fixed seed and kept in index order, so equal shapes give the same sample."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = limit // len(arrays) - 4096            # room for the .npy header
    for name, a in arrays.items():
        if hasattr(a, "detach"):
            a = a.detach().cpu().numpy()
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the workload (the `also` block times its extra configurations with a fixed "
                         "3 steps, 2 for generation)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="teacher_nll", choices=["teacher_nll", "student", "generate", "distill", "encode"])
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "fp16"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the BASELINE config)")
    ap.add_argument("--length", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the extra configurations of the `also` block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth, shard

    rank, local_rank, world = shard.init_from_env()
    torch.cuda.set_device(local_rank)
    peaks = load_peaks()
    dil = synth.DEFAULT_DILATIONS
    P = 128

    defaults = {"teacher_nll": (32, 64000), "student": (64 // max(world, 1) if world > 1 else 8, 64000),
                "generate": (256, 16000), "distill": (4, 64000), "encode": (32, 64000)}
    B, T = defaults[args.workload]
    if args.workload == "student":
        B = 8          # configs[2]: 64 x 64000 over 8 GPUs = 8 per GPU (weak scaling unit)
    B = args.batch or B
    T = args.length or T

    # synthetic inputs, seeded per global utterance index so ranks see different audio
    g0 = rank * B
    enc_h = synth.synthetic_encoding(B, T // P, seed=4321 + rank)
    truth_h = None
    if args.workload in ("student", "distill"):
        teacher = None
        if args.workload == "distill":      # configs[4]: the teacher scores the REAL audio (model.py:326-334)
            teacher = srwn.WaveNetAutoEncoder(T, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=P)
            teacher.set_weights(synth.make_teacher_weights(dil))
            truth_h = synth.synthetic_audio(B, T, seed=1234 + g0)
        model = srwn.ParallelWaveNet(T, 0, dil, teacher, num_flows=4, skip_channels=128, latent_channels=32,
                                     pool_stride=P, alpha=0.25, beta=1.0, gamma=1.0, learning_rate=1e-4)   # student.py:30-33
        model.set_weights(synth.make_student_weights(dil, 4))
        x_h = synth.logistic_noise(B, T, seed=777 + rank)
        flop_per_sample = FLOP_PER_SAMPLE_STUDENT / 4.0     # the dominant kernel is one flow (one launch per flow)
    else:
        model = srwn.WaveNetAutoEncoder(T, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=P)
        w = synth.make_teacher_weights(dil)
        if args.workload == "encode":
            w.update(synth.make_encoder_weights(len(dil)))
        model.set_weights(w)
        x_h = synth.synthetic_audio(B, T, seed=1234 + g0)
        flop_per_sample = FLOP_PER_SAMPLE_TEACHER
    prec = args.precision
    if prec == "auto" and args.workload != "generate":
        prec = "fp16" if "fp16" in model.available_precisions() else "fp32"
    if args.workload == "distill":
        prec = "fp32"                           # student forward/backward run in fp32; the teacher uses its fp16 path
    if args.workload == "generate":
        if prec in ("auto", "fp16"):     # tensor-core generation kernel (fp16 operands and queue state)
            prec = "fp16"
        u1_h, u2_h = synth.sampler_uniforms(B, T, seed=999 + rank)

    x_d, enc_d = torch.from_numpy(x_h).cuda(), torch.from_numpy(enc_h).cuda()
    x_p, enc_p = torch.from_numpy(x_h).pin_memory(), torch.from_numpy(enc_h).pin_memory()
    if args.workload == "generate":
        u1_d, u2_d = torch.from_numpy(u1_h).cuda(), torch.from_numpy(u2_h).cuda()
        u1_p, u2_p = torch.from_numpy(u1_h).pin_memory(), torch.from_numpy(u2_h).pin_memory()

    if truth_h is not None:
        truth_d, truth_p = torch.from_numpy(truth_h).cuda(), torch.from_numpy(truth_h).pin_memory()

    def step_device():
        if args.workload == "distill":
            return model.train_fast(None, x_d, truth_d, enc_d)
        if args.workload == "teacher_nll":
            return model.nll(x_d, enc_d, precision=prec)
        if args.workload == "student":
            return model.generate(None, x_d, enc_d, precision=prec)
        if args.workload == "encode":
            return model.encode(x_d, precision=prec)
        return model.generate(enc_d, u1=u1_d, u2=u2_d, precision=prec)

    def step_e2e():
        if args.workload == "encode":
            return model.encode(x_p, precision=prec)                # ndarray on the host
        if args.workload == "distill":
            return model.train_fast(None, x_p, truth_p, enc_p)      # (loss, power_loss) floats on the host
        if args.workload == "teacher_nll":
            return model.nll(x_p, enc_p, precision=prec)            # float on the host
        if args.workload == "student":
            return model.generate(None, x_p, enc_p, precision=prec)  # ndarray on the host
        return model.generate(enc_p, u1=u1_p, u2=u2_p, precision=prec)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    model._eng.set_profiling(True)
    if args.workload == "encode":
        model._enc_eng.set_profiling(True)
    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    shard.barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = srwn._lib.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kern_ms, kern_launches, kern_name = [], 0, ""
    torch.cuda.synchronize()
    for a, b in ev:
        flush.fill_(1)                      # L2 flush between timed iterations (not timed)
        a.record()
        out = step_device()
        b.record()
        if args.workload == "encode":
            km, kern_launches, kern_name = model._enc_eng.last_ms(), len(dil) + 1, "enc::k_enc_layer"
        else:
            km, kern_launches, kern_name = model._eng.last_kernel_ms()
        kern_ms.append(km)
    torch.cuda.synchronize()
    if prec != "fp32" and args.workload not in ("generate", "distill", "encode"):     # a fused launch that aborted on the device is not a measurement
        model._eng.check_async(srwn._lib.OP_TEACHER_NLL if args.workload == "teacher_nll" else srwn._lib.OP_STUDENT_FORWARD,
                               B, T, srwn._lib.PRECISIONS[prec])
    launches = srwn._lib.launch_count() - launches0
    partition = list(model._eng.last_partition()) if args.workload in ("teacher_nll", "student") and prec == "fp16" else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    if args.dump_outputs and rank == 0:
        names = {"teacher_nll": ("nll",), "student": ("out",), "generate": ("audio",), "encode": ("encoding",),
                 "distill": ("loss", "power_loss")}[args.workload]
        dump_outputs(args.dump_outputs, dict(zip(names, out if isinstance(out, tuple) else (out,))))
    del out
    shard.barrier()

    # end to end through the public API with pinned host buffers
    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    shard.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_serial_s = None
    if args.workload == "teacher_nll":
        # the scoring service's call: WaveNetAutoEncoder.nll_stream takes the batches as they come and uploads batch i+1 on a
        # copy stream while batch i is scored; every step still pays its own H2D copy and its own D2H read of the result
        e2e_serial_s = e2e_s
        list(model.nll_stream([(x_p, enc_p)] * 3, precision=prec))
        torch.cuda.synchronize()
        shard.barrier()
        t0 = time.perf_counter()
        vals = list(model.nll_stream(((x_p, enc_p) for _ in range(args.steps)), precision=prec))
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        assert len(vals) == args.steps and all(np.isfinite(v) for v in vals)
    e2e_dev_noise_s = None
    if args.workload == "student":      # the same call with the logistic noise drawn inside the flow kernel: only the encoding goes up
        for _ in range(2):
            model.generate(None, None, enc_p, precision=prec)
        torch.cuda.synchronize()
        shard.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            model.generate(None, None, enc_p, precision=prec)
        torch.cuda.synchronize()
        e2e_dev_noise_s = time.perf_counter() - t0
    clocks = sampler.stop()

    total_ms_max, e2e_s_max, e2e_dn_max, e2e_serial_max = shard.reduce_scalars([total_ms, e2e_s, e2e_dev_noise_s or 0.0, e2e_serial_s or 0.0], "max")
    units, = shard.reduce_scalars([float(B * T * args.steps)], "sum")
    value = units / (total_ms_max * 1e-3)
    e2e_value = units / e2e_s_max
    h2d = x_h.nbytes + enc_h.nbytes + (u1_h.nbytes + u2_h.nbytes if args.workload == "generate" else 0) + \
        (truth_h.nbytes if truth_h is not None else 0)
    d2h = 4 if args.workload == "teacher_nll" else 16 if args.workload == "distill" else \
        B * (T // P) * 32 * 4 if args.workload == "encode" else B * T * 4
    if args.workload == "encode":
        h2d = x_h.nbytes

    # roofline of the dominant kernel, from this run's CUDA-event bracket around its launches
    k_ms = sum(kern_ms) / len(kern_ms) / max(kern_launches, 1)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get("%s/%s" % (args.workload, prec))
    if args.workload == "distill":
        ach = BYTES_PER_SAMPLE_BWD * B * T / (k_ms * kern_launches * 1e-3) / 1e9     # the bracket spans the whole backward
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s"}
    elif args.workload == "encode":
        # one launch per layer moves the 16-bit image of relu(h): 256 B read + 256 B written per sample (the front layer
        # reads the audio, the last layer writes only pooled sums); the skip path is folded away (DESIGN.md 4.7)
        ach = BYTES_PER_SAMPLE_ENC_LAYER * B * T / (k_ms * 1e-3) / 1e9 * (len(dil) / (len(dil) + 1.0))
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
                "tensor_tflops": FLOP_PER_SAMPLE_ENC * B * T / (k_ms * kern_launches * 1e-3) / 1e12}
    elif args.workload == "generate":
        # queue pop + push of 32 channels per layer + the sample: 7684 B with fp32 state, 3844 B with fp16 state
        ach = (BYTES_PER_SAMPLE_AR if prec == "fp32" else BYTES_PER_SAMPLE_AR_F16) * B * T / (k_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s"}
    elif prec == "fp16":
        ach = flop_per_sample * B * T / (k_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": peaks["tf"], "unit": "TFLOP/s"}
    else:
        ach = BYTES_PER_SAMPLE_LAYER_F32 * B * T / (k_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s"}
    roof.update(frac=roof["achieved"] / roof["peak"], traffic=traffic, kernel=kern_name,
                launches_per_step=kern_launches, kernel_ms=k_ms, peak_source=peaks["source"])

    # the other BASELINE configurations in the same job (device-timed, short): the STRONG split of configs[1] (32 / N
    # utterances per GPU) and configs[3] (256 / N), the per-GPU share of configs[2], and the configs[4] distillation step
    # (4 x 64000 per GPU) with the NCCL all-reduce of its [gradient | loss | power] bucket timed separately
    also = None
    if args.workload == "teacher_nll" and not args.no_also and not (args.batch or args.length):
        del model
        torch.cuda.empty_cache()
        also = {
            "teacher_nll_strong_32_total": quick_measure(srwn, synth, shard, "teacher_nll", max(1, 32 // world), 64000, rank),
            "generate_strong_256_total": quick_measure(srwn, synth, shard, "generate", max(1, 256 // world), 16000, rank, steps=2, warmup=1),
            "student_8_per_gpu": quick_measure(srwn, synth, shard, "student", 8, 64000, rank),
            "distill_4_per_gpu": quick_measure(srwn, synth, shard, "distill", 4, 64000, rank),
        }

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "teacher_nll":
        best, mean, cores, times = cpu_port_samples_per_s(4, 64000, repeats=3)
        cpu_baseline = {"value": best, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "teacher log-likelihood on 4 x 64000 samples, best of 3 "
                                  "(oracle/torch_cpu.py; TF 1.x not installable)"}

    if rank == 0:
        names = {"teacher_nll": "teacher WaveNet teacher-forced log-likelihood (BASELINE.json configs[1])",
                 "student": "student IAF parallel synthesis, 4 flows (BASELINE.json configs[2])",
                 "generate": "teacher autoregressive fast generation, dilation queues (BASELINE.json configs[3])",
                 "encode": "teacher encoder, 31 non-causal 128-channel layers + pooled latent (SURVEY.md 8(f)-1)",
                 "distill": "student distillation training step: teacher scores real audio, KL + power loss, "
                            "all-reduce + clip + Adam (BASELINE.json configs[4])"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {"fp16": "f16", "fp32": "f32"}[prec],
            "data": "synthetic",
            "config": {"workload": names[args.workload], "batch_per_gpu": B, "global_batch": B * world,
                       "samples_per_utterance": T, "layers": len(dil), "parallelism": "batch-sharded x%d" % world,
                       "l2": "flushed between timed iterations (256 MiB write)", "precision_path": prec,
                       "fused_partition_teams_x_ctas": partition},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "e2e_api": "WaveNetAutoEncoder.nll_stream (upload of batch i+1 overlapped with the scoring of batch i, 2 slots)"
            if e2e_serial_s else "one synchronous call per step",
            "e2e_serial": None if not e2e_serial_s else
            {"value": units / e2e_serial_max, "unit": UNIT, "api": "WaveNetAutoEncoder.nll, one synchronous call per step"},
            "e2e_device_noise": None if not e2e_dev_noise_s else
            {"value": units / e2e_dn_max, "unit": UNIT, "h2d_bytes_per_step": int(enc_h.nbytes), "d2h_bytes_per_step": int(d2h),
             "note": "generate(sess, None, encoding): logistic noise drawn inside the flow kernel (Philox), no noise upload"},
            "gpu_launches": int(launches),
            "roofline": roof,
            "cpu_baseline": cpu_baseline,
            "also": also,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
