"""Prints the per-phase clock stamps of the tensor-core training kernels (build with -DSRWN_TUNING:
`tools/exp_build.sh train_tc.cu tune -DSRWN_TUNING`).
usage: SRWN_LIB=tools/exp/libsrwn_tune.so python tools/tc_trace.py"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import sr_wavenet_b200 as srwn
from sr_wavenet_b200 import synth, _lib
B, T = 4, 64000
dil = synth.DEFAULT_DILATIONS
m = srwn.ParallelWaveNet(T, 0, dil, None, num_flows=4, skip_channels=128, latent_channels=32, pool_stride=128)
m.set_weights(synth.make_student_weights(dil, 4))
enc = torch.from_numpy(synth.synthetic_encoding(B, T // 128)).cuda()
z = torch.from_numpy(synth.logistic_noise(B, T)).cuda()
x = torch.from_numpy(synth.synthetic_audio(B, T)).cuda()
tl = torch.randn(B, T, 20, device="cuda") * 0.5
for _ in range(2):
    m.loss_and_grads(z, x, enc, teacher_logits=tl)
torch.cuda.synchronize()
lib = _lib.load()
out = (ctypes.c_longlong * 48)()
lib.srwn_debug_tc_trace.restype = ctypes.c_int
lib.srwn_debug_tc_trace(out)
names = ["fwd", "gate", "conv"]
for k in range(3):
    st = [out[k * 16 + i] for i in range(16)]
    n = max(i for i in range(16) if st[i]) if any(st) else 0
    print(names[k], "stamps (clk since slot 0):", [int(st[i] - st[0]) for i in range(n + 1)])
