"""Prints the clock64 timeline of CTA 0 for a few layers of one chunk (SRWN_TRACE=<chunk index>).
Needs the -DSRWN_TUNING build of the fused kernel: tools/exp_build.sh, then SRWN_LIB=tools/exp/libsrwn_trace.so."""
import sys, os, ctypes
os.environ.setdefault("SRWN_TRACE", "20")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import sr_wavenet_b200 as srwn
from sr_wavenet_b200 import synth, _lib
B, T = 32, 64000
dil = synth.DEFAULT_DILATIONS
m = srwn.WaveNetAutoEncoder(T, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=128)
m.set_weights(synth.make_teacher_weights(dil))
x = torch.from_numpy(synth.synthetic_audio(B, T)).cuda(); enc = torch.from_numpy(synth.synthetic_encoding(B, T // 128)).cuda()
for _ in range(2):
    m.nll(x, enc, precision="fp16")
eng = m._eng
ws, wsn = eng.workspace(_lib.OP_TEACHER_NLL, B, T, _lib.FP16)
n = 7 * 40 * 12
out = (ctypes.c_longlong * n)()
lib = _lib.load()
lib.srwn_debug_read_trace.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int32]
_lib.check(lib.srwn_debug_read_trace(eng.h, B, T, ws, wsn, out, n))
tr = np.array(out[:], dtype=np.int64).reshape(7, 40, 12)
L0, L1 = int(sys.argv[1]) if len(sys.argv) > 1 else 10, int(sys.argv[2]) if len(sys.argv) > 2 else 14
names_e = ["top", "sync1", "G1iss", "D1rdy", "ld1", "math1", "sync2", "G2iss", "D2rdy", "math2", "waits", "arriveH"]
names_l = ["start", "Wempty ok", "G1 ok", "halo arrive", "cp issued", "cp landed"]
base = tr[0, L0, 0]
for l in range(L0, L1):
    print("layer %d (d=%d)" % (l, dil[l]))
    for t in range(3):
        print("  tile%d : " % t + " ".join("%s=%d" % (nm, tr[t, l, i] - base) for i, nm in enumerate(names_e)))
    print("  load : " + " ".join("%s=%d" % (nm, tr[6, l, i] - base) for i, nm in enumerate(names_l)))
per = (tr[0, 29, 0] - tr[0, 1, 0]) / 28.0
print("avg clocks per layer (tile 0):", per)
