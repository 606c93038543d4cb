"""-m gpu: resumable autoregressive generation (srwn_generate_state_*, srwn_teacher_generate_resume).

With the same injected uniforms, generation split into calls through one state is bit for bit the one-shot call; priming
forces real audio through the queues (teacher forcing) and the generator continues from it as the reference's loop,
seeded with that audio, does.  Both kernels: fp32 (k_ar_generate) and fp16 (k_ar_mma); a teacher.py configuration (30
layers, powers of two) and one with dilations that are not powers of two (the t mod d branch); B = 1 and B = 13 (13 leaves
three padding rows in the last CTA of 8 utterances)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from conftest import f64
from primed_ar import naive_ar_loop_primed
from sr_wavenet_b200 import synth

pytestmark = pytest.mark.gpu

CFGS = {
    # dilations, latent channels, mixtures, pool stride, T
    "teacher": (synth.DEFAULT_DILATIONS, 32, 5, 128, 1024),
    "nonpow2": ([1, 2, 4, 8, 3, 5, 7], 8, 3, 64, 512),
}
PRECS = ["fp32", "fp16"]


@pytest.fixture(scope="module")
def srwn(lib):
    import sr_wavenet_b200
    assert torch.cuda.is_available()
    return sr_wavenet_b200


_models = {}


def _teacher(srwn, cfg):
    if cfg not in _models:
        dil, C, M, P, T = CFGS[cfg]
        t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=M, dilations=dil, skip_channels=128,
                                    latent_channels=C, pool_stride=P)
        w = synth.make_teacher_weights(dil, latent_channels=C, num_mixtures=M, seed=11)
        t.set_weights(w)
        _models[cfg] = (t, w)
    return _models[cfg]


def _inputs(cfg, B, T=None, seed=3):
    dil, C, M, P, T0 = CFGS[cfg]
    T = T or T0
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // P, channels=C, seed=seed)).cuda()
    u1, u2 = (torch.from_numpy(a).cuda() for a in synth.sampler_uniforms(B, T, num_mixtures=M, seed=seed + 1))
    return enc, u1, u2


def _chunked(t, enc, u1, u2, prec, sizes, P, prefix=None):
    """generate() over consecutive calls of the given sizes through one state; returns (x, logits, state)."""
    state = t.generation_state(enc.shape[0], prec)
    n = 0 if prefix is None else prefix.shape[1]
    xs, lgs, a = [], [], 0
    for s in sizes:
        b = a + s
        x, lg = t.generate(enc[:, a // P:b // P].contiguous(), u1=u1[:, a:b].contiguous(), u2=u2[:, a:b].contiguous(),
                           return_logits=True, precision=prec, state=state,
                           prefix=prefix[:, a:min(b, n)].contiguous() if a < n else None)
        xs.append(x)
        lgs.append(lg)
        a = b
    return torch.cat(xs, 1), torch.cat(lgs, 1), state


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("B", [1, 13])
def test_chunked_equals_one_shot(srwn, cfg, prec, B):
    """One resume over T after a reset, [P, 3P, rest] and all-P chunks: bit for bit the one-shot call."""
    t, _ = _teacher(srwn, cfg)
    _, _, _, P, T = CFGS[cfg]
    enc, u1, u2 = _inputs(cfg, B)
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True, precision=prec)
    for sizes in ([T], [P, 3 * P, T - 4 * P], [P] * (T // P)):
        xc, lgc, state = _chunked(t, enc, u1, u2, prec, sizes, P)
        assert torch.equal(xc, x), (sizes, (xc - x).abs().max().item())
        assert torch.equal(lgc, lg), sizes
        assert state.position() == T
    state.reset()
    assert state.position() == 0
    xr = t.generate(enc, u1=u1, u2=u2, precision=prec, state=state)       # a reset state starts from silence again
    assert torch.equal(xr, x)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("B", [1, 13])
def test_priming_is_teacher_forcing(srwn, cfg, prec, B):
    """x_out[:, :n] is the prefix; the logits over it are those of the teacher-forced fp32 pass on it; the continuation
    is the reference's loop seeded with the prefix (fp32), or reproduces its own logits under teacher forcing (fp16)."""
    t, w = _teacher(srwn, cfg)
    dil, C, M, P, T = CFGS[cfg]
    enc, u1, u2 = _inputs(cfg, B)
    n = 3 * P
    audio = torch.from_numpy(synth.synthetic_audio(B, T, seed=21)).cuda()
    prefix = audio[:, :n].contiguous()
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True, precision=prec, prefix=prefix)
    assert torch.equal(x[:, :n], prefix)
    tf = t.get_logits(x, enc, precision="fp32")
    err = (lg[:, :n] - tf[:, :n]).abs().max().item()
    if prec == "fp32":
        assert err <= 1e-4 * max(1.0, tf[:, :n].abs().max().item())
        rows = sorted({0, B - 1})                     # the first row and the last (padding rows follow it in its CTA)
        Tn = n + P                                    # the reference's O(T^2) loop over one more latent frame
        ref = naive_ar_loop_primed(f64(w), enc[rows, :Tn // P].double().cpu().numpy(), dil, P, M,
                                   u1[rows, :Tn].double().cpu().numpy(), u2[rows, :Tn].double().cpu().numpy(), Tn,
                                   prefix[rows].double().cpu().numpy())
        assert np.abs(x[rows, :Tn].cpu().numpy() - ref).max() <= 1e-4
    else:
        assert err <= 1e-2
        assert (tf - lg).abs().max().item() <= 1e-2
    # priming a state with n samples in one call, then generating in the next == one call primed with n samples
    x2, lg2, _ = _chunked(t, enc, u1, u2, prec, [n, T - n], P, prefix=prefix)
    assert torch.equal(x2, x) and torch.equal(lg2, lg)


@pytest.mark.parametrize("prec", PRECS)
def test_chunked_256x16000(srwn, prec):
    """The flagship shape in calls of 128, 4096 and 11776 samples, with a primed first frame: bit for bit one call."""
    cfg, B, T = "teacher", 256, 16000
    t, _ = _teacher(srwn, cfg)
    P = CFGS[cfg][3]
    enc, u1, u2 = _inputs(cfg, B, T=T)
    prefix = torch.from_numpy(synth.synthetic_audio(B, P, seed=5)).cuda()
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True, precision=prec, prefix=prefix)
    assert torch.equal(x[:, :P], prefix)
    xc, lgc, state = _chunked(t, enc, u1, u2, prec, [128, 4096, 11776], P, prefix=prefix)
    assert torch.equal(xc, x) and torch.equal(lgc, lg)
    assert state.position() == T


def test_refusals(srwn):
    from sr_wavenet_b200 import _lib
    lib = _lib.load()
    t, _ = _teacher(srwn, "teacher")
    other, _ = _teacher(srwn, "nonpow2")
    eng = t._eng
    B, T, P = 13, 256, 128
    enc, u1, u2 = _inputs("teacher", B, T=T)
    x = torch.empty(B, T, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    ws, wsn = eng.workspace(_lib.OP_TEACHER_GENERATE, B, T, _lib.FP16)

    def resume(state, b=B, prec=_lib.FP16, n=0, xp=None, tt=T, h=eng.h):
        return lib.srwn_teacher_generate_resume(h, state, enc.data_ptr(), u1.data_ptr(), u2.data_ptr(), xp, n,
                                                x.data_ptr(), None, b, tt, prec, ws, wsn, st)

    # the state holds the queues of the precision's kernel, x history and a header; its size does not depend on T
    n16, n32 = ctypes.c_size_t(), ctypes.c_size_t()
    _lib.check(lib.srwn_generate_state_bytes(eng.h, B, _lib.FP16, ctypes.byref(n16)))
    _lib.check(lib.srwn_generate_state_bytes(eng.h, B, _lib.FP32, ctypes.byref(n32)))
    sum_d = sum(synth.DEFAULT_DILATIONS)
    assert n16.value >= -(-B // 8) * sum_d * 512 and n16.value - -(-B // 8) * sum_d * 512 <= 1024
    assert n32.value >= B * sum_d * 32 * 4 and n32.value - B * sum_d * 32 * 4 <= 1024
    ws_small, ws_big = ctypes.c_size_t(), ctypes.c_size_t()
    _lib.check(lib.srwn_workspace_bytes(eng.h, _lib.OP_TEACHER_GENERATE, B, P, _lib.FP16, ctypes.byref(ws_small)))
    _lib.check(lib.srwn_workspace_bytes(eng.h, _lib.OP_TEACHER_GENERATE, B, 16000, _lib.FP16, ctypes.byref(ws_big)))
    assert ws_big.value > ws_small.value                  # the workspace grows with a call's T, the state does not
    assert lib.srwn_generate_state_bytes(eng.h, B, _lib.BF16, ctypes.byref(n16)) == _lib.ERR_UNSUPPORTED

    state = t.generation_state(B, "fp16")
    assert resume(state.data_ptr()) == _lib.OK
    assert resume(state.data_ptr(), b=B - 1) == _lib.ERR_INVALID                 # wrong B
    assert resume(state.data_ptr(), prec=_lib.FP32) == _lib.ERR_INVALID          # wrong precision
    assert resume(state.data_ptr(), h=other._eng.h) == _lib.ERR_INVALID          # reset on another handle
    assert resume(state.data_ptr(), n=T + 1, xp=x.data_ptr()) == _lib.ERR_INVALID   # n_prefix > T
    assert resume(state.data_ptr(), n=-1) == _lib.ERR_INVALID
    assert resume(state.data_ptr(), n=8, xp=None) == _lib.ERR_INVALID            # a prefix length without samples
    assert resume(state.data_ptr(), tt=T - 1) == _lib.ERR_INVALID                # T % P != 0
    assert resume(None) == _lib.ERR_INVALID                                      # null state
    assert resume(x.data_ptr() + 16) == _lib.ERR_INVALID                         # never reset (no allocation starts there)
    assert b"reset" in lib.srwn_last_error()
    assert state.position() == T                                                 # refused calls leave the state alone
    # the Python layer checks shapes before it calls
    with pytest.raises(ValueError):
        t.generate(enc, u1=u1, u2=u2, precision="fp16", prefix=torch.zeros(B, T + P, device="cuda"))
    with pytest.raises(ValueError):
        t.generate(enc[:1], u1=u1[:1], u2=u2[:1], precision="fp16", state=state)
    with pytest.raises(ValueError):
        t.generate(enc, u1=u1, u2=u2, precision="fp32", state=state)
    with pytest.raises(ValueError):
        t.generate(enc[:, :1], u1=u1, u2=u2, precision="fp16", state=state, num_samples=T)


def test_teacher_driver_prime_and_chunk(srwn, tmp_path):
    import teacher as drv
    from scipy.io import wavfile
    tdir, out = str(tmp_path / "teacher"), str(tmp_path / "out")
    t = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=5, dilations=drv.DILATIONS,
                                latent_channels=32, skip_channels=128, pool_stride=128)
    assert t.save(tdir, 7, force=True)
    common = ["--teacher", tdir, "--test-slow", "--num-samples", "1024", "--batch-size", "2", "--clips", "1",
              "--out-dir", out, "--precision", "fp32"]
    res = drv.main(common + ["--prime", "256", "--chunk", "512", "--check-naive", "320"])
    assert res["naive_max_abs_diff"] <= 1e-4             # the reference's loop seeded with the same 256 samples
    _, clip = wavfile.read(os.path.join(out, "test_wav_0.wav"))
    _, regen = wavfile.read(os.path.join(out, "regen_wav_0.wav"))
    assert regen.shape == (1024,) and np.array_equal(regen[:256], clip[:256]) and regen[-1] == 0.0
    drv.main(common + ["--prime", "256"])                 # one call, primed: the same audio
    _, one = wavfile.read(os.path.join(out, "regen_wav_0.wav"))
    assert np.array_equal(one, regen)
    with pytest.raises(SystemExit):
        drv.main(common + ["--prime", "100"])             # not a multiple of --pool-stride
