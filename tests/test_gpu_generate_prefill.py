"""-m gpu: parallel prefill of a generation state (srwn_generate_state_prefill, WaveNetAutoEncoder.prefill).

The state after a prefill of n samples is, byte for byte, the state a resume call of T = n with those samples as x_prefix
leaves (the step kernel teacher-forcing them one by one), for fp32 (k_ar_generate) and fp16 (k_ar_mma), from a fresh
state and from one that has already generated samples.  The fp16 prefill fills all 16 rows of each mma.sync with time
steps where the step kernel uses 8; these equalities are what checks that a row's result depends on that row alone."""
import ctypes
import os

import numpy as np
import pytest
import torch

from sr_wavenet_b200 import synth

pytestmark = pytest.mark.gpu

CFGS = {
    # dilations, latent channels, mixtures, pool stride, n past the window (sum(d) + 2)
    "teacher": (synth.DEFAULT_DILATIONS, 32, 5, 128, 3328),
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
        dil, C, M, P, _ = CFGS[cfg]
        t = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=M, dilations=dil, skip_channels=128,
                                    latent_channels=C, pool_stride=P)
        t.set_weights(synth.make_teacher_weights(dil, latent_channels=C, num_mixtures=M, seed=11))
        _models[cfg] = t
    return _models[cfg]


def _inputs(cfg, B, T, seed=3):
    dil, C, M, P, _ = CFGS[cfg]
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // P, channels=C, seed=seed)).cuda()
    u1, u2 = (torch.from_numpy(a).cuda() for a in synth.sampler_uniforms(B, T, num_mixtures=M, seed=seed + 1))
    audio = torch.from_numpy(synth.synthetic_audio(B, T, seed=seed + 2)).cuda()
    return enc, u1, u2, audio


def _pair(t, cfg, B, prec, lead):
    """Two states that have generated the same `lead` samples (none: fresh)."""
    P = CFGS[cfg][3]
    a, b = t.generation_state(B, prec), t.generation_state(B, prec)
    if lead:
        enc, u1, u2, _ = _inputs(cfg, B, lead, seed=17)
        for s in (a, b):
            t.generate(enc, u1=u1, u2=u2, precision=prec, state=s)
        assert torch.equal(a.buffer, b.buffer) and a.position() == lead
    return a, b


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("B", [1, 13])
def test_prefill_equals_stepwise_priming(srwn, cfg, prec, B):
    t = _teacher(srwn, cfg)
    dil, _, _, P, n_far = CFGS[cfg]
    for lead in (0, 2 * P):                            # fresh, and a splice into a state that has generated samples
        for n in (P, n_far):                           # P < sum(d): taps before t0 read the old queues
            seq, par = _pair(t, cfg, B, prec, lead)
            enc, u1, u2, audio = _inputs(cfg, B, n, seed=n + lead)
            t.generate(enc, u1=u1, u2=u2, precision=prec, state=seq, prefix=audio)
            t.prefill(par, audio, enc)
            assert par.position() == lead + n
            assert torch.equal(par.buffer, seq.buffer), (lead, n, (par.buffer != seq.buffer).sum().item())


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("B", [1, 13])
def test_prefill_then_generate_equals_primed_call(srwn, cfg, prec, B):
    t = _teacher(srwn, cfg)
    dil, _, _, P, _ = CFGS[cfg]
    T, n = 1024, 384
    enc, u1, u2, audio = _inputs(cfg, B, T)
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True, precision=prec, prefix=audio[:, :n].contiguous())
    s = t.generation_state(B, prec)
    t.prefill(s, audio[:, :n].contiguous(), enc[:, :n // P].contiguous())
    xc, lgc = t.generate(enc[:, n // P:].contiguous(), u1=u1[:, n:].contiguous(), u2=u2[:, n:].contiguous(),
                         return_logits=True, precision=prec, state=s)
    assert torch.equal(xc, x[:, n:]) and torch.equal(lgc, lg[:, n:])
    assert s.position() == T


def test_prefill_256x4096_fp16(srwn):
    t = _teacher(srwn, "teacher")
    B, n = 256, 4096
    seq, par = _pair(t, "teacher", B, "fp16", 0)
    enc, u1, u2, audio = _inputs("teacher", B, n, seed=8)
    t.generate(enc, u1=u1, u2=u2, precision="fp16", state=seq, prefix=audio)
    t.prefill(par, audio, enc)
    assert par.position() == n
    assert torch.equal(par.buffer, seq.buffer)


@pytest.mark.parametrize("prec", PRECS)
def test_workspace_is_bounded(srwn, prec):
    from sr_wavenet_b200 import _lib
    t = _teacher(srwn, "teacher")
    lib, P = t._eng.lib, 128
    win = sum(synth.DEFAULT_DILATIONS) + 2
    sizes = []
    for k in (2, 20):
        n = -(-k * win // P) * P
        b = ctypes.c_size_t()
        _lib.check(lib.srwn_workspace_bytes(t._eng.h, _lib.OP_TEACHER_PREFILL, 13, n, _lib.PRECISIONS[prec], ctypes.byref(b)))
        sizes.append(b.value)
    assert sizes[0] == sizes[1] > 0


def test_refusals(srwn):
    from sr_wavenet_b200 import _lib
    t = _teacher(srwn, "teacher")
    other = _teacher(srwn, "nonpow2")
    lib, eng = t._eng.lib, t._eng
    B, n, P = 13, 256, 128
    enc, _, _, audio = _inputs("teacher", B, n)
    st = torch.cuda.current_stream().cuda_stream
    ws, wsn = eng.workspace(_lib.OP_TEACHER_PREFILL, B, n, _lib.FP16)
    state = t.generation_state(B, "fp16")
    t.prefill(state, audio, enc)
    before = state.buffer.clone()

    def call(s=state.data_ptr(), x=audio.data_ptr(), e=enc.data_ptr(), nn=n, b=B, prec=_lib.FP16, w=ws, wn=wsn, h=eng.h):
        return lib.srwn_generate_state_prefill(h, s, x, e, nn, b, prec, w, wn, st)

    assert call(nn=0) == _lib.ERR_INVALID
    assert call(nn=-P) == _lib.ERR_INVALID
    assert call(nn=n - 1) == _lib.ERR_INVALID                        # not a multiple of pool_stride
    assert call(x=None) == _lib.ERR_INVALID
    assert call(e=None) == _lib.ERR_INVALID
    assert call(s=None) == _lib.ERR_INVALID
    assert call(s=audio.data_ptr() + 16) == _lib.ERR_INVALID         # never reset
    assert call(b=B - 1) == _lib.ERR_INVALID                         # reset for another B
    assert call(prec=_lib.FP32) == _lib.ERR_INVALID                  # reset for another precision
    assert call(h=other._eng.h) == _lib.ERR_INVALID                  # reset on another handle
    need = ctypes.c_size_t()                                         # the engine's cached workspace may be larger
    _lib.check(lib.srwn_workspace_bytes(eng.h, _lib.OP_TEACHER_PREFILL, B, n, _lib.FP16, ctypes.byref(need)))
    assert 0 < need.value <= wsn
    assert call(wn=need.value - 1) == _lib.ERR_WORKSPACE
    assert call(w=None) == _lib.ERR_WORKSPACE
    assert call(prec=_lib.BF16) == _lib.ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.equal(state.buffer, before)                         # refused calls leave the state alone
    assert lib.srwn_supports(eng.h, _lib.OP_TEACHER_PREFILL, _lib.FP16) == 1
    assert lib.srwn_supports(eng.h, _lib.OP_TEACHER_PREFILL, _lib.FP32) == 1
    # a student handle
    dil = synth.DEFAULT_DILATIONS
    stu = srwn.ParallelWaveNet(input_size=1024, condition_size=0, dilations=dil, teacher=None, num_flows=2,
                               skip_channels=128, latent_channels=32, pool_stride=P)
    assert lib.srwn_supports(stu._eng.h, _lib.OP_TEACHER_PREFILL, _lib.FP32) == 0
    assert call(h=stu._eng.h, prec=_lib.FP32) == _lib.ERR_INVALID
    # fp16 on a configuration the tensor-core generation kernel does not cover (more than 30 layers)
    big = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=5, dilations=[1, 2] * 16,
                                  skip_channels=128, latent_channels=32, pool_stride=P)
    assert lib.srwn_supports(big._eng.h, _lib.OP_TEACHER_PREFILL, _lib.FP16) == 0
    assert call(h=big._eng.h) == _lib.ERR_UNSUPPORTED
    # the Python layer
    with pytest.raises(ValueError):
        t.prefill(state, audio[:1], enc)                             # batch
    with pytest.raises(ValueError):
        t.prefill(state, audio[:, :n - 1], enc)                      # audio and encoding disagree
    with pytest.raises(ValueError):
        t.prefill(state, audio, enc[:, :1])
    with pytest.raises(ValueError):
        t.prefill(t.generation_state(B - 1, "fp16"), audio, enc)     # a state for another batch size
    with pytest.raises(ValueError):
        other.prefill(state, audio, enc)                             # a state of another model
    with pytest.raises(ValueError):
        t.prefill(state, audio[:, :, None], enc)                     # not [B, n]
    torch.cuda.synchronize()
    assert torch.equal(state.buffer, before)


@pytest.mark.parametrize("chunk", [None, "384"])
def test_teacher_driver_prefill(srwn, tmp_path, chunk):
    import teacher as drv
    from scipy.io import wavfile
    tdir, out = str(tmp_path / "teacher"), str(tmp_path / "out")
    t = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=5, dilations=drv.DILATIONS,
                                latent_channels=32, skip_channels=128, pool_stride=128)
    assert t.save(tdir, 7, force=True)
    common = ["--teacher", tdir, "--test-slow", "--num-samples", "1024", "--batch-size", "2", "--clips", "1",
              "--out-dir", out, "--prime", "512"] + (["--chunk", chunk] if chunk else [])
    for prec in PRECS:
        drv.main(common + ["--precision", prec])
        _, ref = wavfile.read(os.path.join(out, "regen_wav_0.wav"))
        drv.main(common + ["--precision", prec, "--prefill"])
        _, got = wavfile.read(os.path.join(out, "regen_wav_0.wav"))
        assert got.shape == (1024,) and np.array_equal(got, ref)
