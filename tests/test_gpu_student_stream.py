"""-m gpu: chunked student synthesis through a carried flow state (srwn_student_state_*, srwn_student_forward_resume).

With injected noise, a clip split into calls of any multiples of pool_stride gives bit for bit the out, s_tot, mu_tot and
x_last of one forward_all over the clip: fp32 (layer kernels) and fp16 (fused flow kernel, any team size); the student.py
configuration (4 flows, P = 128, latent 32) and one with dilations that are not powers of two, one flow and global
conditions; B = 1 and B = 13.  Device noise, reset, position, the refusals, and the one-call path after stream calls."""
import ctypes

import numpy as np
import pytest
import torch

from sr_wavenet_b200 import synth, _lib

pytestmark = pytest.mark.gpu

CFGS = {
    # dilations, flows, latent channels, condition_size, pool stride, T
    "student": (synth.DEFAULT_DILATIONS, 4, 32, 0, 128, 16384),
    "nonpow2": ([1, 2, 4, 8, 3, 5, 7, 6, 100, 300], 1, 8, 3, 128, 16384),
}
H = {"student": 3072, "nonpow2": 512}        # (2 - 1) * sum(d) + 2 rounded up to P: 3071 -> 3072, 438 -> 512
SPLITS = {
    "all_P": lambda T, P: [P] * (T // P),
    "below_H": lambda T, P: [384] * (T // 384) + ([T % 384] if T % 384 else []),
    "straddle_H": lambda T, P: [128, 2944, 4096, 256, 3072] + [T - 10496],
    "one_call": lambda T, P: [T],
}
PRECS = ["fp32", "fp16"]


@pytest.fixture(scope="module")
def srwn(lib):
    import sr_wavenet_b200
    assert torch.cuda.is_available()
    return sr_wavenet_b200


_models = {}


def _student(srwn, cfg):
    if cfg not in _models:
        dil, F, C, cs, P, T = CFGS[cfg]
        s = srwn.ParallelWaveNet(input_size=T, condition_size=cs, dilations=dil, teacher=None, num_flows=F,
                                 skip_channels=128, latent_channels=C, pool_stride=P)
        s.set_weights(synth.make_student_weights(dil, num_flows=F, latent_channels=C + cs, seed=17))
        _models[cfg] = s
    return _models[cfg]


def _inputs(cfg, B, seed=5):
    dil, F, C, cs, P, T = CFGS[cfg]
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // P, channels=C, seed=seed)).cuda()
    z = torch.from_numpy(synth.logistic_noise(B, T, seed=seed + 1)).cuda()
    cond = torch.from_numpy(np.random.default_rng(seed + 2).standard_normal((B, cs)).astype(np.float32)).cuda() if cs else None
    return z, enc, cond


def _need(srwn, cfg, prec):
    s = _student(srwn, cfg)
    if not s._eng.lib.srwn_supports(s._eng.h, _lib.OP_STUDENT_STREAM, _lib.PRECISIONS[prec]):
        pytest.skip("%s stream not built for this configuration" % prec)
    return s


def _chunked(s, z, enc, cond, prec, sizes, P, state=None):
    state = state or s.synthesis_state(enc.shape[0], prec)
    parts, a = [], 0
    for n in sizes:
        r = s.forward_all(None if z is None else z[:, a:a + n].contiguous(), enc[:, a // P:(a + n) // P].contiguous(),
                          conditions=cond, state=state)
        parts.append(r)
        a += n
    return {k: torch.cat([p[k] for p in parts], 1) for k in parts[0]}, state


def _assert_equal(got, ref, keys=("out", "s_tot", "mu_tot", "x_last")):
    for k in keys:
        assert torch.equal(got[k], ref[k]), "%s differs (max %.3e)" % (k, (got[k] - ref[k]).abs().max().item())


@pytest.mark.parametrize("split", list(SPLITS))
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("B", [1, 13])
def test_chunked_equals_one_call(srwn, cfg, prec, B, split):
    s = _need(srwn, cfg, prec)
    P, T = CFGS[cfg][4], CFGS[cfg][5]
    z, enc, cond = _inputs(cfg, B)
    sizes = SPLITS[split](T, P)
    assert sum(sizes) == T and all(n > 0 and n % P == 0 for n in sizes)
    ref = s.forward_all(z, enc, conditions=cond, precision=prec)
    got, state = _chunked(s, z, enc, cond, prec, sizes, P)
    _assert_equal(got, ref)
    assert state.position() == T


@pytest.mark.parametrize("G", [1, 2, 4, 0])
def test_fp16_team_sizes(srwn, G):
    s = _need(srwn, "student", "fp16")
    P, T = 128, CFGS["student"][5]
    z, enc, cond = _inputs("student", 13, seed=9)
    ref = s.forward_all(z, enc, precision="fp16")
    try:
        s._eng.set_team_size(G)
        got, _ = _chunked(s, z, enc, cond, "fp16", SPLITS["straddle_H"](T, P), P)
    finally:
        s._eng.set_team_size(0)
    _assert_equal(got, ref)


@pytest.mark.parametrize("prec", PRECS)
def test_device_noise_reproduced_by_its_draws(srwn, prec):
    s = _need(srwn, "nonpow2", prec)
    P, T = 128, CFGS["nonpow2"][5]
    _, enc, cond = _inputs("nonpow2", 13, seed=21)
    got, _ = _chunked(s, None, enc, cond, prec, SPLITS["straddle_H"](T, P), P)
    ref = s.forward_all(got["z"].contiguous(), enc, conditions=cond, precision=prec)
    _assert_equal(got, ref)


@pytest.mark.parametrize("prec", PRECS)
def test_reset_and_position(srwn, prec):
    s = _need(srwn, "student", prec)
    P = 128
    z, enc, _ = _inputs("student", 1, seed=33)
    sizes = [256, 4096, 1024]
    state = s.synthesis_state(1, prec)
    assert state.position() == 0
    first, a = [], 0
    for n in sizes:
        first.append(s.generate(None, z[:, a:a + n].contiguous(), enc[:, a // P:(a + n) // P].contiguous(), state=state))
        a += n
        assert state.position() == a
    state.reset()
    assert state.position() == 0
    again, _ = _chunked(s, z[:, :a], enc[:, :a // P], None, prec, sizes, P, state=state)
    assert torch.equal(torch.cat(first, 1)[:, :, 0], again["out"])


def test_refusals_before_any_launch(srwn):
    s = _need(srwn, "student", "fp16")
    lib, h = s._eng.lib, s._eng.h
    P, B, S = 128, 2, 512
    z, enc, _ = _inputs("student", B, seed=41)
    z, enc = z[:, :S].contiguous(), enc[:, :S // P].contiguous()
    out = torch.empty(B, S, device="cuda")
    state = s.synthesis_state(B, "fp16")
    other = s.synthesis_state(B + 1, "fp16")
    f32 = s.synthesis_state(B, "fp32")
    ws, wsn = s._eng.workspace(_lib.OP_STUDENT_STREAM, B, S + P, _lib.FP16)
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream

    def call(state_ptr=state.data_ptr(), t0=0, enc_ptr=enc.data_ptr(), out_ptr=out.data_ptr(), n=S, prec=_lib.FP16,
             handle=h, b=B):
        return lib.srwn_student_forward_resume(handle, state_ptr, t0, z.data_ptr(), 0, 0, enc_ptr, out_ptr, None, None,
                                               None, None, b, n, prec, ws, wsn, st)

    teacher = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=5, dilations=[1, 2], skip_channels=128,
                                      latent_channels=32, pool_stride=128)
    n0 = _lib.launch_count()
    assert call(state_ptr=None) == _lib.ERR_INVALID
    assert call(enc_ptr=None) == _lib.ERR_INVALID
    assert call(out_ptr=None) == _lib.ERR_INVALID
    assert call(handle=teacher._eng.h) == _lib.ERR_INVALID
    assert call(n=0) == _lib.ERR_INVALID and call(n=-P) == _lib.ERR_INVALID and call(n=S - 1) == _lib.ERR_INVALID
    assert call(t0=-P) == _lib.ERR_INVALID and call(t0=P // 2) == _lib.ERR_INVALID
    assert call(state_ptr=other.data_ptr()) == _lib.ERR_INVALID            # reset for B + 1
    assert call(state_ptr=f32.data_ptr()) == _lib.ERR_INVALID              # reset for fp32
    assert call(state_ptr=out.data_ptr()) == _lib.ERR_INVALID              # never reset
    assert call(prec=_lib.BF16) == _lib.ERR_UNSUPPORTED
    assert _lib.launch_count() == n0
    with pytest.raises(ValueError):
        s.generate(None, z, enc, state=other)
    with pytest.raises(ValueError):
        s.generate(None, z, enc, precision="fp32", state=state)
    with pytest.raises(ValueError):
        s.generate(None, z, enc, state=s._flow_model("Flow0").synthesis_state(B, "fp16"))


@pytest.mark.parametrize("prec", PRECS)
def test_wrong_position_aborts_and_leaves_the_state(srwn, prec):
    """A t0 that disagrees with the state raises the abort words on the device: the next call is refused until
    check_async reports it, and the state still continues the clip from where it was."""
    s = _need(srwn, "student", prec)
    P, B = 128, 2
    z, enc, _ = _inputs("student", B, seed=51)
    ref = s.forward_all(z[:, :2048].contiguous(), enc[:, :16].contiguous(), precision=prec)
    state = s.synthesis_state(B, prec)
    first, _ = _chunked(s, z, enc, None, prec, [1024], P, state=state)
    state._t0 = 512                                    # the host's position no longer matches the device's (1024)
    s.forward_all(z[:, 1024:2048].contiguous(), enc[:, 8:16].contiguous(), state=state)
    torch.cuda.synchronize()
    with pytest.raises(_lib.SrwnError, match="t0"):
        s.forward_all(z[:, 1024:2048].contiguous(), enc[:, 8:16].contiguous(), state=state)
    with pytest.raises(_lib.SrwnError, match="t0=512 but its state was at t0=1024"):
        s._eng.check_async(_lib.OP_STUDENT_STREAM, B, 1024, _lib.PRECISIONS[prec])
    assert state.position() == 1024
    state._t0 = 1024
    second, _ = _chunked(s, z[:, 1024:2048].contiguous(), enc[:, 8:16].contiguous(), None, prec, [1024], P, state=state)
    _assert_equal({k: torch.cat([first[k], second[k]], 1) for k in first}, ref)


@pytest.mark.parametrize("prec", PRECS)
def test_one_call_after_stream_calls(srwn, prec):
    """The fused work partition is cached per (B, T, output start): a one-call launch over the same rows as an earlier
    stream buffer (Heff + S) must not reuse the stream's partition."""
    s = _need(srwn, "student", prec)
    P, B, T = 128, 13, 4096
    z, enc, _ = _inputs("student", B, seed=61)
    z, enc = z[:, :T].contiguous(), enc[:, :T // P].contiguous()
    state = s.synthesis_state(B, prec)
    for a in range(0, 3072 + 1024, 1024):             # the last call runs a buffer of 3072 + 1024 = T rows
        s.forward_all(torch.zeros(B, 1024, device="cuda"), enc[:, :8].contiguous(), state=state)
    got = s.forward_all(z, enc, precision=prec)
    fresh = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=CFGS["student"][0], teacher=None, num_flows=4,
                                 skip_channels=128, latent_channels=32, pool_stride=P)
    fresh.set_weights(s.get_weights())
    _assert_equal(got, fresh.forward_all(z, enc, precision=prec))
