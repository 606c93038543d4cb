"""-m gpu: splicing utterances between generation states (srwn_generate_state_splice, GenerationState.splice) and the
continuous-batching loop built on it (WaveNetAutoEncoder.generate_requests).

A spliced utterance's queues are rotated from the source's phase t0 mod d_l to the destination's; the source sits at
t0 = 3P and the destination at 6P, a difference that some dilations of both configurations do not divide (384 against
256 and 512; 192 against 5 and 7), so a splice that forgot the rotation would fail here.  Generation after a splice
continues each utterance bit for bit as its source state would, whichever utterances share its CTA or its group of 8;
the scheduler's audio is bit for bit that of generating each request alone."""
import ctypes

import numpy as np
import pytest
import torch

from sr_wavenet_b200 import synth

pytestmark = pytest.mark.gpu

CFGS = {
    # dilations, latent channels, mixtures, pool stride
    "teacher": (synth.DEFAULT_DILATIONS, 32, 5, 128),
    "nonpow2": ([1, 2, 4, 8, 3, 5, 7], 8, 3, 64),
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
        dil, C, M, P = CFGS[cfg]
        t = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=M, dilations=dil, skip_channels=128,
                                    latent_channels=C, pool_stride=P)
        t.set_weights(synth.make_teacher_weights(dil, latent_channels=C, num_mixtures=M, seed=11))
        _models[cfg] = t
    return _models[cfg]


def _inputs(cfg, B, T, seed):
    dil, C, M, P = CFGS[cfg]
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // P, channels=C, seed=seed)).cuda()
    u1, u2 = (torch.from_numpy(a).cuda() for a in synth.sampler_uniforms(B, T, num_mixtures=M, seed=seed + 1))
    audio = torch.from_numpy(synth.synthetic_audio(B, T, seed=seed + 2)).cuda()
    return enc, u1, u2, audio


def _state_at(t, cfg, B, prec, n, seed, prime=0):
    """A state of B utterances at position n: `prime` samples through prefill, then n - prime generated."""
    s = t.generation_state(B, prec)
    if n == 0:
        return s
    enc, u1, u2, audio = _inputs(cfg, B, n, seed)
    P = CFGS[cfg][3]
    if prime:
        t.prefill(s, audio[:, :prime].contiguous(), enc[:, :prime // P].contiguous())
    if n > prime:
        t.generate(enc[:, prime // P:].contiguous(), u1=u1[:, prime:].contiguous(), u2=u2[:, prime:].contiguous(),
                   precision=prec, state=s)
    return s


def _clone(t, s):
    c = t.generation_state(s.batch_size, s.precision)
    c.buffer.copy_(s.buffer)
    return c


def _parts(buf, cfg, B, prec):
    """(t0, x history [B, 2], queues) of a state's bytes, from the documented layout (include/srwn.h, gen_state.cuh):
    header | x history at byte 256 | queues at the next multiple of 256; fp32 queues [B, sum_d, 32] floats, fp16
    [B/8 groups, sum_d, 8 utterances, 64 bytes] (utterance u owns lane quads 4u..4u+3 of a 512-byte slot)."""
    b = buf.cpu().numpy()
    sum_d = sum(CFGS[cfg][0])
    xq = 256 + -(-B * 8 // 256) * 256
    t0 = int(b[:8].view(np.int64)[0])
    xh = b[256:256 + 8 * B].view(np.float32).reshape(B, 2)
    if prec == "fp32":
        q = b[xq:xq + B * sum_d * 128].view(np.float32).reshape(B, sum_d, 32)
    else:
        q = b[xq:xq + -(-B // 8) * sum_d * 512].reshape(-1, sum_d, 8, 64)
    return t0, xh, q


def _utt(q, b, prec):
    return q[b] if prec == "fp32" else q[b >> 3, :, b & 7]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
def test_layout(srwn, cfg, prec):
    """Each spliced utterance is the source's bytes rotated per layer; every other byte of dst, and all of src, stay."""
    t = _teacher(srwn, cfg)
    dil, _, _, P = CFGS[cfg]
    Bs, Bd = 6, 13
    src = _state_at(t, cfg, Bs, prec, 3 * P, seed=31)
    dst = _state_at(t, cfg, Bd, prec, 6 * P, seed=41)
    src0, dst0 = src.buffer.clone(), dst.buffer.clone()
    rows, src_rows = [8, 12, 0, 5, 9], [1, 0, 5, 1, 3]          # 8 and 12 in the padded last group; a source row twice
    dst.splice(rows, src, src_rows)
    torch.cuda.synchronize()
    assert torch.equal(src.buffer, src0)
    ts, xs, qs = _parts(src0, cfg, Bs, prec)
    td = _parts(dst0, cfg, Bd, prec)[0]
    assert (ts, td) == (3 * P, 6 * P)
    assert any((td - ts) % d for d in dil)                       # the rotation is not a no-op for every layer
    exp = dst0.cpu().numpy().copy()                                 # the expected bytes, edited through views
    ex = exp[256:256 + 8 * Bd].view(np.float32).reshape(Bd, 2)
    xq = 256 + -(-Bd * 8 // 256) * 256
    eq = (exp[xq:].view(np.float32).reshape(Bd, -1, 32) if prec == "fp32"
          else exp[xq:].reshape(-1, sum(dil), 8, 64))
    qoff = np.concatenate([[0], np.cumsum(dil)[:-1]])
    for db, sb in zip(rows, src_rows):
        ex[db] = xs[sb]
        s_u, d_u = _utt(qs, sb, prec), _utt(eq, db, prec)
        for d, o in zip(dil, qoff):
            j = np.arange(-d, 0)
            d_u[o + (td + j) % d] = s_u[o + (ts + j) % d]
    got = dst.buffer.cpu().numpy()
    assert np.array_equal(got, exp), int((got != exp).sum())
    assert not np.array_equal(got, dst0.cpu().numpy())


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
@pytest.mark.parametrize("Bs,Bd", [(1, 1), (13, 13), (1, 13), (13, 1)])
def test_continuation(srwn, cfg, prec, Bs, Bd):
    """After a splice from a prefilled state into one that has generated samples, the spliced slots give the samples and
    logits the source utterances give when the source continues by itself; the other slots are unaffected."""
    t = _teacher(srwn, cfg)
    P = CFGS[cfg][3]
    src = _state_at(t, cfg, Bs, prec, 3 * P, seed=51, prime=2 * P)
    dst = _state_at(t, cfg, Bd, prec, 6 * P, seed=61)
    # (destination rows, source rows) by (src B, dst B)
    pairs = {(1, 1): ([0], [0]), (13, 13): ([8, 12, 3], [0, 12, 7]), (1, 13): ([12], [0]), (13, 1): ([0], [12])}
    rows, src_rows = pairs[(Bs, Bd)]
    keep = _clone(t, dst)                                         # dst as it would continue without the splice
    dst.splice(rows, src, src_rows)
    T = 4 * P
    es, u1s, u2s, _ = _inputs(cfg, Bs, T, seed=71)
    ed, u1d, u2d, _ = _inputs(cfg, Bd, T, seed=81)
    xk, lk = t.generate(ed, u1=u1d, u2=u2d, return_logits=True, precision=prec, state=keep)
    for r, sr in zip(rows, src_rows):
        ed[r], u1d[r], u2d[r] = es[sr], u1s[sr], u2s[sr]
    xs, ls = t.generate(es, u1=u1s, u2=u2s, return_logits=True, precision=prec, state=src)
    xd, ld = t.generate(ed, u1=u1d, u2=u2d, return_logits=True, precision=prec, state=dst)
    assert torch.equal(xd[rows], xs[src_rows]), (xd[rows] - xs[src_rows]).abs().max().item()
    assert torch.equal(ld[rows], ls[src_rows])
    other = [b for b in range(Bd) if b not in rows]
    assert torch.equal(xd[other], xk[other]) and torch.equal(ld[other], lk[other])
    assert dst.position() == 10 * P and src.position() == 7 * P


def _requests(cfg, n_req, seed):
    dil, C, M, P = CFGS[cfg]
    rng = np.random.default_rng(seed)
    reqs = []
    for i in range(n_req):
        F = int(rng.integers(2, 12))
        n0 = P * int(rng.integers(0, 3)) if i % 3 == 0 else 0          # some primed, with two prime lengths
        n0 = min(n0, (F - 1) * P)
        enc = synth.synthetic_encoding(1, F, channels=C, seed=seed + i)[0]
        u1, u2 = synth.sampler_uniforms(1, F * P - n0, num_mixtures=M, seed=seed + 100 + i)
        r = {"encoding": torch.from_numpy(enc).cuda(), "u1": torch.from_numpy(u1[0]).cuda(),
             "u2": torch.from_numpy(u2[0]).cuda()}
        if n0:
            r["prime"] = torch.from_numpy(synth.synthetic_audio(1, n0, seed=seed + 200 + i)[0]).cuda()
        reqs.append(r)
    return reqs


def _alone(t, r, prec, P):
    s = t.generation_state(1, prec)
    e = r["encoding"][None]
    n0 = 0 if "prime" not in r else r["prime"].shape[0]
    if n0:
        t.prefill(s, r["prime"][None], e[:, :n0 // P].contiguous())
    return t.generate(e[:, n0 // P:].contiguous(), u1=r["u1"][None], u2=r["u2"][None], precision=prec, state=s)[0]


_refs = {}


@pytest.mark.parametrize("chunk_frames", [1, 3])
@pytest.mark.parametrize("slots", [8, 13])
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cfg", list(CFGS))
def test_scheduler(srwn, cfg, prec, slots, chunk_frames):
    """generate_requests over 20 requests of different lengths, some primed: each request's audio is, bit for bit, the
    audio of generating it alone (B = 1, the same prime through prefill, the same uniforms)."""
    t = _teacher(srwn, cfg)
    P = CFGS[cfg][3]
    reqs = _requests(cfg, 20, seed=5)
    if (cfg, prec) not in _refs:
        _refs[(cfg, prec)] = [_alone(t, r, prec, P) for r in reqs]
    ref = _refs[(cfg, prec)]
    seen = set()
    for i, x in t.generate_requests(reqs, slots=slots, chunk=chunk_frames * P, precision=prec):
        assert i not in seen
        seen.add(i)
        assert x.shape == ref[i].shape and torch.equal(x, ref[i]), (i, (x - ref[i]).abs().max().item())
    assert seen == set(range(len(reqs)))


def test_refusals(srwn):
    from sr_wavenet_b200 import _lib
    t = _teacher(srwn, "teacher")
    other = _teacher(srwn, "nonpow2")
    lib, eng = t._eng.lib, t._eng
    P = CFGS["teacher"][3]
    dst = _state_at(t, "teacher", 13, "fp16", 2 * P, seed=91)
    src = _state_at(t, "teacher", 5, "fp16", P, seed=93)
    d0, s0 = dst.buffer.clone(), src.buffer.clone()
    st = torch.cuda.current_stream().cuda_stream

    def call(d=dst.data_ptr(), db=13, dr=(0, 8), s=src.data_ptr(), sb=5, sr=(1, 4), n=None, prec=_lib.FP16, h=eng.h):
        n = len(dr) if n is None else n
        da = (ctypes.c_int32 * max(len(dr), 1))(*dr) if dr is not None else None
        sa = (ctypes.c_int32 * max(len(sr), 1))(*sr) if sr is not None else None
        return lib.srwn_generate_state_splice(h, d, db, da, s, sb, sa, n, prec, st)

    assert call(d=None) == _lib.ERR_INVALID
    assert call(s=None) == _lib.ERR_INVALID
    assert call(d=d0.data_ptr() + 16) == _lib.ERR_INVALID              # never reset
    assert call(s=s0.data_ptr() + 16) == _lib.ERR_INVALID
    assert call(db=12) == _lib.ERR_INVALID                             # reset for another B
    assert call(sb=6) == _lib.ERR_INVALID
    assert call(prec=_lib.FP32) == _lib.ERR_INVALID                    # reset for another precision
    assert call(h=other._eng.h) == _lib.ERR_INVALID                    # reset on another handle
    assert call(s=dst.data_ptr(), sb=13) == _lib.ERR_INVALID           # src == dst
    assert call(n=-1) == _lib.ERR_INVALID
    assert call(dr=None, sr=None, n=2) == _lib.ERR_INVALID             # rows missing
    assert call(dr=(0, 13)) == _lib.ERR_INVALID                        # destination row out of range
    assert call(dr=(-1, 0)) == _lib.ERR_INVALID
    assert call(sr=(1, 5)) == _lib.ERR_INVALID                         # source row out of range
    assert call(dr=(3, 3)) == _lib.ERR_INVALID                         # destination row named twice
    assert call(prec=_lib.BF16) == _lib.ERR_UNSUPPORTED
    stu = srwn.ParallelWaveNet(input_size=1024, condition_size=0, dilations=synth.DEFAULT_DILATIONS, teacher=None,
                               num_flows=2, skip_channels=128, latent_channels=32, pool_stride=P)
    assert call(h=stu._eng.h, prec=_lib.FP32) == _lib.ERR_INVALID      # a student handle
    big = srwn.WaveNetAutoEncoder(input_size=1024, condition_size=0, num_mixtures=5, dilations=[1, 2] * 16,
                                  skip_channels=128, latent_channels=32, pool_stride=P)
    assert call(h=big._eng.h) == _lib.ERR_UNSUPPORTED                  # fp16 kernel does not cover 32 layers
    assert call(dr=(), sr=(), n=0) == _lib.OK                          # a valid call that does nothing
    torch.cuda.synchronize()
    assert torch.equal(dst.buffer, d0) and torch.equal(src.buffer, s0)
    # the Python layer
    with pytest.raises(ValueError):
        dst.splice([0], dst)                                           # src == dst
    with pytest.raises(ValueError):
        dst.splice([0], _state_at(other, "nonpow2", 5, "fp16", 0, seed=1))   # a state of another model
    with pytest.raises(ValueError):
        dst.splice([0], _state_at(t, "teacher", 5, "fp32", 0, seed=1))       # another precision
    with pytest.raises(ValueError):
        dst.splice([0, 1], src, [0])                                   # lengths disagree
    with pytest.raises(ValueError):
        dst.splice([13], src)
    with pytest.raises(ValueError):
        dst.splice([0], src, [5])
    with pytest.raises(ValueError):
        dst.splice([2, 2], src)
    with pytest.raises(ValueError):
        dst.splice([0], src.buffer)                                    # not a state
    with pytest.raises(ValueError):
        list(t.generate_requests([{"encoding": np.zeros((4, 32), np.float32)}], slots=4, chunk=P + 1))
    with pytest.raises(ValueError):
        list(t.generate_requests([{"encoding": np.zeros((4, 32), np.float32), "prime": np.zeros(P + 1)}], 4, P))
    torch.cuda.synchronize()
    assert torch.equal(dst.buffer, d0) and torch.equal(src.buffer, s0)
