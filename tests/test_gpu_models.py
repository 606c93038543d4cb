"""-m gpu: model.py mirror (teacher scoring, autoregressive generation, student synthesis) through
the C ABI vs the NumPy oracle and the committed golden vectors.

Tolerances (BASELINE.json north_star): fp32 path <= 1e-4 relative; 16-bit tensor-core path <= 2e-2
max-abs on logits / per-sample log-likelihood, identical mixture argmax under teacher forcing.

The 16-bit path is fp16 operands (fp32 accumulate and residual stream): measured max |dlogits| ~3e-3,
asserted <= 1e-2 (inside the 2e-2 bound).  bf16 operands are not offered: the bound cannot hold for the
30-layer stack (exact arithmetic on bf16-rounded operands already gives 2.45e-2, tools/bf16_emulation.py),
so the library refuses SRWN_BF16 instead of shipping a looser tolerance (test_bf16_is_refused)."""
import os

import numpy as np
import pytest
import torch

from conftest import f64
from oracle import srwn_oracle as orc
from sr_wavenet_b200 import synth

pytestmark = pytest.mark.gpu

REL = 1e-4
TOL16 = {"fp16": 1e-2}


def _teacher(srwn, dil, C=32, M=5, P=128, seed=42, T=4096):
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=M, dilations=dil,
                                skip_channels=128, latent_channels=C, pool_stride=P)
    w = synth.make_teacher_weights(dil, latent_channels=C, num_mixtures=M, seed=seed)
    t.set_weights(w)
    return t, w


# student: 4 chained flows x 30 layers and an exp() amplify operand rounding; out is clipped to [-1,1]
STUDENT_TOL = {"fp32": 1e-4, "fp16": 2e-2}


def _student(srwn, dil, F, C=32, P=128, seed=43, T=4096):
    s = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=None, num_flows=F,
                             skip_channels=128, latent_channels=C, pool_stride=P)
    w = synth.make_student_weights(dil, num_flows=F, latent_channels=C, seed=seed)
    s.set_weights(w)
    return s, w


@pytest.fixture(scope="module")
def srwn(lib):
    import sr_wavenet_b200
    assert torch.cuda.is_available()
    return sr_wavenet_b200


def _tol(ref, prec):
    return TOL16[prec] if prec in TOL16 else REL * max(1.0, float(np.abs(ref).max()))


def test_teacher_golden_small(srwn, golden_small):
    g = golden_small
    dil = [int(d) for d in g["dilations"]]
    t, _ = _teacher(srwn, dil, C=int(g["C"]), M=int(g["M"]), P=int(g["P"]), seed=int(g["teacher_seed"]))
    for prec in t.available_precisions():
        logits = t.get_logits(g["x"], g["enc"], precision=prec)
        assert np.abs(logits - g["logits"]).max() <= _tol(g["logits"], prec), prec
        nll = t.nll(g["x"], g["enc"], sum_all=False, precision=prec)
        assert np.abs(nll - g["nll"]).max() <= (2 * TOL16[prec] if prec in TOL16 else 2e-4), prec
        tot = t.nll(g["x"], g["enc"], precision=prec)
        assert abs(tot - float(g["nll_sum"])) <= (2e-3 if prec in TOL16 else REL) * abs(float(g["nll_sum"]))
        rec = t.reconstruct_with_encoding(g["x"], g["enc"], u1=g["u1"], u2=g["u2"], precision=prec)
        assert rec.shape == g["x"].shape
        if prec == "fp32":
            np.testing.assert_allclose(rec, g["sample"][:, :, 0], rtol=1e-4, atol=1e-4)


def test_teacher_golden_default_cfg(srwn, golden_default):
    g = golden_default
    B, T, P = int(g["B"]), int(g["T"]), int(g["P"])
    t, _ = _teacher(srwn, synth.DEFAULT_DILATIONS)
    x, enc = synth.synthetic_audio(B, T), synth.synthetic_encoding(B, T // P)
    for prec in t.available_precisions():
        logits = t.get_logits(x, enc, precision=prec)
        assert np.abs(logits - g["logits"]).max() <= _tol(g["logits"], prec), prec
        tot = t.nll(x, enc, precision=prec)
        assert abs(tot - float(g["nll_sum"])) <= (1e-3 if prec in TOL16 else REL) * abs(float(g["nll_sum"]))
        t._eng.check_async(1, B, T, {"fp32": 0, "fp16": 2}[prec])


@pytest.mark.parametrize("B,T", [(1, 128), (3, 3072), (2, 8192), (2, 13440)])
def test_teacher_vs_oracle_shapes(srwn, B, T):
    """Ragged sizes: minimum length (one latent frame), tile-unaligned, longer than the receptive field."""
    dil = synth.DEFAULT_DILATIONS
    t, w = _teacher(srwn, dil)
    x, enc = synth.synthetic_audio(B, T, seed=77), synth.synthetic_encoding(B, T // 128, seed=78)
    ref = orc.teacher_decoder_logits(f64(w), x.astype(np.float64), enc.astype(np.float64), dil, 128)
    for prec in t.available_precisions():
        logits = t.get_logits(x, enc, precision=prec)
        assert np.abs(logits - ref).max() <= _tol(ref, prec), prec
        if prec in TOL16:      # identical Gumbel-argmax mixture indices under teacher forcing (ops.py:187)
            u1, u2 = synth.sampler_uniforms(B, T)
            flips, could = mixture_flips(srwn, ref, logits, u1, u2)
            print("teacher %s %dx%d: %d mixture-index flips of %d positions (%d within reach of the measured error)"
                  % (prec, B, T, flips, B * T, could))


def mixture_flips(srwn, ref_logits, logits, u1, u2, M=5):
    """Exact count of positions where the Gumbel-argmax mixture index (ops.py:187) of the 16-bit logits differs from the
    oracle's, given the same uniforms.  A flip is legitimate only where the oracle's own top-two perturbed logits are
    closer than twice the MEASURED max error of the mixture logits (an adversarial perturbation of that size flips the
    oracle there too); every flip must lie in that set.  Returns (flips, positions within reach)."""
    _, k_ref = orc.sample_from_discretized_mix_logistic(ref_logits, M, u1.astype(np.float64),
                                                        u2.astype(np.float64)[:, :, None], True)
    _, k = srwn.ops.sample_from_discretized_mix_logistic(logits, M, u1, u2, return_index=True)
    k = k.cpu().numpy() if hasattr(k, "cpu") else np.asarray(k)
    eps = float(np.abs(np.asarray(logits, np.float64)[:, :, :M] - ref_logits[:, :, :M]).max())
    pert = ref_logits[:, :, :M] - np.log(-np.log(u1.astype(np.float64)))
    srt = np.sort(pert, axis=2)
    reach = (srt[:, :, -1] - srt[:, :, -2]) <= 2 * eps
    flipped = k != k_ref
    assert not (flipped & ~reach).any(), "a mixture index flipped where the logits differ by more than the gap allows"
    assert flipped.sum() <= reach.sum()
    return int(flipped.sum()), int(reach.sum())


def test_bf16_is_refused(srwn):
    t, _ = _teacher(srwn, synth.DEFAULT_DILATIONS)
    assert "bf16" not in t.available_precisions()
    lib = srwn._lib.load()
    assert lib.srwn_supports(t._eng.h, srwn._lib.OP_TEACHER_LOGITS, srwn._lib.BF16) == 0
    x = torch.zeros(1, 128, device="cuda")
    enc = torch.zeros(1, 1, 32, device="cuda")
    out = torch.zeros(1, 128, 20, device="cuda")
    ws, wsn = t._eng.workspace(srwn._lib.OP_TEACHER_LOGITS, 1, 128, srwn._lib.FP16)
    rc = lib.srwn_teacher_logits(t._eng.h, x.data_ptr(), enc.data_ptr(), out.data_ptr(), 1, 128, srwn._lib.BF16, ws, wsn, 0)
    assert rc == srwn._lib.ERR_UNSUPPORTED


def test_fp16_operands_saturate_instead_of_overflowing(srwn):
    """Encodings scaled until the conditioning pushes |h| past the fp16 range (65504): the 16-bit operand image
    saturates (cvt.rn.satfinite), so logits stay finite instead of turning into inf/NaN for every later layer; below
    the range the usual bound holds relative to the size of the activations."""
    dil = synth.DEFAULT_DILATIONS
    t, w = _teacher(srwn, dil)
    B, T = 1, 1024
    x = synth.synthetic_audio(B, T, seed=3)
    enc100 = synth.synthetic_encoding(B, T // 128, seed=4) * 100.0
    ref = orc.teacher_decoder_logits(f64(w), x.astype(np.float64), enc100.astype(np.float64), dil, 128)
    lg = t.get_logits(x, enc100, precision="fp16")
    assert np.isfinite(lg).all()
    assert np.abs(lg - ref).max() <= 2e-2 * max(1.0, np.abs(ref).max())
    huge = t.get_logits(x, enc100 * 3000.0, precision="fp16")          # |h| ~ 1e6 > 65504
    assert np.isfinite(huge).all()


def test_teacher_pool_stride_and_conditions(srwn):
    """pool_stride != 128, small latent, and a global condition vector (model.py:161-165)."""
    dil = [1, 2, 4, 8, 16, 32]
    B, T, P, C, ncond = 2, 960, 64, 6, 3
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=ncond, num_mixtures=3, dilations=dil,
                                skip_channels=128, latent_channels=C, pool_stride=P)
    w = synth.make_teacher_weights(dil, latent_channels=C + ncond, num_mixtures=3, seed=5)
    t.set_weights(w)
    x, enc = synth.synthetic_audio(B, T, seed=1), synth.synthetic_encoding(B, T // P, C, seed=2)
    cond = np.random.default_rng(3).normal(size=(B, ncond)).astype(np.float32)
    full = np.concatenate([enc, np.tile(cond[:, None, :], [1, T // P, 1])], axis=2)
    ref = orc.teacher_decoder_logits(f64(w), x.astype(np.float64), full.astype(np.float64), dil, P)
    for prec in t.available_precisions():
        logits = t.get_logits(x, enc, cond, precision=prec)
        assert np.abs(logits - ref).max() <= _tol(ref, prec), prec


def test_teacher_causality_on_gpu(srwn):
    dil = synth.DEFAULT_DILATIONS
    t, _ = _teacher(srwn, dil)
    B, T, t0 = 1, 4096, 3500
    x, enc = synth.synthetic_audio(B, T), synth.synthetic_encoding(B, T // 128)
    x2 = x.copy()
    x2[:, t0:] = -x2[:, t0:]
    for prec in t.available_precisions():
        a, b = t.get_logits(x, enc, precision=prec), t.get_logits(x2, enc, precision=prec)
        np.testing.assert_array_equal(a[:, :t0 + 1], b[:, :t0 + 1])
        assert np.abs(a[:, t0 + 1:] - b[:, t0 + 1:]).max() > 0


def test_teacher_errors(srwn):
    t, _ = _teacher(srwn, [1, 2, 4])
    x = synth.synthetic_audio(1, 200)
    with pytest.raises(ValueError):
        t.get_logits(x, synth.synthetic_encoding(1, 1))        # 200 != 128 * 1 (model.py:183)
    with pytest.raises(RuntimeError):
        t._eng.set_weights({"WaveNetAutoEncoder/Decoder/nonsense": np.zeros(3, np.float32)})
    with pytest.raises(RuntimeError):
        t._eng.set_weights({"WaveNetAutoEncoder/Decoder/conv1d_1/kernel": np.zeros((1, 32, 31), np.float32)})
    with pytest.raises(NotImplementedError):
        t.train(x)


@pytest.mark.parametrize("kind", ["teacher", "student"])
def test_encoding_channel_count_is_refused_before_any_launch(srwn, kind):
    """The library reads latent_channels + condition_size floats per frame and is only given a pointer: an encoding with
    one channel too few would be read past its end, one too many would be misread.  Both are refused before a launch."""
    C, P, B, T = 32, 128, 2, 512
    x, z = synth.synthetic_audio(B, T), synth.logistic_noise(B, T)
    if kind == "teacher":
        m, _ = _teacher(srwn, [1, 2, 4], C=C, P=P)
        calls = [lambda e: m.get_logits(x, e), lambda e: m.nll(x, e), lambda e: m.generate(e)]
    else:
        m, _ = _student(srwn, [1, 2, 4], 2, C=C, P=P)
        calls = [lambda e: m.generate(None, z, e), lambda e: m.generate(None, None, e),
                 lambda e: m.forward_all(z, e), lambda e: m.loss_and_grads(z, x, e)]
    launches = srwn._lib.launch_count()
    for channels in (C - 1, C + 1):
        enc = synth.synthetic_encoding(B, T // P, channels)
        for call in calls:
            with pytest.raises(ValueError):
                call(enc)
    assert srwn._lib.launch_count() == launches


def test_generate_golden_small(srwn, golden_small):
    g = golden_small
    dil = [int(d) for d in g["dilations"]]
    t, _ = _teacher(srwn, dil, C=int(g["C"]), M=int(g["M"]), P=int(g["P"]), seed=int(g["teacher_seed"]))
    x, lg = t.generate(g["enc"], u1=g["u1"], u2=g["u2"], return_logits=True)
    np.testing.assert_allclose(lg, g["ar_logits"], rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(x, g["ar_x"], rtol=1e-3, atol=1e-3)
    xz = t.generate(g["enc"], u1=g["u1"], u2=g["u2"], zero_last=True)
    assert np.all(xz[:, -1] == 0)                               # teacher.py:170


def test_generate_vs_oracle_default_cfg(srwn):
    """Queue-based generation == the reference's naive loop semantics (via the oracle's queue
    restatement, itself checked against the naive loop) over 384 steps (3 latent frames)."""
    dil = synth.DEFAULT_DILATIONS
    t, w = _teacher(srwn, dil)
    B, T = 3, 384
    enc = synth.synthetic_encoding(B, T // 128)
    u1, u2 = synth.sampler_uniforms(B, T)
    ref_x, ref_lg = orc.queue_ar(f64(w), enc.astype(np.float64), dil, 128, 5, u1.astype(np.float64),
                                 u2.astype(np.float64), T, return_logits=True)
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True)
    assert np.abs(lg - ref_lg).max() <= 2e-3
    assert np.abs(x - ref_x).max() <= 2e-3


def test_generate_self_consistency_long(srwn):
    """Size-independent property: teacher-forcing the generated audio reproduces the logits the
    generator saw, and re-sampling them with the same noise reproduces the audio."""
    dil = synth.DEFAULT_DILATIONS
    t, _ = _teacher(srwn, dil)
    B, T = 5, 4096                      # > receptive field 3071, odd batch (U=2 tail path at B>SMs not hit)
    enc = synth.synthetic_encoding(B, T // 128)
    u1, u2 = synth.sampler_uniforms(B, T)
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True)
    tf_logits = t.get_logits(x, enc, precision="fp32")
    assert np.abs(tf_logits - lg).max() <= 1e-3
    again = t.reconstruct_with_encoding(x, enc, u1=u1, u2=u2)
    assert np.abs(again - x).max() <= 1e-3
    assert x.min() >= -1 and x.max() <= 1


def _mixture_index(logits, u1, M):
    """ops.py:187: Gumbel-argmax over the mixture logits."""
    return np.argmax(logits[..., :M] - np.log(-np.log(u1)), axis=-1)


@pytest.mark.parametrize("cfg", ["default", "small"])
def test_generate_fp16_tensor_core_path(srwn, cfg):
    """Tensor-core generation kernel (fp16 operands + fp16 queue state, fp32 accumulate / stream).
    (1) against the oracle's queue restatement on the prefix where both pick the same mixture component
    (a flipped near-tie legitimately forks the trajectory): <= 2e-2 max-abs on logits and audio;
    (2) size-independent property: teacher-forcing the generated audio through the fp32 path reproduces
    the logits the generator saw (<= 1e-2, the fp16 operand bound) and the same mixture choices."""
    if cfg == "default":
        dil, C, M, P, B, T = synth.DEFAULT_DILATIONS, 32, 5, 128, 11, 512
    else:
        dil, C, M, P, B, T = [1, 2, 4, 8, 3, 5], 8, 3, 64, 3, 256
    t, w = _teacher(srwn, dil, C=C, M=M, P=P, seed=7)
    if not srwn._lib.load().srwn_supports(t._eng.h, srwn._lib.OP_TEACHER_GENERATE, srwn._lib.FP16):
        pytest.skip("fp16 generation kernel does not cover this configuration")
    enc = synth.synthetic_encoding(B, T // P, channels=C)
    u1, u2 = synth.sampler_uniforms(B, T, num_mixtures=M)
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True, precision="fp16")
    assert x.min() >= -1 and x.max() <= 1 and np.isfinite(lg).all()
    # (2) self-consistency through the fp32 teacher-forced path
    tf_logits = t.get_logits(x, enc, precision="fp32")
    assert np.abs(tf_logits - lg).max() <= 1e-2
    k_ar, k_tf = _mixture_index(lg, u1, M), _mixture_index(tf_logits, u1, M)
    assert (k_ar == k_tf).mean() >= 0.995
    # (1) oracle prefix
    Tq = min(T, 256)
    ref_x, ref_lg = orc.queue_ar(f64(w), enc.astype(np.float64), dil, P, M, u1.astype(np.float64),
                                 u2.astype(np.float64), Tq, return_logits=True)
    k_ref = _mixture_index(ref_lg, u1[:, :Tq], M)
    for b in range(B):
        same = k_ref[b] == k_ar[b, :Tq]
        n = Tq if same.all() else int(np.argmin(same))
        assert n >= 32, "trajectory forked after %d steps" % n
        assert np.abs(lg[b, :n] - ref_lg[b, :n]).max() <= 2e-2
        assert np.abs(x[b, :n] - ref_x[b, :n]).max() <= 2e-2


def test_student_golden_small(srwn, golden_small):
    g = golden_small
    dil = [int(d) for d in g["dilations"]]
    s, _ = _student(srwn, dil, int(g["F"]), C=int(g["C"]), P=int(g["P"]), seed=int(g["student_seed"]))
    for prec in s.available_precisions():
        r = s.forward_all(g["z"], g["enc"], precision=prec)
        tol = STUDENT_TOL[prec]
        assert np.abs(r["out"] - g["student_out"][:, :, 0]).max() <= tol
        assert np.abs(r["s_tot"] / g["s_tot"][:, :, 0] - 1).max() <= tol
        assert np.all(np.abs(r["mu_tot"] - g["mu_tot"][:, :, 0]) <= tol * (1 + np.abs(g["mu_tot"][:, :, 0])))
        assert np.all(np.abs(r["x_last"] - g["x_last"][:, :, 0]) <= tol * (1 + np.abs(g["x_last"][:, :, 0])))
    out = s.generate(None, g["z"], g["enc"])
    assert out.shape == g["student_out"].shape                  # [B,T,1] like model.py:570-576


def test_student_golden_default_cfg(srwn, golden_default):
    g = golden_default
    B, T, P = int(g["B"]), int(g["T"]), int(g["P"])
    s, _ = _student(srwn, synth.DEFAULT_DILATIONS, 4)
    z, enc = synth.logistic_noise(B, T), synth.synthetic_encoding(B, T // P)
    for prec in s.available_precisions():
        r = s.forward_all(z, enc, precision=prec)
        tol = STUDENT_TOL[prec]
        assert np.abs(r["out"] - g["student_out"][:, :, 0]).max() <= tol
        assert np.abs(r["s_tot"] / g["s_tot"][:, :, 0] - 1).max() <= 2 * tol
        s._eng.check_async(3, B, T, {"fp32": 0, "fp16": 2}[prec])
    ent = s.getEntropy_fast(None, z, enc)
    ref_ent = float(np.sum(np.log(g["s_tot"].astype(np.float64)) + 2.0))      # model.py:356
    assert abs(ent - ref_ent) <= 1e-3 * abs(ref_ent)
    per = s.getEntropy(None, z, enc)
    assert per.shape == (B,) and abs(per.sum() - ref_ent) <= 1e-3 * abs(ref_ent)


def test_checkpoint_roundtrip(srwn, tmp_path):
    dil = [1, 2, 4]
    t, w = _teacher(srwn, dil)
    assert t.load(str(tmp_path / "nope")) is None                # model.py:217-228
    assert t.save(str(tmp_path), 7, force=False) is False        # throttled: < 60 s since construction
    assert t.save(str(tmp_path), 7, force=True) is True
    x, enc = synth.synthetic_audio(1, 256), synth.synthetic_encoding(1, 2)
    a = t.get_logits(x, enc)
    t2 = srwn.WaveNetAutoEncoder(256, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=128)
    assert np.abs(t2.get_logits(x, enc) - a).max() > 0
    assert t2.load(str(tmp_path)) is True
    np.testing.assert_array_equal(t2.get_logits(x, enc), a)
    k = synth.TEACHER_PREFIX + "conv1d_1/kernel"
    np.testing.assert_array_equal(t2._eng.get_weight(k, (1, 32, 32)), w[k])


def test_tf_bundle_checkpoint_roundtrip(srwn, tmp_path):
    """A checkpoint directory in TensorFlow's tensor-bundle format (what the reference's Saver writes, model.py:230-239)
    restores into the model; optimizer slots and other variables the graph does not have are ignored."""
    from sr_wavenet_b200 import tf_checkpoint as tfc
    dil = [1, 2, 4]
    t, w = _teacher(srwn, dil)
    t.checkpoint_format = "tf"
    assert t.save(str(tmp_path / "a"), 3, force=True) is True
    assert os.path.exists(str(tmp_path / "a" / "model.ckpt-3.index"))
    x, enc = synth.synthetic_audio(1, 256), synth.synthetic_encoding(1, 2)
    a = t.get_logits(x, enc)
    t2 = srwn.WaveNetAutoEncoder(256, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=128)
    assert t2.load(str(tmp_path / "a")) is True
    np.testing.assert_array_equal(t2.get_logits(x, enc), a)
    # a Saver checkpoint also carries Adam slots, beta powers and the step counter
    full = dict(t.get_weights())
    k = synth.TEACHER_PREFIX + "conv1d_1/kernel"
    full[k + "/Adam"] = np.zeros_like(full[k])
    full[k + "/Adam_1"] = np.ones_like(full[k])
    full["beta1_power"] = np.array(0.9, dtype=np.float32)
    full["global_step"] = np.array(3, dtype=np.int64)
    os.makedirs(str(tmp_path / "b"))
    tfc.write_checkpoint(str(tmp_path / "b" / "model.ckpt-9"), full)
    open(str(tmp_path / "b" / "checkpoint"), "w").write('model_checkpoint_path: "model.ckpt-9"\n')
    t3 = srwn.WaveNetAutoEncoder(256, 0, 5, dil, skip_channels=128, latent_channels=32, pool_stride=128)
    assert t3.load(str(tmp_path / "b")) is True
    np.testing.assert_array_equal(t3.get_logits(x, enc), a)
    # ParallelWaveNet(teacher=<directory>) (model.py:323-334) takes such a directory as it is
    s = srwn.ParallelWaveNet(256, 0, dil, str(tmp_path / "b"), num_flows=2, skip_channels=128, latent_channels=32, pool_stride=128)
    assert s.teacher.num_mixtures == 5 and s.teacher.skip_channels == 128
    np.testing.assert_array_equal(s.teacher.get_logits(x, enc), a)
    # a directory written by WaveNetAutoEncoder.save also carries the .meta skeleton; the student checks the placeholders of
    # its input_map and the collections it reads (model.py:326-341)
    assert os.path.exists(str(tmp_path / "a" / "model.ckpt-3.meta"))
    s2 = srwn.ParallelWaveNet(256, 0, dil, str(tmp_path / "a"), num_flows=2, skip_channels=128, latent_channels=32, pool_stride=128)
    assert set(s2.teacher.meta_collections) == {"Logits_d", "Encoding_output", "Inputs_e", "Out_e", "Out_d"}
    from sr_wavenet_b200 import tf_meta
    nodes, cols = tf_meta.teacher_meta_skeleton()
    del cols["Out_d"]
    tf_meta.write_meta(str(tmp_path / "a" / "model.ckpt-3.meta"), nodes, cols)
    with pytest.raises(IndexError):
        srwn.ParallelWaveNet(256, 0, dil, str(tmp_path / "a"), num_flows=2, skip_channels=128, latent_channels=32, pool_stride=128)


def test_device_resident_path(srwn):
    """CUDA tensors in -> CUDA tensors out (no host copies), same numbers as the NumPy boundary."""
    t, _ = _teacher(srwn, synth.DEFAULT_DILATIONS)
    x, enc = synth.synthetic_audio(2, 1024), synth.synthetic_encoding(2, 8)
    a = t.get_logits(x, enc)
    b = t.get_logits(torch.from_numpy(x).cuda(), torch.from_numpy(enc).cuda())
    assert isinstance(b, torch.Tensor) and b.is_cuda
    np.testing.assert_array_equal(b.cpu().numpy(), a)


def test_nll_stream_matches_nll_batch_by_batch(srwn):
    """The pipelined scoring call (uploads on a copy stream, results read back one batch late) returns, in order, exactly
    what the synchronous call returns for each batch -- pinned and pageable inputs, batches of different content, 1 and 5
    batches, empty sequence."""
    dil, T = [1, 2, 4, 8, 16, 32], 1024
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=5, dilations=dil, skip_channels=128,
                                latent_channels=32, pool_stride=128)
    t.set_weights(synth.make_teacher_weights(dil))
    batches = []
    for k in range(5):
        x, e = synth.synthetic_audio(3, T, seed=50 + k), synth.synthetic_encoding(3, T // 128, seed=70 + k)
        batches.append((torch.from_numpy(x).pin_memory(), torch.from_numpy(e).pin_memory()) if k % 2 else (x, e))
    for prec in ("fp32", "fp16"):
        ref = [t.nll(np.asarray(x), np.asarray(e), precision=prec) for x, e in batches]
        got = list(t.nll_stream(iter(batches), precision=prec))
        assert got == ref, (prec, got, ref)
        assert list(t.nll_stream(batches[:1], precision=prec)) == ref[:1]
        assert list(t.nll_stream([], precision=prec)) == []
        assert list(t.nll_stream(batches, precision=prec, depth=3)) == ref


def test_nll_stream_survives_an_early_stop(srwn):
    """A consumer that stops after the first result (generator closed with work in flight) leaves the handle usable."""
    dil, T = [1, 2, 4, 8], 512
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=5, dilations=dil, skip_channels=128,
                                latent_channels=32, pool_stride=128)
    t.set_weights(synth.make_teacher_weights(dil))
    batches = [(synth.synthetic_audio(2, T, seed=k), synth.synthetic_encoding(2, T // 128, seed=9 + k)) for k in range(4)]
    ref = [t.nll(x, e) for x, e in batches]
    gen = t.nll_stream(iter(batches))
    assert next(gen) == ref[0]
    gen.close()
    assert list(t.nll_stream(batches)) == ref
    with pytest.raises(ValueError):
        list(t.nll_stream([(batches[0][0], batches[0][1][:, :1])]))          # encoding of the wrong length: refused, nothing hangs
    assert t.nll(*batches[1]) == ref[1]


@pytest.mark.parametrize("C", [1, 6, 7, 13])
def test_conditioning_channel_counts_not_multiples_of_four(srwn, C):
    """The conditioning fold of the 16-bit path (fused::k_cond_fold) reads the encoding four channels at a time with a
    remainder loop: latent sizes that are not multiples of four, teacher (model.py:180) and student (model.py:431), on a
    length that spans several chunks and ends inside a latent frame's tile."""
    dil = [1, 2, 4, 8, 16, 32, 1, 2, 4, 8]
    B, T, P = 3, 1664, 128
    x, enc = synth.synthetic_audio(B, T, seed=11), synth.synthetic_encoding(B, T // P, C, seed=12)
    t, w = _teacher(srwn, dil, C=C, M=5, P=P, seed=31)
    ref = orc.teacher_decoder_logits(f64(w), x.astype(np.float64), enc.astype(np.float64), dil, P)
    for prec in t.available_precisions():
        logits = t.get_logits(x, enc, precision=prec)
        assert np.abs(logits - ref).max() <= _tol(ref, prec), (prec, C)
    s, ws = _student(srwn, dil, 2, C=C, P=P, seed=32)
    z = synth.logistic_noise(B, T, seed=13)
    rs = orc.student_network(f64(ws), z.astype(np.float64), enc.astype(np.float64), dil, P, 2)
    for prec in s.available_precisions():
        r = s.forward_all(z, enc, precision=prec)
        assert np.abs(r["out"] - rs["out"][:, :, 0]).max() <= STUDENT_TOL[prec], (prec, C)
