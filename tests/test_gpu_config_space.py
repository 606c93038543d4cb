"""-m gpu: the 16-bit kernels against the float64 oracle across the configurations they accept, and the ones they refuse.

What the kernels accept (fused.cu fused_supported / fused_check_batch, ar_mma.cu ar_mma_supported) reaches code that runs
only for some configurations: the fused head's M = 5 fast path and the generic one beside it with head2 columns
zero-padded to 32, stacks of 1..40 layers with a dilation of exactly 512, latent frames of 2..4 tiles that straddle the
384-row chunk, batches past 64 utterances (more than 8 teams of a large team size hold), past the SM count, and at the
1184-utterance limit; in the generation kernel every L mod 3 tail of the unrolled layer loop on both sides of the
hidden-tile overlay (L >= 20), 1..6 mixtures (M = 6 fills all three logit n-tiles), frame tables that reload every step
or at odd strides, and a grid with more CTAs than SMs and a ragged last CTA.

Tolerances are the north star's (BASELINE.json): 16-bit logits, per-sample NLL and student outputs <= 2e-2 max-abs
relative to max(1, max |ref|); the reduced NLL <= 2e-3 relative; generated trajectories agree with the oracle for at
least 32 steps before a mixture choice forks them.  Every case prints its measured error."""
import numpy as np
import pytest
import torch

from conftest import f64
from oracle import srwn_oracle as orc
from sr_wavenet_b200 import synth, _lib

pytestmark = pytest.mark.gpu

TOL16 = 2e-2
TOL_SUM = 2e-3


@pytest.fixture(scope="module")
def srwn(lib):
    import sr_wavenet_b200
    assert torch.cuda.is_available()
    return sr_wavenet_b200


def dilations(L):
    """L layers of the 1..512 doubling cycle (every stack past 9 layers has a dilation of exactly 512)."""
    return [1 << (i % 10) for i in range(L)]


def rel_err(got, ref):
    return float(np.abs(np.asarray(got, np.float64) - ref).max() / max(1.0, np.abs(ref).max()))


def teacher(srwn, dil, M, P, T, seed):
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=M, dilations=dil, skip_channels=128,
                                latent_channels=32, pool_stride=P)
    w = synth.make_teacher_weights(dil, num_mixtures=M, seed=seed)
    t.set_weights(w)
    return t, w


def student(srwn, dil, F, P, T, seed):
    s = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=None, num_flows=F, skip_channels=128,
                             latent_channels=32, pool_stride=P)
    w = synth.make_student_weights(dil, num_flows=F, seed=seed)
    s.set_weights(w)
    return s, w


def oracle_teacher(w, x, enc, dil, P):
    ref = orc.teacher_decoder_logits(f64(w), x.astype(np.float64), enc.astype(np.float64), dil, P)
    nll = orc.discretized_mix_logistic_loss(x.astype(np.float64)[:, :, None], ref, sum_all=False)[:, :, 0]
    return ref, nll


# ---- fused teacher ----------------------------------------------------------------------------------------------------
# (M, dilations, P, B, T): every M the head takes (the M = 5 fast path is the bench's), 1 / 2 / 31 / 40 layers, frames of
# 2, 3 and 4 tiles against the 384-row chunk, T past the receptive field where it is affordable (pieces that start
# mid-utterance warm up through the whole dependency cone)
TEACHER_CASES = [
    (1, [512], 256, 3, 1792),
    (2, [3, 512], 384, 3, 3456),
    (4, dilations(30) + [100], 512, 2, 4096),
    (6, dilations(40), 256, 2, 4352),
    (7, dilations(31), 256, 3, 3840),
    (8, dilations(40), 512, 2, 4608),
    (8, [512], 384, 4, 1152),
]


@pytest.mark.parametrize("M,dil,P,B,T", TEACHER_CASES, ids=["M%d-L%d-P%d" % (c[0], len(c[1]), c[2]) for c in TEACHER_CASES])
def test_fused_teacher_vs_oracle(srwn, M, dil, P, B, T):
    t, w = teacher(srwn, dil, M, P, T, seed=10 + M)
    assert "fp16" in t.available_precisions()
    x = synth.synthetic_audio(B, T, seed=M)
    enc = synth.synthetic_encoding(B, T // P, seed=M + 1)
    ref, ref_nll = oracle_teacher(w, x, enc, dil, P)
    logits = t.get_logits(x, enc, precision="fp16")
    nll = t.nll(x, enc, sum_all=False, precision="fp16")[:, :, 0]
    tot = t.nll(x, enc, precision="fp16")
    e_lg, e_nll = rel_err(logits, ref), rel_err(nll, ref_nll)
    e_tot = abs(tot - ref_nll.sum()) / abs(ref_nll.sum())
    print("fused teacher M=%d L=%d P=%d %dx%d partition %s: logits %.2e, nll %.2e, reduced nll %.2e"
          % (M, len(dil), P, B, T, t._eng.last_partition(), e_lg, e_nll, e_tot))
    assert e_lg <= TOL16 and e_nll <= TOL16 and e_tot <= TOL_SUM


@pytest.mark.parametrize("B", [65, 148, 149, 1184])
def test_fused_teacher_large_batches(srwn, B):
    """One 256-row utterance each (T = P): utterance 0, the last one and the first of the second team against the oracle,
    every utterance bit for bit what it is in a permuted batch (it lands in another team and piece there)."""
    dil, M, P, T = synth.DEFAULT_DILATIONS, 5, 256, 256
    t, w = teacher(srwn, dil, M, P, T, seed=3)
    x = synth.synthetic_audio(B, T, seed=B)
    enc = synth.synthetic_encoding(B, 1, seed=B + 1)
    logits = t.get_logits(x, enc, precision="fp16")
    nll = t.nll(x, enc, sum_all=False, precision="fp16")[:, :, 0]
    tot = t.nll(x, enc, precision="fp16")
    teams, G = t._eng.last_partition()
    assert teams * G <= torch.cuda.get_device_properties(0).multi_processor_count
    pick = sorted({0, -(-B // teams), B - 1})                  # the first utterance of the second team (pieces in order)
    ref, ref_nll = oracle_teacher(w, x[pick], enc[pick], dil, P)
    e_lg, e_nll = rel_err(logits[pick], ref), rel_err(nll[pick], ref_nll)
    print("fused teacher B=%d partition (%d, %d), utterances %s: logits %.2e, nll %.2e" % (B, teams, G, pick, e_lg, e_nll))
    assert e_lg <= TOL16 and e_nll <= TOL16
    np.testing.assert_allclose(tot, nll.astype(np.float64).sum(), rtol=1e-5)
    perm = np.random.default_rng(B).permutation(B)
    assert np.array_equal(t.get_logits(x[perm], enc[perm], precision="fp16"), logits[perm])
    assert np.array_equal(t.nll(x[perm], enc[perm], sum_all=False, precision="fp16")[:, :, 0], nll[perm])


# ---- fused student ----------------------------------------------------------------------------------------------------
# (F, P, B, T), 40 layers: 1..16 flows, frames of 2 and 4 tiles, 65 and 200 utterances; F = 1 runs past the receptive
# field (4092 rows), so pieces start mid-utterance
STUDENT_CASES = [(1, 256, 65, 5120), (3, 512, 200, 2048), (8, 256, 65, 1024), (16, 512, 200, 1024)]


def fp16_operand_layer(inputs, fk, fb, rk, rb, sk, sb, dilation_rate=1):
    """orc.residual_dilation_layer (student: no skip) in exact arithmetic on the fused kernel's 16-bit GEMM operands: the
    layer input and the filter weights, the gate output and the residual weights rounded to fp16, the rest float64."""
    h16 = lambda a: a.astype(np.float16).astype(np.float64)
    f = np.tanh(orc.dilated_causal_conv1d(h16(inputs), h16(fk), dilation_rate) + fb)
    residual = h16(f * orc.sigmoid(f)) @ h16(rk[0]) + rb
    return (inputs + residual) * np.sqrt(0.5), None


@pytest.mark.parametrize("F,P,B,T", STUDENT_CASES, ids=["F%d-P%d-B%d" % c[:3] for c in STUDENT_CASES])
def test_fused_student_vs_oracle(srwn, monkeypatch, F, P, B, T):
    """The composed outputs against the oracle, then each flow alone, fed the oracle's own input of that flow: a flow
    whose scale or mean were wrong shows there even when the chain hides or amplifies it."""
    dil = dilations(40)
    s, w = student(srwn, dil, F, P, T, seed=20 + F)
    assert "fp16" in s.available_precisions()
    z = synth.logistic_noise(B, T, seed=F)
    enc = synth.synthetic_encoding(B, T // P, seed=F + 1)
    r = s.forward_all(z, enc, precision="fp16")
    pick = [0, B // 2, B - 1]
    z64, e64 = z[pick].astype(np.float64), enc[pick].astype(np.float64)
    full = orc.student_network(f64(w), z64, e64, dil, P, F)
    ref = {k: full[k][:, :, 0] for k in ("out", "s_tot", "mu_tot", "x_last")}
    e_out = float(np.abs(r["out"][pick] - ref["out"]).max())
    e_s = float(np.abs(r["s_tot"][pick] / ref["s_tot"] - 1).max())
    e_mu, e_x = rel_err(r["mu_tot"][pick], ref["mu_tot"]), rel_err(r["x_last"][pick], ref["x_last"])
    # flow by flow
    x, e_flow = z64, 0.0
    for f in range(F):
        pre = synth.student_prefix(f)
        one = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=None, num_flows=1,
                                   skip_channels=128, latent_channels=32, pool_stride=P)
        one.set_weights({k.replace(pre, synth.student_prefix(0)): v for k, v in w.items() if k.startswith(pre)})
        r1 = one.forward_all(x.astype(np.float32), e64.astype(np.float32), precision="fp16")
        sc, mn = full["scales"][f][:, :, 0], full["means"][f][:, :, 0]
        x_next = x * sc + mn
        e_flow = max(e_flow, float(np.abs(np.log(r1["s_tot"] / sc)).max()), rel_err(r1["mu_tot"], mn),
                     rel_err(r1["x_last"], x_next))
        x = x_next
    # what exact arithmetic on the kernel's fp16 operands reaches on the same inputs
    monkeypatch.setattr(orc, "residual_dilation_layer", fp16_operand_layer)
    q = orc.student_network(f64(w), z64, e64, dil, P, F)["out"][:, :, 0]
    e_q, e_kq = float(np.abs(q - ref["out"]).max()), float(np.abs(r["out"][pick] - q).max())
    print("fused student F=%d P=%d %dx%d partition %s: out %.2e, s_tot %.2e (rel), mu_tot %.2e, x_last %.2e; worst single "
          "flow %.2e; exact arithmetic on fp16 operands: out %.2e from the oracle, %.2e from the kernel"
          % (F, P, B, T, s._eng.last_partition(), e_out, e_s, e_mu, e_x, e_flow, e_q, e_kq))
    # mu_tot and out are one composition (model.py:535), up to fp32 rounding of terms as large as |mu_tot|
    zs = z * r["s_tot"]
    assert (np.abs(r["out"] - np.clip(zs + r["mu_tot"], -1, 1)) <= 1e-6 * (1 + np.abs(zs) + np.abs(r["mu_tot"]))).all()
    assert max(e_s, e_mu, e_x, e_flow) <= TOL16
    perm = np.random.default_rng(F).permutation(B)
    rp = s.forward_all(z[perm], enc[perm], precision="fp16")
    for k in ("out", "s_tot", "mu_tot", "x_last"):
        assert np.array_equal(rp[k], r[k][perm]), k
    # `out` is the small difference of z * s_tot and mu_tot; where the chain makes those large (8 flows here: per-flow
    # scales up to 19, |mu_tot| up to 26) fp16 operands alone move it by more than 2e-2 -- exact arithmetic on them does
    # (3.1e-2 at F = 8; every single flow stays at the fp16 unit roundoff).  The kernel is held to 2e-2 from that
    # operand-grade result in every case, and to 2e-2 from the oracle wherever the operand grade allows it.
    assert e_kq <= TOL16
    assert e_out <= max(TOL16, e_q)


# ---- tensor-core generation -------------------------------------------------------------------------------------------
def mixture_index(logits, u1, M):
    return np.argmax(logits[..., :M] - np.log(-np.log(u1)), axis=-1)


def check_generation(t, w, dil, M, P, enc, u1, u2, oracle_rows, tag):
    """(1) the oracle's queue restatement on the prefix before the first flipped mixture choice, (2) teacher forcing of
    the generated audio through the fp32 path reproduces the logits the generator saw and its mixture choices."""
    x, lg = t.generate(enc, u1=u1, u2=u2, return_logits=True, precision="fp16")
    assert x.min() >= -1 and x.max() <= 1 and np.isfinite(lg).all()
    tf = t.get_logits(x, enc, precision="fp32")
    e_tf = rel_err(lg, tf.astype(np.float64))
    agree = float((mixture_index(lg, u1, M) == mixture_index(tf, u1, M)).mean())
    T = x.shape[1]
    ref_x, ref_lg = orc.queue_ar(f64(w), enc[oracle_rows].astype(np.float64), dil, P, M, u1[oracle_rows].astype(np.float64),
                                 u2[oracle_rows].astype(np.float64), T, return_logits=True)
    k_ref, k_ar = mixture_index(ref_lg, u1[oracle_rows], M), mixture_index(lg[oracle_rows], u1[oracle_rows], M)
    fork, e_lg, e_x = T, 0.0, 0.0
    for i in range(len(oracle_rows)):
        same = k_ref[i] == k_ar[i]
        n = T if same.all() else int(np.argmin(same))
        fork = min(fork, n)
        e_lg = max(e_lg, rel_err(lg[oracle_rows[i], :n], ref_lg[i, :n]))
        e_x = max(e_x, float(np.abs(x[oracle_rows[i], :n] - ref_x[i, :n]).max()))
    print("generation %s: oracle logits %.2e, audio %.2e, first fork at step %d; teacher-forced logits %.2e, "
          "mixture choices %.4f the same" % (tag, e_lg, e_x, fork, e_tf, agree))
    assert fork >= 32 and e_lg <= TOL16 and e_x <= TOL16
    assert e_tf <= TOL16 and agree >= 0.995


# (L, M, P): every L mod 3 below the overlay switch (3..14) and above it (20..29), M up to 6, frames of 1, 3 and 100 steps
GEN_CASES = [(3, 1, 1), (4, 2, 3), (5, 4, 100), (13, 6, 1), (14, 1, 3), (20, 2, 100), (21, 4, 1), (22, 6, 3), (29, 6, 100)]


@pytest.mark.parametrize("L,M,P", GEN_CASES, ids=["L%d-M%d-P%d" % c for c in GEN_CASES])
def test_generation_tensor_core_vs_oracle(srwn, L, M, P):
    dil, B, T = dilations(L), 9, 300                           # 9 utterances: a full CTA of 8 and a ragged one
    t, w = teacher(srwn, dil, M, P, T, seed=30 + L)
    assert _lib.load().srwn_supports(t._eng.h, _lib.OP_TEACHER_GENERATE, _lib.FP16) == 1
    enc = synth.synthetic_encoding(B, T // P, seed=L)
    u1, u2 = synth.sampler_uniforms(B, T, num_mixtures=M, seed=L + 1)
    check_generation(t, w, dil, M, P, enc, u1, u2, list(range(B)), "L=%d M=%d P=%d" % (L, M, P))


def test_generation_tensor_core_more_ctas_than_sms(srwn):
    """1185 utterances: 149 CTAs of 8 on 148 SMs, the last one holding a single utterance."""
    dil, M, P, B, T = synth.DEFAULT_DILATIONS, 5, 128, 1185, 128
    t, w = teacher(srwn, dil, M, P, T, seed=5)
    enc = synth.synthetic_encoding(B, 1, seed=6)
    u1, u2 = synth.sampler_uniforms(B, T, num_mixtures=M, seed=7)
    check_generation(t, w, dil, M, P, enc, u1, u2, [0, 1183, 1184], "B=%d" % B)


# ---- what the kernels refuse ------------------------------------------------------------------------------------------
def refused_before_launch(calls):
    """Each call raises the library's SRWN_ERR_UNSUPPORTED (or the host layer's refusal of that precision) without a launch."""
    before = _lib.launch_count()
    for call in calls:
        with pytest.raises(RuntimeError) as e:
            call()
        if isinstance(e.value, _lib.SrwnError):
            assert e.value.code == _lib.ERR_UNSUPPORTED, str(e.value)
    assert _lib.launch_count() == before


FUSED_REFUSED = {"L41": (dilations(40) + [1], 128), "d513": ([1, 513], 128), "P64": ([1, 2, 4], 64)}


@pytest.mark.parametrize("name", list(FUSED_REFUSED))
def test_fused_refusals_match_srwn_supports(srwn, name):
    dil, P = FUSED_REFUSED[name]
    B, T = 2, 4 * P
    lib = _lib.load()
    t, _ = teacher(srwn, dil, 5, P, T, seed=1)
    s, _ = student(srwn, dil, 2, P, T, seed=2)
    assert t.available_precisions() == ["fp32"] and s.available_precisions() == ["fp32"]
    for op in (_lib.OP_TEACHER_LOGITS, _lib.OP_TEACHER_NLL):
        assert lib.srwn_supports(t._eng.h, op, _lib.FP16) == 0
    assert lib.srwn_supports(s._eng.h, _lib.OP_STUDENT_FORWARD, _lib.FP16) == 0
    x, z = synth.synthetic_audio(B, T), synth.logistic_noise(B, T)
    enc = synth.synthetic_encoding(B, T // P)
    refused_before_launch([lambda: t.get_logits(x, enc, precision="fp16"), lambda: t.nll(x, enc, precision="fp16"),
                           lambda: s.forward_all(z, enc, precision="fp16")])
    assert np.isfinite(t.get_logits(x, enc, precision="fp32")).all()        # the fp32 path still serves the configuration


@pytest.mark.parametrize("L,M", [(15, 5), (16, 5), (17, 5), (18, 5), (19, 5), (10, 7)])
def test_generation_refusals_match_srwn_supports(srwn, L, M):
    dil, P, B, T = dilations(L), 128, 2, 256
    t, _ = teacher(srwn, dil, M, P, T, seed=1)
    assert _lib.load().srwn_supports(t._eng.h, _lib.OP_TEACHER_GENERATE, _lib.FP16) == 0
    enc = synth.synthetic_encoding(B, T // P)
    u1, u2 = synth.sampler_uniforms(B, T, num_mixtures=M)
    refused_before_launch([lambda: t.generate(enc, u1=u1, u2=u2, precision="fp16")])


def test_batch_past_the_fused_limit_is_refused(srwn):
    """8 utterances per SM (1184 on 148 SMs) is what one fused launch takes: one more is refused before any launch by every
    16-bit call that runs the fused kernel, with a message that names the limit."""
    limit = 8 * torch.cuda.get_device_properties(0).multi_processor_count
    B, T, P = limit + 1, 256, 128
    t, _ = teacher(srwn, [1, 2, 4], 5, P, T, seed=1)
    s, _ = student(srwn, [1, 2, 4], 2, P, T, seed=2)
    x, z = synth.synthetic_audio(B, T), synth.logistic_noise(B, T)
    enc = synth.synthetic_encoding(B, T // P)
    state = s.synthesis_state(B, "fp16")
    calls = [lambda: t.get_logits(x, enc, precision="fp16"), lambda: t.nll(x, enc, precision="fp16"),
             lambda: s.forward_all(z, enc, precision="fp16"), lambda: s.generate(None, None, enc, precision="fp16"),
             lambda: s.forward_all(z, enc, precision="fp16", state=state)]
    before = _lib.launch_count()
    for call in calls:
        with pytest.raises(_lib.SrwnError) as e:
            call()
        assert e.value.code == _lib.ERR_UNSUPPORTED and str(limit) in str(e.value), str(e.value)
    assert _lib.launch_count() == before
    assert state.position() == 0
    # the limit itself runs
    assert np.isfinite(t.get_logits(x[:limit], enc[:limit], precision="fp16")).all()
