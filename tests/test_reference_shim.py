"""Pins the oracle by EXECUTING the reference's own source: ops.py and model.py of $SRWN_REFERENCE_DIR are imported
unmodified on top of the NumPy TensorFlow stand-in (tests/tf_shim) and compared with oracle/srwn_oracle.py in
float64.  The graph structure, operation order, variable creation order and every reference quirk
(SURVEY.md F1-F8) come from the reference; only the semantics of single tf.* operations are restated (listed in
tests/tf_shim/tensorflow/__init__.py).  Each test fails if the corresponding fact is restated wrongly in the oracle
or in the synthetic-weight naming (sr-wavenet_b200/synth.py).

The reference (a checkout of tachitachi/SR-WaveNet) is not part of this repository.  Every comparison goes through
``pinned``: with SRWN_REFERENCE_DIR set, the reference's value is computed and compared with the oracle's, and the
committed fixture tests/golden/reference_shim.npz is checked against the reference too; without it, the oracle's
value is compared with the fixture, at the same tolerance.  The fixture holds the values these comparisons held the
reference to (arrays over SAMPLE elements as a seeded sample).  Running this module with
SRWN_REFERENCE_SHIM_RECORD=<path> writes them: the reference's values when it is present, else the oracle's.  The
committed fixture holds the oracle's values, written with the same oracle, synth.py and stand-in under which every
comparison here had last passed against the reference; with SRWN_REFERENCE_DIR set it is checked against the reference
itself.  Only the checks of the reference against itself (its conv known answers, its placeholder names, its own
bookkeeping of gradients) need the reference to run."""
import contextlib
import os

import numpy as np
import pytest

import refshim
import sr_wavenet_b200.synth as synth
from conftest import GOLDEN, f64
from oracle import srwn_oracle as orc

LIVE = refshim.available()
FIXTURE = os.path.join(GOLDEN, "reference_shim.npz")
RECORD = os.environ.get("SRWN_REFERENCE_SHIM_RECORD")
SAMPLE = 512
needs_reference = pytest.mark.skipif(not LIVE, reason="SRWN_REFERENCE_DIR does not name a reference checkout")

TOL = dict(rtol=1e-11, atol=1e-12)
DIL = synth.DEFAULT_DILATIONS                      # teacher.py:55-57

_stored, _recorded = {}, {}
if os.path.exists(FIXTURE):
    with np.load(FIXTURE) as _z:
        _stored = {k: _z[k] for k in _z.files}


def _stored_form(a):
    """The array as the fixture keeps it: whole, or SAMPLE elements of it at seeded positions in index order."""
    a = np.asarray(a)
    if a.dtype.kind in "US" or a.size <= SAMPLE:
        return a
    idx = np.sort(np.random.default_rng(0).choice(a.size, SAMPLE, replace=False))
    return a.reshape(-1)[idx]


def _same(actual, desired, exact, tol, what):
    if exact:
        assert np.asarray(actual).shape == np.asarray(desired).shape and np.array_equal(actual, desired), what
    else:
        np.testing.assert_allclose(actual, desired, err_msg=what, **tol)


def pinned(key, reference, oracle, exact=False, **tol):
    """Compares the reference's value ``reference()`` with ``oracle`` (``exact``: bit for bit / name for name, else
    assert_allclose(reference, oracle, **tol)) and returns the reference's value.  Without the reference, the
    fixture's value stands in for it (the stored sample when the array is large; then None is returned)."""
    o = np.asarray(oracle)
    shape = np.array(o.shape, dtype=np.int64)
    if LIVE:
        r = np.asarray(reference())
        _same(r, o, exact, tol, key)
        if key in _stored:
            _same(_stored[key], _stored_form(r), exact, tol, "fixture vs reference: " + key)
        if RECORD:
            _recorded[key], _recorded[key + "#shape"] = _stored_form(r), np.array(r.shape, dtype=np.int64)
        return r
    if RECORD:
        _recorded[key], _recorded[key + "#shape"] = _stored_form(o), shape
        return o
    assert key in _stored, "%s is not in %s" % (key, FIXTURE)
    assert np.array_equal(_stored[key + "#shape"], shape), (key, _stored[key + "#shape"], o.shape)
    _same(_stored[key], _stored_form(o), exact, tol, "fixture vs oracle: " + key)
    return _stored[key] if _stored[key].size == o.size else None


def _names(names):
    return np.array(sorted(names))


def _variables(shapes):
    """name -> shape as sorted 'name (d0, d1, ...)' strings."""
    return _names("%s %s" % (n, tuple(int(d) for d in sh)) for n, sh in shapes.items())


@pytest.fixture(scope="module", autouse=True)
def _record_fixture():
    yield
    if RECORD and _recorded:
        np.savez_compressed(RECORD, **_recorded)


@pytest.fixture(scope="module")
def ref():
    return refshim.load() if LIVE else (None, None, None)


def _teacher(ref, dil, T, P=128, C=32, S=128, M=5, E=128):
    tf, _, rmodel = ref
    with refshim.quiet():
        t = rmodel.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=M, dilations=dil,
                                      encoder_channels=E, skip_channels=S, latent_channels=C, pool_stride=P)
    return t


def _teacher_weights(dil, C=32, S=128, M=5, E=128, seed=42):
    w = synth.make_teacher_weights(dil, skip_channels=S, latent_channels=C, num_mixtures=M, seed=seed)
    w.update(synth.make_encoder_weights(len(dil), 2, E, S, C, seed=seed + 2))
    return f64(w)


# ------------------------------------------------------------------------------------------ ops.py
@needs_reference
def test_reference_conv_known_answers(ref, conv_kat):
    """ops.py:243-254, run through the reference's _DilatedCausalConv1d (not typed in)."""
    tf, rops, _ = ref
    x = conv_kat["x"].reshape(1, -1, 1)
    run = lambda t: tf.Session().run(t)
    for key, f in (("l243", [1, 1]), ("l244", [1, 0, 1]), ("l245", [1, 0, 0, 0, 1])):
        w = np.array(f, np.float32).reshape(len(f), 1, 1)
        np.testing.assert_array_equal(run(rops._DilatedCausalConv1d(x, w)).ravel(), conv_kat[key])
    for key, d in (("l246", 2), ("l247", 3), ("l248", 4), ("l249", 6)):
        np.testing.assert_array_equal(run(rops._DilatedCausalConv1d(x, np.ones((2, 1, 1), np.float32), dilation_rate=d)).ravel(),
                                      conv_kat[key])
    f4 = np.array([[1, 2, 1, 2]], np.float32).reshape(2, 1, 2)
    np.testing.assert_array_equal(run(rops._DilatedCausalConv1d(x, f4))[0], conv_kat["l252"])
    np.testing.assert_array_equal(run(tf.nn.convolution(x, f4, padding='VALID', dilation_rate=[1]))[0], conv_kat["l254"])


@pytest.mark.parametrize("K,d,R,S", [(2, 1, 32, 128), (2, 4, 8, 4), (3, 5, 6, 10)])
def test_reference_block_matches_oracle(ref, K, d, R, S):
    """ops.py:23-46 incl. F1 (gate = sigmoid of the tanh'd filter conv, _gate variables dead) and F2."""
    tf, rops, _ = ref
    tag = "block_%d_%d_%d_%d/" % (K, d, R, S)
    rng = np.random.default_rng(3)
    shapes = {'blk_filter/blk_Kernel': (K, R, R), 'blk_filter/blk_Bias': (1, 1, R), 'blk_gate/blk_Kernel': (K, R, R),
              'blk_gate/blk_Bias': (1, 1, R), 'conv1d/kernel': (1, R, R), 'conv1d/bias': (R,),
              'conv1d_1/kernel': (1, R, S), 'conv1d_1/bias': (S,)}
    names = list(shapes)
    if LIVE:
        g = tf.Graph()
        with g.as_default():
            x = tf.placeholder(tf.float32, [None, None, R])
            dense, skip = rops.ResidualDilationLayer(x, K, R, S, dilation_rate=d, name='blk')
        sess = tf.Session(graph=g)
    pinned(tag + "names", lambda: np.array(list(g.variables)), np.array(names), exact=True)
    pinned(tag + "shapes", lambda: _variables({n: v._shape for n, v in g.variables.items()}), _variables(shapes),
           exact=True)
    W = {n: rng.normal(0, 0.3, shapes[n]) for n in names}      # the reference draws them in creation order too
    xv = rng.normal(0, 1, (2, 37, R))
    if LIVE:
        for n in names:
            g.variables[n].value = W[n]
    od, os_ = orc.residual_dilation_layer(xv, W['blk_filter/blk_Kernel'], W['blk_filter/blk_Bias'], W['conv1d/kernel'],
                                          W['conv1d/bias'], W['conv1d_1/kernel'], W['conv1d_1/bias'], d)
    rd = pinned(tag + "dense", lambda: sess.run(dense, {x: xv}), od, **TOL)
    pinned(tag + "skip", lambda: sess.run(skip, {x: xv}), os_, **TOL)
    if LIVE:
        # F1: the gate conv has no forward contribution
        g.variables['blk_gate/blk_Kernel'].value = rng.normal(0, 5, g.variables['blk_gate/blk_Kernel']._shape)
        np.testing.assert_array_equal(sess.run(dense, {x: xv}), rd)
    pinned(tag + "live", lambda: _names(v.var_name for v in tf._reachable_variables(dense + tf.reduce_sum(skip))),
           _names(set(names) - {'blk_gate/blk_Kernel', 'blk_gate/blk_Bias'}), exact=True)


def test_reference_shift_resize(ref):
    tf, rops, _ = ref
    rng = np.random.default_rng(4)
    x = rng.normal(size=(2, 9, 3))
    with (tf.Graph().as_default() if LIVE else contextlib.nullcontext()):
        ph = tf.placeholder(tf.float32, [None, None, 3]) if LIVE else None
        for s in (1, 2):
            pinned("shift_%d" % s, lambda: tf.Session().run(rops.RightShift(ph, s), {ph: x}), orc.right_shift(x, s),
                   exact=True)
        for out in (9, 18, 9 * 128):
            pinned("resize_%d" % out, lambda: tf.Session().run(rops.ResizeEmbeddingNearestNeighbor(ph, out), {ph: x}),
                   orc.resize_embedding_nearest_neighbor(x, out), exact=True)


def _mol_inputs(rng, B=3, T=50, M=5):
    l = rng.normal(0, 1.5, (B, T, 4 * M))
    l[..., 2 * M:3 * M] -= 2.0                     # log-scales around -2
    l[0, :5, 2 * M:3 * M] = -12.0                  # below the -7 clamp (ops.py:135)
    x = np.clip(rng.normal(0, 0.6, (B, T, 1)), -1, 1)
    x[0, 0], x[0, 1], x[1, 2], x[1, 3] = 1.0, -1.0, 0.9995, -0.9995          # edge branches (ops.py:167)
    l[2, :10, M:2 * M] = 40.0                      # cdf_delta < 1e-5 -> log_pdf_mid branch
    return x, l


def test_reference_mol_loss_matches_oracle(ref):
    tf, rops, _ = ref
    x, l = _mol_inputs(np.random.default_rng(5))
    if LIVE:
        with tf.Graph().as_default():
            xp, lp = tf.placeholder(tf.float32, [None, None, 1]), tf.placeholder(tf.float32, [None, None, 20])
            s = tf.Session()
            tot = s.run(rops.discretized_mix_logistic_loss(xp, lp), {xp: x, lp: l})
            per = s.run(rops.discretized_mix_logistic_loss(xp, lp, sum_all=False), {xp: x, lp: l})
    pinned("mol_loss_total", lambda: tot, orc.discretized_mix_logistic_loss(x, l, True), rtol=1e-12)
    per = pinned("mol_loss_per_sample", lambda: per, orc.discretized_mix_logistic_loss(x, l, False), **TOL)
    assert per.shape == (3, 50, 1) and np.isfinite(per).all()


def test_reference_mol_sampler_matches_oracle(ref):
    tf, rops, _ = ref
    rng = np.random.default_rng(6)
    _, l = _mol_inputs(rng)
    u1 = rng.uniform(1e-5, 1 - 1e-5, (3, 50, 5))
    u2 = rng.uniform(1e-5, 1 - 1e-5, (3, 50, 1))
    if LIVE:
        with tf.Graph().as_default():
            lp = tf.placeholder(tf.float32, [None, None, 20])
            with refshim.inject_uniforms(tf, [u1, u2]):
                out = tf.Session().run(rops.sample_from_discretized_mix_logistic(lp, 5), {lp: l})
    ref_out, idx = orc.sample_from_discretized_mix_logistic(l, 5, u1, u2, return_index=True)
    out = pinned("mol_sample", lambda: out, ref_out, **TOL)
    assert out.min() >= -1 and out.max() <= 1 and len(np.unique(idx)) > 1


# ------------------------------------------------------------------------------------------ model.py: teacher
def test_reference_teacher_variable_names(ref):
    """The TF1 naming rule synth.py / the checkpoint loader rely on (SURVEY 8b), produced by the reference's own
    constructor: conv1d_{3i} conditioning, conv1d_{3i+1} residual, conv1d_{3i+2} skip, conv1d_90/91 head; encoder."""
    w = _teacher_weights(DIL)
    want = _variables({n: v.shape for n, v in w.items()})
    if LIVE:
        t = _teacher(ref, DIL, 512)
        got = {n: v._shape for n, v in t.graph.variables.items()}
        assert [v.var_name for v in t.network_params] == list(t.graph.variables)      # reuse=True created nothing new
        assert list(t.graph.placeholders) == ['WaveNetAutoEncoder/inputs_placeholder:0', 'WaveNetAutoEncoder/inputs_truth_placeholder:0',
                                              'WaveNetAutoEncoder/conditions_placeholder:0',
                                              'WaveNetAutoEncoder/encoding_nodecoder_placeholder:0']
    got = pinned("teacher_variables", lambda: _variables(got), want, exact=True)
    assert 'WaveNetAutoEncoder/Decoder/conv1d_91/kernel (1, 128, 20)' in got


@pytest.mark.parametrize("dil,T,P,C", [(DIL, 1024, 128, 32), ([1, 2, 4, 1, 2, 4], 64, 16, 8)])
def test_reference_teacher_matches_oracle(ref, dil, T, P, C):
    """get_logits / loss_encoding / encode / reconstruct_with_encoding (model.py:137-200, 250-285) vs the oracle."""
    tf, _, _ = ref
    tag = "teacher_%d_%d_%d_%d/" % (len(dil), T, P, C)
    w = _teacher_weights(dil, C=C)
    B, M = 2, 5
    x = synth.synthetic_audio(B, T).astype(np.float64)
    enc = synth.synthetic_encoding(B, T // P, C).astype(np.float64)
    u1, u2 = (a.astype(np.float64) for a in synth.sampler_uniforms(B, T, M))
    if LIVE:
        t = _teacher(ref, dil, T, P=P, C=C)
        refshim.set_variables(t.graph, w, strict_prefix='WaveNetAutoEncoder/')
        with tf.Session(graph=t.graph).as_default() as sess:
            logits = t.get_logits(x, enc)
            nll = sess.run(t.loss_encoding, {t.inputs_truth: x, t.encoding_isolated: enc})
            with refshim.inject_uniforms(tf, [u1, u2[:, :, None]]):
                rec = t.reconstruct_with_encoding(x, enc)
            encoding = t.encode(x)
            loss_e = sess.run(t.loss, {t.inputs: x, t.inputs_truth: x})
        # the _gate convs exist in the checkpoint and receive no gradient (F1)
        grads = tf.train.AdamOptimizer().compute_gradients(t.loss, t.network_params)
    o_logits = orc.teacher_decoder_logits(w, x, enc, dil, P)
    pinned(tag + "logits", lambda: logits, o_logits, **TOL)
    pinned(tag + "nll", lambda: nll, orc.teacher_nll(w, x, enc, dil, P), rtol=1e-12)
    pinned(tag + "sample", lambda: rec, orc.sample_from_discretized_mix_logistic(o_logits, M, u1, u2[:, :, None])[:, :, 0], **TOL)
    o_enc = orc.teacher_encoder(w, x, len(dil), P)
    pinned(tag + "encoding", lambda: encoding, o_enc, **TOL)
    # model.py:114: the training loss scores the audio under logits decoded from its OWN encoding
    pinned(tag + "loss", lambda: loss_e, orc.teacher_nll(w, x, o_enc, dil, P), rtol=1e-11)
    n, p = len(dil), 'WaveNetAutoEncoder/'
    expect = {'%sDecoder/dilated_conv_%d_gate/dilated_conv_%d_%s' % (p, i, i, k) for i in range(n) for k in ('Kernel', 'Bias')}
    for c in ('Encoder/conv1d_1',                    # nc_conv's skip is discarded (model.py:141)
              'Encoder/conv1d_%d' % (2 * n),         # the last encoder layer's residual output is never read (model.py:144-150)
              'Decoder/conv1d_%d' % (3 * (n - 1) + 1)):   # likewise the last decoder layer's residual 1x1 (model.py:185-190)
        expect |= {p + c + '/kernel', p + c + '/bias'}
    dead = pinned(tag + "dead", lambda: _names(v.var_name for g, v in grads if g is None), _names(expect), exact=True)
    assert sum('_gate/' in n for n in dead) == 2 * len(dil)


def test_reference_naive_ar_loop_matches_oracle(ref):
    """teacher.py:153-170 (the loop body, calling the reference's reconstruct_with_encoding) vs the oracle's naive loop
    and its queue restatement -- the semantics srwn_teacher_generate must reproduce (F4)."""
    tf, _, _ = ref
    dil, T, P, C, M, B = [1, 2, 4, 1, 2, 4], 48, 16, 8, 5, 2
    w = _teacher_weights(dil, C=C, seed=11)
    enc = synth.synthetic_encoding(B, T // P, C, seed=6).astype(np.float64)
    u1, u2 = (a.astype(np.float64) for a in synth.sampler_uniforms(B, T, M, seed=8))
    x_so_far = np.zeros((B, T))
    if LIVE:
        t = _teacher(ref, dil, T, P=P, C=C)
        refshim.set_variables(t.graph, w, strict_prefix='WaveNetAutoEncoder/')
        with tf.Session(graph=t.graph).as_default():
            for i in range(T):                                   # teacher.py:161-167
                x_so_far[:, i:] = 0
                with refshim.inject_uniforms(tf, [u1, u2[:, :, None]]):
                    x_so_far[:, i] = t.reconstruct_with_encoding(x_so_far, enc)[:, i]
    x_so_far = pinned("naive_ar", lambda: x_so_far, orc.naive_ar_loop(w, enc, dil, P, M, u1, u2, T), **TOL)
    np.testing.assert_allclose(x_so_far, orc.queue_ar(w, enc, dil, P, M, u1, u2, T), rtol=1e-9, atol=1e-10)


# ------------------------------------------------------------------------------------------ model.py: student
def _student(ref, tmp_path, dil, T, P, C, F, teacher_w, alpha=0.25, beta=1.0, gamma=1.0):
    tf, _, rmodel = ref
    t = _teacher(ref, dil, T, P=P, C=C)
    refshim.set_variables(t.graph, teacher_w, strict_prefix='WaveNetAutoEncoder/')
    tdir = str(tmp_path / 'teacher')
    with tf.Session(graph=t.graph).as_default():
        assert t.save(tdir, 7, force=True)                   # model.py:230-239 -> model.ckpt-7(.meta)
    with refshim.quiet():
        s = rmodel.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=tdir, num_flows=F,
                                   skip_channels=128, latent_channels=C, pool_stride=P,
                                   alpha=alpha, beta=beta, gamma=gamma)
    return t, s


@pytest.mark.parametrize("dil,T,P,C,F", [(DIL, 1024, 128, 32, 4), ([1, 2, 4, 1, 2, 4], 1024, 16, 8, 2)])
def test_reference_student_matches_oracle(ref, tmp_path, dil, T, P, C, F):
    """createNetwork / createFlow (model.py:415-535), the distillation loss graph (model.py:316-379, incl. F5: the
    imported teacher is teacher-forced on the truth through input_map) and the dead-variable set (F1, F6)."""
    tf, _, _ = ref
    tag = "student_%d_%d_%d_%d_%d/" % (len(dil), T, P, C, F)
    tw = _teacher_weights(dil, C=C)
    sw = f64(synth.make_student_weights(dil, num_flows=F, latent_channels=C))
    B = 2
    z = synth.logistic_noise(B, T).astype(np.float64)
    x = synth.synthetic_audio(B, T).astype(np.float64)
    enc = synth.synthetic_encoding(B, T // P, C).astype(np.float64)
    if LIVE:
        t, s = _student(ref, tmp_path, dil, T, P, C, F, tw)
        variables = {n: v._shape for n, v in s.graph.variables.items()}
        refshim.set_variables(s.graph, sw, strict_prefix='ParallelWaveNet/')
        sess = tf.Session(graph=s.graph)
        s.load(sess, None)                                        # restores the teacher through the imported saver
        out = s.generate(sess, z, enc)
        s_tot, mu_tot = sess.run([s.s_tot, s.mu_tot], {s.inputs: z, s.encoding: enc})
        entropy = s.getEntropy_fast(sess, z, enc)
        feed = {s.inputs: z, s.encoding: enc, s.inputs_truth: x}
        loss, power, tlog = sess.run([s.loss, s.power_loss, s.teacher_logits], feed)
        # student.encode / reconstruct go through the imported teacher (model.py:644-656)
        encoding = s.encode(sess, x)
        # variables without gradient: the gate convs (F1) and the skip 1x1 convs (F6); everything else is live
        live = {v.var_name for g, v in zip(s.grads, [v for g, v in
                tf.train.AdamOptimizer().compute_gradients(s.loss, s.network_params) if g is not None])}
        assert len(s.grads) == len(live) == len(s.placeholder_grads)
    pinned(tag + "variables", lambda: _variables(variables), _variables({n: v.shape for n, v in sw.items()}), exact=True)
    net = orc.student_network(sw, z, enc, dil, P, F)
    pinned(tag + "out", lambda: out, net['out'], **TOL)
    pinned(tag + "s_tot", lambda: s_tot, net['s_tot'], **TOL)
    pinned(tag + "mu_tot", lambda: mu_tot, net['mu_tot'], **TOL)
    pinned(tag + "entropy", lambda: entropy, np.sum(np.log(net['s_tot']) + 2.0), rtol=1e-12)
    o_loss, o_power, _ = orc.distillation_loss(sw, tw, z, x, enc, dil, P, F, alpha=0.25, beta=1.0, gamma=1.0)
    pinned(tag + "teacher_logits", lambda: tlog, orc.teacher_decoder_logits(tw, x, enc, dil, P), **TOL)      # F5
    pinned(tag + "power_loss", lambda: power, o_power, rtol=1e-10)
    pinned(tag + "loss", lambda: loss, o_loss, rtol=1e-10)
    pinned(tag + "encode", lambda: encoding, orc.teacher_encoder(tw, x, len(dil), P), **TOL)
    expect_dead = set()
    for f in range(F):
        p = synth.student_prefix(f)
        for i in range(len(dil)):
            expect_dead |= {'%sdilated_conv_%d_gate/dilated_conv_%d_Kernel' % (p, i, i),
                            '%sdilated_conv_%d_gate/dilated_conv_%d_Bias' % (p, i, i),
                            '%sconv1d_%d/kernel' % (p, 3 * i + 2), '%sconv1d_%d/bias' % (p, 3 * i + 2)}
    dead = pinned(tag + "dead", lambda: _names(set(s.graph.variables) - live), _names(expect_dead), exact=True)
    live_params = sum(int(np.prod(v.shape)) for n, v in sw.items() if n not in set(dead))
    if dil == DIL and F == 4:
        assert live_params == 4 * 125922                      # SURVEY 8(a) a10: live parameters per flow


def test_reference_student_per_example_train_semantics(ref, tmp_path):
    """model.py:603-632 (ParallelWaveNet.train): one B=1 graph evaluation per example with the WHOLE truth batch,
    losses averaged on the host.  Checks the loss / power-loss values that loop reports against the oracle."""
    tf, _, _ = ref
    dil, T, P, C, F, B = [1, 2, 4, 1, 2, 4], 1024, 16, 8, 2, 1
    tw = _teacher_weights(dil, C=C)
    sw = f64(synth.make_student_weights(dil, num_flows=F, latent_channels=C))
    z = synth.logistic_noise(B, T).astype(np.float64)
    x = synth.synthetic_audio(B, T).astype(np.float64)
    enc = synth.synthetic_encoding(B, T // P, C).astype(np.float64)
    if LIVE:
        t, s = _student(ref, tmp_path, dil, T, P, C, F, tw)
        refshim.set_variables(s.graph, sw, strict_prefix='ParallelWaveNet/')
        sess = tf.Session(graph=s.graph)
        s.load(sess, None)
        loss, power = sess.run([s.loss, s.power_loss], {s.inputs: [z[0]], s.encoding: enc, s.inputs_truth: x})
        with pytest.raises(NotImplementedError):              # the stand-in builds the update op but cannot run it
            s.train_fast(sess, z, x, enc)
    o_loss, o_power, _ = orc.distillation_loss(sw, tw, z[:1], x, enc, dil, P, F, alpha=0.25)
    pinned("per_example_train", lambda: [loss, power], [o_loss, o_power], rtol=1e-10)
