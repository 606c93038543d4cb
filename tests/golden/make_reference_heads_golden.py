"""Writes tests/golden/reference_heads.npz by EXECUTING the reference's WaveNet (model.py:8-72) and SiameseWaveNet
(model.py:660-798) classes, imported unmodified from a checkout of tachitachi/SR-WaveNet on top of the NumPy
TensorFlow stand-in (tests/tf_shim), in float64 on seeded weights and inputs.  The CUDA path is held to the fixture
(tests/test_gpu_heads.py); tests/test_heads.py re-derives it when SRWN_REFERENCE_DIR names the checkout.

Run from the repo root:  SRWN_REFERENCE_DIR=<reference checkout> python tests/golden/make_reference_heads_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
import refshim  # noqa: E402

CFG = dict(input_size=96, dilations=[1, 2, 4, 8, 3], filter_width=2, dilation_channels=32, skip_channels=24,
           output_channels=7, output_dimensions=6, margin=1.5)


def seeded_weights(variables, seed):
    """Every trainable variable of the graph, by name (without ':0'), float32 values uniform in +-0.3 (biases too: zero biases would hide
    a bias that is not applied)."""
    rng = np.random.default_rng(seed)
    return {v.name.split(':')[0]: rng.uniform(-0.3, 0.3, size=tuple(int(d) for d in v.shape)).astype(np.float32) for v in variables}


def compute():
    tf, _, rmodel = refshim.load()
    c = CFG
    rng = np.random.default_rng(7)
    out = {'cfg_' + k: np.asarray(v) for k, v in c.items()}
    # ---- classifier
    g = tf.Graph()
    with refshim.quiet(), g.as_default():
        m = rmodel.WaveNet(input_size=c['input_size'], output_size=c['output_channels'], dilations=c['dilations'],
                           filter_width=c['filter_width'], dilation_channels=c['dilation_channels'],
                           skip_channels=c['skip_channels'], output_channels=c['output_channels'])
    w = seeded_weights(m.network_params, 101)
    refshim.set_variables(g, {k: v.astype(np.float64) for k, v in w.items()}, strict_prefix='WaveNet/')
    x = rng.normal(0, 0.5, size=(3, c['input_size'])).astype(np.float32)
    x_long = rng.normal(0, 0.5, size=(2, c['input_size'] + 5)).astype(np.float32)           # the pooling window slides: 6 output frames
    targets = np.eye(c['output_channels'])[[1, 4, 6]]
    with tf.Session(graph=g).as_default() as sess:
        out['wn_logits'] = sess.run(m.logits, {m.inputs: x})
        out['wn_out'] = m.predict(x)
        out['wn_loss'] = np.asarray(sess.run(m.loss, {m.inputs: x, m.targets: targets}))
        out['wn_logits_long'] = sess.run(m.logits, {m.inputs: x_long})
    out.update({'wn_x': x, 'wn_x_long': x_long, 'wn_targets': targets, 'wn_names': np.array(sorted(w))})
    out.update({'wn_w/' + k: v for k, v in w.items()})
    # ---- siamese
    with refshim.quiet():
        s = rmodel.SiameseWaveNet(input_size=c['input_size'], output_dimensions=c['output_dimensions'], dilations=c['dilations'],
                                  margin=c['margin'], filter_width=c['filter_width'], dilation_channels=c['dilation_channels'],
                                  skip_channels=c['skip_channels'])
    w = seeded_weights(s.network_params, 202)
    refshim.set_variables(s.graph, {k: v.astype(np.float64) for k, v in w.items()}, strict_prefix='SiameseWaveNet/')
    xl, xr = (rng.normal(0, 0.5, size=(4, c['input_size'])).astype(np.float32) for _ in range(2))
    labels = np.array([1.0, 0.0, 1.0, 0.0])
    sess = tf.Session(graph=s.graph)
    out['si_embedding'] = s.get_embedding(sess, xl)
    out['si_distance'] = s.get_distance(sess, xl, xr)
    out['si_loss'] = np.asarray(sess.run(s.loss, {s.inputs_left: xl, s.inputs_right: xr, s.labels: labels}))
    out.update({'si_xl': xl, 'si_xr': xr, 'si_labels': labels, 'si_names': np.array(sorted(w))})
    out.update({'si_w/' + k: v for k, v in w.items()})
    # ---- the remaining building blocks of ops.py: the non-causal block (ops.py:48-57) and the two log helpers (ops.py:111-122)
    _, rops, _ = refshim.load()
    for K in (2, 3):
        g = tf.Graph()
        with refshim.quiet(), g.as_default():
            with tf.variable_scope('NCtest'):
                xin = tf.placeholder(tf.float32, [None, None, 5])
                res, skip = rops.ResidualDilationLayerNC(xin, K, dilation_channels=6, skip_channels=4, dilation_rate=7, name='blk')
            variables = tf.get_collection(tf.GraphKeys.TRAINABLE_VARIABLES, 'NCtest')
        w = seeded_weights(variables, 300 + K)
        refshim.set_variables(g, {k: v.astype(np.float64) for k, v in w.items()}, strict_prefix='NCtest/')
        x = rng.normal(0, 1, size=(2, 37, 5)).astype(np.float32)
        with tf.Session(graph=g).as_default() as sess:
            r, sk = sess.run([res, skip], {xin: x})
        out.update({'nc%d_x' % K: x, 'nc%d_residual' % K: r, 'nc%d_skip' % K: sk, 'nc%d_names' % K: np.array(sorted(w))})
        out.update({'nc%d_w/' % K + k: v for k, v in w.items()})
    g = tf.Graph()
    with g.as_default():
        xin = tf.placeholder(tf.float32, [None, None, 7])
        lp, lse = rops.log_prob_from_logits(xin), rops.log_sum_exp(xin)
    x = (rng.normal(0, 3, size=(2, 5, 7)) + 40.0).astype(np.float32)          # shifted: the helpers exist for exactly this
    with tf.Session(graph=g).as_default() as sess:
        a, b = sess.run([lp, lse], {xin: x})
    out.update({'lse_x': x, 'lse_log_prob': a, 'lse_log_sum_exp': b})
    return out


if __name__ == '__main__':
    out = compute()
    path = os.path.join(HERE, 'reference_heads.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, '%d arrays, %.0f KB' % (len(out), os.path.getsize(path) / 1024))
