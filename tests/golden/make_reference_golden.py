"""Writes tests/golden/reference_*.npz by EXECUTING the reference's own ops.py / model.py (imported unmodified
from a checkout of tachitachi/SR-WaveNet on top of the NumPy TensorFlow stand-in, tests/tf_shim) in float64 on
seeded inputs.

These are outputs of the reference's code path (its graph construction, operation order, variable naming), not of
the oracle; the per-operation TensorFlow semantics are the stand-in's (see its docstring).  The reference is not part
of this repository, the fixtures are: tests/test_oracle_golden.py holds the oracle to them and
tests/test_gpu_reference_golden.py the CUDA path.

Run from the repo root:  SRWN_REFERENCE_DIR=<reference checkout> python tests/golden/make_reference_golden.py
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]
import refshim  # noqa: E402
import sr_wavenet_b200.synth as synth  # noqa: E402


def f64(d):
    return {k: np.asarray(v, np.float64) for k, v in d.items()}


def make(tag, dil, B, T, P, C, F, M=5, ar_T=0, seeds=(42, 43)):
    tf, _, rmodel = refshim.load()
    tw = synth.make_teacher_weights(dil, latent_channels=C, num_mixtures=M, seed=seeds[0])
    tw.update(synth.make_encoder_weights(len(dil), 2, 128, 128, C, seed=seeds[0] + 2))
    sw = synth.make_student_weights(dil, num_flows=F, latent_channels=C, seed=seeds[1])
    with refshim.quiet():
        t = rmodel.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=M, dilations=dil,
                                      skip_channels=128, latent_channels=C, pool_stride=P)
    refshim.set_variables(t.graph, f64(tw), strict_prefix='WaveNetAutoEncoder/')
    x = synth.synthetic_audio(B, T)
    x[0, 10], x[1 % B, 20] = 1.0, -1.0                     # edge branches of ops.py:167
    enc = synth.synthetic_encoding(B, T // P, C)
    z = synth.logistic_noise(B, T)
    u1, u2 = synth.sampler_uniforms(B, T, M)
    out = dict(dilations=np.array(dil), B=B, T=T, P=P, C=C, F=F, M=M, teacher_seed=seeds[0], student_seed=seeds[1],
               x=x, enc=enc, z=z, u1=u1, u2=u2)
    with tempfile.TemporaryDirectory() as tmp:
        with tf.Session(graph=t.graph).as_default() as sess:
            out['logits'] = t.get_logits(x, enc)                                         # model.py:279-285
            out['nll'] = sess.run(rmodel.discretized_mix_logistic_loss(tf.expand_dims(t.inputs_truth, 2),
                                                                         t.logits_from_encoding, sum_all=False),
                                  {t.inputs_truth: x, t.encoding_isolated: enc})          # ops.py:124-175
            out['nll_sum'] = sess.run(t.loss_encoding, {t.inputs_truth: x, t.encoding_isolated: enc})
            with refshim.inject_uniforms(tf, [u1.astype(np.float64), u2.astype(np.float64)[:, :, None]]):
                out['sample'] = t.reconstruct_with_encoding(x, enc)                      # model.py:264-270
            out['encoding'] = t.encode(x)                                                # model.py:250-255
            if ar_T:                                                                     # teacher.py:153-170
                xs = np.zeros((B, ar_T))
                e = enc[:, :ar_T // P]
                for i in range(ar_T):
                    xs[:, i:] = 0
                    with refshim.inject_uniforms(tf, [u1[:, :ar_T].astype(np.float64), u2[:, :ar_T, None].astype(np.float64)]):
                        xs[:, i] = t.reconstruct_with_encoding(xs, e)[:, i]
                out['ar_x'] = xs
            t.save(tmp, 1, force=True)
        with refshim.quiet():
            s = rmodel.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=tmp, num_flows=F,
                                       skip_channels=128, latent_channels=C, pool_stride=P,
                                       alpha=0.25, beta=1.0, gamma=1.0)                  # student.py:30-33
        refshim.set_variables(s.graph, f64(sw), strict_prefix='ParallelWaveNet/')
        sess = tf.Session(graph=s.graph)
        s.load(sess, None)
        out['student_out'] = s.generate(sess, z, enc)                                    # model.py:570-576
        out['s_tot'], out['mu_tot'] = sess.run([s.s_tot, s.mu_tot], {s.inputs: z, s.encoding: enc})
        out['entropy'] = s.getEntropy_fast(sess, z, enc)
        out['loss'], out['power_loss'] = sess.run([s.loss, s.power_loss],
                                                  {s.inputs: z, s.encoding: enc, s.inputs_truth: x})   # model.py:634-642
    np.savez_compressed(os.path.join(HERE, 'reference_%s.npz' % tag), **out)
    print('reference_%s.npz' % tag, {k: np.shape(v) for k, v in out.items() if np.ndim(v) > 0})


if __name__ == '__main__':
    assert refshim.available(), 'set SRWN_REFERENCE_DIR to a checkout of the reference'
    make('small', [1, 2, 4, 1, 2, 4], B=2, T=1024, P=16, C=8, F=2, ar_T=64, seeds=(11, 12))
    make('default', synth.DEFAULT_DILATIONS, B=2, T=1024, P=128, C=32, F=4)               # teacher.py:55-62
