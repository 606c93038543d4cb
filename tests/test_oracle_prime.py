"""Priming on the CPU: the reference's per-sample loop seeded with real audio (teacher.py:153-170 with x[:, :n] given)
and the queue restatement forcing the same samples (tests/primed_ar.py) agree, keep the prefix, teacher-force it, and
with an empty prefix are the oracle's unprimed loops."""
import numpy as np

from conftest import f64
from oracle import srwn_oracle as orc
from primed_ar import naive_ar_loop_primed, queue_ar_primed
import sr_wavenet_b200.synth as synth


def _setup(golden_small, T=48):
    g = golden_small
    dil = [int(d) for d in g["dilations"]]
    tw = f64(synth.make_teacher_weights(dil, latent_channels=int(g["C"]), num_mixtures=int(g["M"]),
                                        seed=int(g["teacher_seed"])))
    P, M = int(g["P"]), int(g["M"])
    enc = g["enc"].astype(np.float64)[:, :T // P]
    u1, u2 = g["u1"].astype(np.float64)[:, :T], g["u2"].astype(np.float64)[:, :T]
    return g, dil, tw, P, M, enc, u1, u2, T


def test_primed_queue_ar_equals_primed_naive_loop(golden_small):
    g, dil, tw, P, M, enc, u1, u2, T = _setup(golden_small)
    n = 20                                              # not a frame boundary: priming ends inside a latent frame
    prefix = g["x"].astype(np.float64)[:, :n]
    naive = naive_ar_loop_primed(tw, enc, dil, P, M, u1, u2, T, prefix)
    fast, lg = queue_ar_primed(tw, enc, dil, P, M, u1, u2, T, prefix)
    np.testing.assert_array_equal(naive[:, :n], prefix)
    np.testing.assert_array_equal(fast[:, :n], prefix)
    np.testing.assert_allclose(fast, naive, rtol=1e-10, atol=1e-12)
    # the logits over the prefix are those of teacher forcing on it, and the rest continues from the real audio
    tf = orc.teacher_decoder_logits(tw, fast, enc, dil, P)
    np.testing.assert_allclose(lg, tf, rtol=1e-9, atol=1e-9)
    unprimed = orc.queue_ar(tw, enc, dil, P, M, u1, u2, T)
    assert np.abs(unprimed[:, n:] - fast[:, n:]).max() > 0


def test_empty_and_full_prefix(golden_small):
    g, dil, tw, P, M, enc, u1, u2, T = _setup(golden_small, T=32)
    empty = np.zeros((enc.shape[0], 0))
    plain, plain_lg = orc.queue_ar(tw, enc, dil, P, M, u1, u2, T, return_logits=True)
    x, lg = queue_ar_primed(tw, enc, dil, P, M, u1, u2, T, empty)
    np.testing.assert_array_equal(x, plain)
    np.testing.assert_array_equal(lg, plain_lg)
    np.testing.assert_array_equal(naive_ar_loop_primed(tw, enc, dil, P, M, u1, u2, T, empty),
                                  orc.naive_ar_loop(tw, enc, dil, P, M, u1, u2, T))
    full = g["x"].astype(np.float64)[:, :T]
    np.testing.assert_array_equal(naive_ar_loop_primed(tw, enc, dil, P, M, u1, u2, T, full), full)
    np.testing.assert_array_equal(queue_ar_primed(tw, enc, dil, P, M, u1, u2, T, full)[0], full)
