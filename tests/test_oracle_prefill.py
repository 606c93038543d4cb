"""The window argument of the parallel prefill on the CPU (tests/prefill_ref.py): the state after n forced samples,
computed from the last sum(d) + 2 samples only (plus the prior state where that window reaches before t0), equals the
state of the queue loop stepped over all n samples.  Fresh states and states at t0 > 0; n below, at and far past the
window; the teacher.py dilations and a set that is not powers of two."""
import numpy as np
import pytest

from conftest import f64
from prefill_ref import fresh_state, prefill_state, step_state
import sr_wavenet_b200.synth as synth

NONPOW2 = [1, 2, 4, 8, 3, 5, 7]            # sum 30: window 32


def _model(dil, C=8, seed=5):
    return f64(synth.make_teacher_weights(dil, latent_channels=C, num_mixtures=3, seed=seed))


def _data(B, n, P, C, seed):
    x = synth.synthetic_audio(B, max(n, 64), seed=seed).astype(np.float64)[:, :n]
    enc = synth.synthetic_encoding(B, -(-n // P), channels=C, seed=seed + 1).astype(np.float64)
    return x, enc


def _assert_same(a, b):
    assert a["t0"] == b["t0"]
    np.testing.assert_array_equal(a["xh"], b["xh"])
    for qa, qb in zip(a["queues"], b["queues"]):
        np.testing.assert_allclose(qa, qb, rtol=1e-12, atol=1e-13)


def _start(w, dil, P, C, B, t0):
    s = fresh_state(B, dil)
    if t0:
        x, enc = _data(B, t0, P, C, seed=40)
        s = step_state(w, enc, dil, P, x, s)
        assert np.abs(np.concatenate([q.reshape(-1) for q in s["queues"]])).max() > 0
    return s


@pytest.mark.parametrize("t0", [0, 13])
@pytest.mark.parametrize("n", [1, 7, 29, 31, 32, 33, 64, 150])     # window sum(d) + 2 = 32
def test_prefill_equals_stepping_nonpow2(t0, n):
    dil, P, C, B = NONPOW2, 4, 8, 3
    w = _model(dil)
    s0 = _start(w, dil, P, C, B, t0)
    x, enc = _data(B, n, P, C, seed=7 + n)
    ref = step_state(w, enc, dil, P, x, s0)
    got, rows = prefill_state(w, enc, dil, P, x, s0, return_rows=True)
    _assert_same(got, ref)
    # only the cone is computed: layer l over min(n, D_l) positions
    assert rows == [min(n, sum(dil[l:])) for l in range(len(dil))]


@pytest.mark.parametrize("t0,n", [(0, 1000), (0, 3070), (0, 3071), (256, 512), (256, 3200), (384, 7000)])
def test_prefill_equals_stepping_teacher_dilations(t0, n):
    dil, P, C, B = synth.DEFAULT_DILATIONS, 128, 32, 2
    assert sum(dil) + 2 == 3071
    w = _model(dil, C=C, seed=11)
    s0 = _start(w, dil, P, C, B, t0)
    x, enc = _data(B, n, P, C, seed=3)
    ref = step_state(w, enc, dil, P, x, s0)
    got = prefill_state(w, enc, dil, P, x, s0)
    _assert_same(got, ref)


def test_state_depends_on_the_window_only():
    """Samples before the last sum(d) + 2 do not reach the state."""
    dil, P, C, B = NONPOW2, 4, 8, 2
    w = _model(dil)
    n = 96
    x, enc = _data(B, n, P, C, seed=9)
    a = prefill_state(w, enc, dil, P, x, fresh_state(B, dil))
    x2 = x.copy()
    x2[:, :n - sum(dil) - 2] = 0.5
    b = step_state(w, enc, dil, P, x2, fresh_state(B, dil))
    _assert_same(a, b)
    x2[:, n - sum(dil) - 2] = 0.25                     # the first sample of the window does
    c = step_state(w, enc, dil, P, x2, fresh_state(B, dil))
    assert max(np.abs(qa - qc).max() for qa, qc in zip(a["queues"], c["queues"])) > 0
