"""The windowing rule of chunked student synthesis on the float64 oracle: each flow run over [the last Heff rows of its
input | this call's rows], Heff = min(t0, H), gives the full-clip flows on this call's rows, where H is the flow's
dependency window (filter_width - 1) * sum(d) + filter_width rounded up to a multiple of pool_stride.  A history one
frame shorter than H changes some output: the rounding rule is needed, not merely enough.  The student.py dilations and
a set that is not powers of two with one flow and global conditions appended to the encoding."""
import numpy as np
import pytest

from conftest import f64
from oracle import srwn_oracle as orc
import sr_wavenet_b200.synth as synth

NONPOW2 = [1, 2, 4, 8, 3, 5, 7, 6]            # sum 36: window 38, H = 64 at P = 32


def history_rows(dilations, P, K=2):
    """H: the rows one output sample of a flow depends on, rounded up to whole frames."""
    need = (K - 1) * sum(dilations) + K
    return -(-need // P) * P


def _stream(w, z, enc, dil, P, F, sizes, H):
    """The chunked synthesis of csrc/student_stream.cu on the oracle: out, s_tot, mu_tot, x_last of every call."""
    B, T = z.shape
    Hf = H // P
    hist = [np.zeros((B, H)) for _ in range(F)]
    fh = np.zeros((B, Hf, enc.shape[2]))
    t0, got = 0, {k: [] for k in ("out", "s_tot", "mu_tot", "x_last")}
    for S in sizes:
        heff = min(t0, H)
        ebuf = np.concatenate([fh[:, Hf - heff // P:], enc[:, t0 // P:(t0 + S) // P]], axis=1)
        x = np.concatenate([hist[0][:, H - heff:], z[:, t0:t0 + S]], axis=1)
        inputs, scales, means = [], [], []
        for f in range(F):
            inputs.append(x)
            s, m, y = orc.student_flow(w, x[:, :, None], ebuf, dil, P, f)
            scales.append(s[:, heff:, 0])
            means.append(m[:, heff:, 0])
            x = np.concatenate([hist[f + 1][:, H - heff:], y[:, heff:, 0]], axis=1) if f + 1 < F else y
        s_tot, mu_tot = np.ones((B, S)), np.zeros((B, S))
        for i in range(F):
            s_tot = s_tot * scales[i]
            mu = means[i]
            for j in range(i + 1, F):
                mu = mu * scales[j]
            mu_tot = mu_tot + mu
        zc = z[:, t0:t0 + S]
        got["out"].append(np.clip(zc * s_tot + mu_tot, -1, 1))
        got["s_tot"].append(s_tot)
        got["mu_tot"].append(mu_tot)
        got["x_last"].append(x[:, heff:, 0])
        for f in range(F):
            hist[f] = np.concatenate([hist[f], inputs[f][:, heff:]], axis=1)[:, -H:]
        fh = np.concatenate([fh, enc[:, t0 // P:(t0 + S) // P]], axis=1)[:, -Hf:]
        t0 += S
    assert t0 == T
    return {k: np.concatenate(v, axis=1) for k, v in got.items()}


def _case(dil, P, F, C, cond, B, T, seed):
    w = f64(synth.make_student_weights(dil, num_flows=F, latent_channels=C + cond, seed=seed))
    enc = synth.synthetic_encoding(B, T // P, channels=C, seed=seed + 1).astype(np.float64)
    if cond:
        g = np.random.default_rng(seed + 2).standard_normal((B, cond))
        enc = np.concatenate([enc, np.repeat(g[:, None, :], enc.shape[1], axis=1)], axis=2)
    z = synth.logistic_noise(B, T, seed=seed + 3).astype(np.float64)
    return w, z, enc


def _full(w, z, enc, dil, P, F):
    r = orc.student_network(w, z, enc, dil, P, F)
    return {k: r[k][:, :, 0] for k in ("out", "s_tot", "mu_tot", "x_last")}


def _assert_same(got, ref):
    for k in ref:
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-11, atol=1e-12, err_msg=k)


def test_history_rows():
    assert history_rows(synth.DEFAULT_DILATIONS, 128) == 3072            # (2 - 1) * 3069 + 2 = 3071 -> 24 frames
    assert history_rows(synth.DEFAULT_DILATIONS, 512) == 3072
    assert history_rows(NONPOW2, 32) == 64                               # 36 + 2 = 38 -> 2 frames
    assert history_rows(NONPOW2, 16) == 48
    assert history_rows([1, 2, 4, 8, 16, 32, 64, 128, 256, 512] * 3 + [511], 128) == 3584   # 3582 -> 28 frames


@pytest.mark.parametrize("sizes", [[32] * 16, [96, 32, 64, 160, 160], [64, 448], [512]])
def test_windowed_flows_equal_full_clip_nonpow2(sizes):
    dil, P, F, C, cond, B, T = NONPOW2, 32, 1, 4, 3, 2, 512
    H = history_rows(dil, P)
    w, z, enc = _case(dil, P, F, C, cond, B, T, seed=21)
    _assert_same(_stream(w, z, enc, dil, P, F, sizes, H), _full(w, z, enc, dil, P, F))


@pytest.mark.parametrize("sizes", [[384] * 12, [128, 2944, 1536], [4608]])
def test_windowed_flows_equal_full_clip_student_config(sizes):
    dil, P, F, C, B, T = synth.DEFAULT_DILATIONS, 128, 2, 8, 1, 4608
    H = history_rows(dil, P)
    w, z, enc = _case(dil, P, F, C, 0, B, T, seed=31)
    _assert_same(_stream(w, z, enc, dil, P, F, sizes, H), _full(w, z, enc, dil, P, F))


@pytest.mark.parametrize("dil,P,F,T,sizes", [(NONPOW2, 32, 1, 512, [128] * 4),
                                              (synth.DEFAULT_DILATIONS, 128, 1, 4608, [3072, 1536])])
def test_one_frame_short_history_differs(dil, P, F, T, sizes):
    H = history_rows(dil, P)
    w, z, enc = _case(dil, P, F, 4, 0, 1, T, seed=41)
    ref = _full(w, z, enc, dil, P, F)
    ok = _stream(w, z, enc, dil, P, F, sizes, H)
    _assert_same(ok, ref)
    short = _stream(w, z, enc, dil, P, F, sizes, H - P)
    # the sample sum(d) + 2 rows back reaches the output through every layer: a small change, but far above rounding
    d_ok, d_short = (np.abs(r["x_last"] - ref["x_last"]).max() for r in (ok, short))
    assert d_short > 1e-12 and d_short > 1e3 * d_ok
