"""Reference of the parallel prefill for the tests (test infrastructure, like the oracle): the generation state after n
known samples, computed two ways from the oracle's functions.

A state is (t0, x history, queues): ``xh[b] = (x[t0-1], x[t0-2])`` and ``queues[l][b, s]`` holding layer l's input at the
position p in [t0 - d_l, t0) with p mod d_l = s (zero before position 0, the zero padding of ops.py:9).

* ``step_state``: the queue loop of ``primed_ar.queue_ar_primed`` stepped over the n samples with every one forced;
* ``prefill_state``: the window restatement.  It computes layer l only over the last D_l = d_l + ... + d_{L-1} positions
  and layer 0 from the last D_0 + 2 samples, reading taps and x before t0 from the prior state, and vectorises each layer
  over time."""
import numpy as np

from oracle import srwn_oracle as orc

_PFX = 'WaveNetAutoEncoder/Decoder/'


def _layers(weights, encoding, dilations):
    W = lambda name: weights[_PFX + name]
    conds = [encoding @ W(('conv1d' if i == 0 else 'conv1d_%d' % (3 * i)) + '/kernel')[0] +
             W(('conv1d' if i == 0 else 'conv1d_%d' % (3 * i)) + '/bias') for i in range(len(dilations))]
    layers = []
    for i in range(len(dilations)):
        name = 'dilated_conv_%d' % i
        layers.append((W('%s_filter/%s_Kernel' % (name, name)), W('%s_filter/%s_Bias' % (name, name)).reshape(-1),
                       W('conv1d_%d/kernel' % (3 * i + 1))[0], W('conv1d_%d/bias' % (3 * i + 1))))
    return conds, layers, W('causal_conv_Kernel'), W('causal_conv_Bias').reshape(-1)


def fresh_state(B, dilations, R=32):
    return {"t0": 0, "xh": np.zeros((B, 2)), "queues": [np.zeros((B, d, R)) for d in dilations]}


def _copy(state):
    return {"t0": state["t0"], "xh": state["xh"].copy(), "queues": [q.copy() for q in state["queues"]]}


def _layer(h, tap, lw):
    fk, fb, rk, rb = lw
    f = np.tanh(tap @ fk[0] + h @ fk[1] + fb)
    c = f * orc.sigmoid(f)
    return (h + c @ rk + rb) * orc.SQRT_HALF


def step_state(weights, encoding, dilations, pool_stride, x, state):
    """Steps t = 0 .. n-1 (positions t0 + t) forcing x [B,n]; encoding [B,ceil(n/P),C] are the frames of those steps."""
    conds, layers, ck, cb = _layers(weights, encoding, dilations)
    s = _copy(state)
    t0, xm1, xm2 = s["t0"], s["xh"][:, 0].copy(), s["xh"][:, 1].copy()
    for t in range(x.shape[1]):
        h = xm2[:, None] * ck[0, 0][None, :] + xm1[:, None] * ck[1, 0][None, :] + cb
        for i, d in enumerate(dilations):
            h = h + conds[i][:, t // pool_stride, :]
            slot = (t0 + t) % d
            tap = s["queues"][i][:, slot].copy()
            s["queues"][i][:, slot] = h
            h = _layer(h, tap, layers[i])
        xm2, xm1 = xm1, x[:, t].copy()
    s["t0"] = t0 + x.shape[1]
    s["xh"] = np.stack([xm1, xm2], axis=1)
    return s


def prefill_state(weights, encoding, dilations, pool_stride, x, state, return_rows=False):
    """The same state from the window only.  With return_rows, also the number of (utterance-independent) positions
    computed per layer."""
    conds, layers, ck, cb = _layers(weights, encoding, dilations)
    s = _copy(state)
    B, n = x.shape
    t0, L = s["t0"], len(dilations)
    D = [int(sum(dilations[l:])) for l in range(L + 1)]
    lo = max(0, n - D[0])
    pos = np.arange(lo, n)
    xx = lambda p: np.where(p[None, :] >= 0, x[:, np.maximum(p, 0)], s["xh"][:, np.clip(-1 - p, 0, 1)])
    fr = lambda p: p // pool_stride
    h = (xx(pos - 2)[:, :, None] * ck[0, 0] + xx(pos - 1)[:, :, None] * ck[1, 0] + cb) + conds[0][:, fr(pos)]
    rows = [len(pos)]
    for l, d in enumerate(dilations):
        # h holds layer l's input over positions pos = [max(0, n - D_l), n)
        q_old = s["queues"][l]
        if l + 1 < L:
            out = np.arange(max(0, n - D[l + 1]), n)
            cur = h[:, out - pos[0]]
            tp = out - d
            tap = np.where((tp >= 0)[None, :, None], h[:, np.maximum(tp - pos[0], 0)], q_old[:, (t0 + out) % d])
            h_next = _layer(cur, tap, layers[l]) + conds[l + 1][:, fr(out)]
            rows.append(len(out))
        keep = np.arange(max(0, n - d), n)
        q_new = q_old.copy()
        q_new[:, (t0 + keep) % d] = h[:, keep - pos[0]]
        s["queues"][l] = q_new
        if l + 1 < L:
            h, pos = h_next, out
    s["t0"] = t0 + n
    s["xh"] = np.stack([x[:, n - 1], x[:, n - 2] if n >= 2 else s["xh"][:, 0]], axis=1)
    return (s, rows) if return_rows else s
