"""Reference loops of primed generation for the tests (test infrastructure, like the oracle): the autoregressive loop of
teacher.py:153-170 seeded with real audio, x[:, :n] given instead of drawn.  Built from the oracle's functions, which
stay as they are.

* ``naive_ar_loop_primed``: the reference's loop itself, one full decoder pass per sample (O(T^2));
* ``queue_ar_primed``: the per-layer dilation-queue restatement (O(T)) forcing the same samples, with the logits of
  every step, the forced ones included."""
import numpy as np

from oracle import srwn_oracle as orc


def naive_ar_loop_primed(weights, encoding, dilations, pool_stride, num_mixtures, u1, u2, T, x_prefix):
    """``orc.naive_ar_loop`` with ``x[:, :n]`` starting as ``x_prefix`` [B,n] and kept: the loop runs i = n .. T-1."""
    B = encoding.shape[0]
    n = x_prefix.shape[1]
    x = np.zeros((B, T), dtype=encoding.dtype)
    x[:, :n] = x_prefix
    for i in range(n, T):
        x[:, i:] = 0                                                      # teacher.py:164
        logits = orc.teacher_decoder_logits(weights, x, encoding, dilations, pool_stride)
        s = orc.sample_from_discretized_mix_logistic(logits, num_mixtures, u1, u2[:, :, None])
        x[:, i] = s[:, i, 0]                                              # teacher.py:167
    return x


def queue_ar_primed(weights, encoding, dilations, pool_stride, num_mixtures, u1, u2, T, x_prefix,
                    prefix='WaveNetAutoEncoder/Decoder/'):
    """``orc.queue_ar`` (same arithmetic per step) with the first n = x_prefix.shape[1] samples forced.
    Returns (x [B,T], logits [B,T,4M])."""
    W = lambda name: weights[prefix + name]
    B = encoding.shape[0]
    dt = encoding.dtype
    L = len(dilations)
    n_prefix = x_prefix.shape[1]
    R = W('causal_conv_Kernel').shape[2]
    x = np.zeros((B, T), dtype=dt)
    all_logits = np.zeros((B, T, 4 * num_mixtures), dtype=dt)
    conds = [encoding @ W(('conv1d' if i == 0 else 'conv1d_%d' % (3 * i)) + '/kernel')[0] +
             W(('conv1d' if i == 0 else 'conv1d_%d' % (3 * i)) + '/bias') for i in range(L)]
    hist = [np.zeros((B, T, R), dtype=dt) for _ in range(L)]
    ck, cb = W('causal_conv_Kernel'), W('causal_conv_Bias').reshape(-1)
    sq = dt.type(orc.SQRT_HALF)
    for t in range(T):
        xm1 = x[:, t - 1] if t >= 1 else np.zeros(B, dt)
        xm2 = x[:, t - 2] if t >= 2 else np.zeros(B, dt)
        h = xm2[:, None] * ck[0, 0][None, :] + xm1[:, None] * ck[1, 0][None, :] + cb
        total = 0
        for i, d in enumerate(dilations):
            h = h + conds[i][:, min(t // pool_stride, conds[i].shape[1] - 1), :]
            hist[i][:, t] = h
            tap = hist[i][:, t - d] if t >= d else np.zeros_like(h)
            name = 'dilated_conv_%d' % i
            fk = W('%s_filter/%s_Kernel' % (name, name))
            fb = W('%s_filter/%s_Bias' % (name, name)).reshape(-1)
            f = np.tanh(tap @ fk[0] + h @ fk[1] + fb)
            c = f * orc.sigmoid(f)
            res = c @ W('conv1d_%d/kernel' % (3 * i + 1))[0] + W('conv1d_%d/bias' % (3 * i + 1))
            total = total + (c @ W('conv1d_%d/kernel' % (3 * i + 2))[0] + W('conv1d_%d/bias' % (3 * i + 2)))
            h = (h + res) * sq
        total = np.maximum(total, 0)
        total = np.maximum(total @ W('conv1d_%d/kernel' % (3 * L))[0] + W('conv1d_%d/bias' % (3 * L)), 0)
        logits = total @ W('conv1d_%d/kernel' % (3 * L + 1))[0] + W('conv1d_%d/bias' % (3 * L + 1))
        all_logits[:, t] = logits
        if t < n_prefix:
            x[:, t] = x_prefix[:, t]
        else:
            s = orc.sample_from_discretized_mix_logistic(logits[:, None, :], num_mixtures, u1[:, t:t + 1],
                                                         u2[:, t:t + 1, None])
            x[:, t] = s[:, 0, 0]
    return x, all_logits
