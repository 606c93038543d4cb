"""The two other users of the residual block in the reference: ``WaveNet`` (a clip classifier, model.py:8-72) and
``SiameseWaveNet`` (an embedding network trained with a contrastive loss, model.py:660-798).  Same constructor
signatures, variable names and method names; the forward passes run on the device through the C ABI's generic
kernels (``srwn_dilated_causal_conv1d``, ``srwn_residual_dilation_layer``, ``srwn_relu``, ``srwn_avg_pool_time``,
``srwn_softmax``, ``srwn_pair_distance``), torch being the memory host only.  Neither network is on the hot path of this
build (SURVEY.md 8f-4): inference, loss values and checkpoints are provided, ``train`` is not (no backward pass through
the skip path exists on the device).

Graph (both heads, model.py:33-57 / 692-713): ``h = causal_conv(x)`` (no right shift, no conditioning) -> L residual
blocks -> sum of the skip outputs -> relu -> 1x1 (skip_channels) -> relu -> 1x1 (outputs) -> average over a window of
``input_size`` time steps (``tf.nn.pool(AVG, VALID)``: one output frame when the clip is ``input_size`` long).
"""
import os
import time

import numpy as np
import torch

from . import _lib
from .model import _cuda_f32


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _BlockStack(object):
    """Variables and forward pass of ``causal_conv -> blocks -> skip sum -> two 1x1 convs -> average pool`` under one
    variable scope.  Variable names follow TF1's rules (ops.py:13-46: ``<name>_Kernel`` / ``<name>_Bias`` for the dilated
    convs, ``conv1d``, ``conv1d_1``, ... in creation order for the ``tf.layers.conv1d`` calls)."""

    def __init__(self, scope, input_size, outputs, dilations, filter_width, dilation_channels, skip_channels, seed=None):
        self.scope, self.input_size, self.outputs = scope, int(input_size), int(outputs)
        self.dilations, self.K = [int(d) for d in dilations], int(filter_width)
        self.R, self.S = int(dilation_channels), int(skip_channels)
        rng = np.random.default_rng(seed)
        self.shapes = {}
        K, R, S, L = self.K, self.R, self.S, len(self.dilations)
        self._add('causal_conv_Kernel', (K, 1, R)); self._add('causal_conv_Bias', (1, 1, R))
        for i in range(L):
            n = 'dilated_conv_%d' % i
            for part in ('filter', 'gate'):                    # the gate conv is dead (ops.py:31-33) but exists in checkpoints
                self._add('%s_%s/%s_Kernel' % (n, part, n), (K, R, R)); self._add('%s_%s/%s_Bias' % (n, part, n), (1, 1, R))
            self._add(self._layer(2 * i) + '/kernel', (1, R, R)); self._add(self._layer(2 * i) + '/bias', (R,))
            self._add(self._layer(2 * i + 1) + '/kernel', (1, R, S)); self._add(self._layer(2 * i + 1) + '/bias', (S,))
        self._add(self._layer(2 * L) + '/kernel', (1, S, S)); self._add(self._layer(2 * L) + '/bias', (S,))
        self._add(self._layer(2 * L + 1) + '/kernel', (1, S, self.outputs)); self._add(self._layer(2 * L + 1) + '/bias', (self.outputs,))
        self.host, self._dev_vars = {}, None
        for name, shape in self.shapes.items():                # Xavier-uniform kernels, zero biases (ops.py:15,18; tf.layers defaults)
            if name.endswith('ias'):
                self.host[name] = np.zeros(shape, np.float32)
            else:
                k, cin, cout = shape
                lim = np.sqrt(6.0 / (k * cin + k * cout))
                self.host[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)

    @staticmethod
    def _layer(i):
        return 'conv1d' if i == 0 else 'conv1d_%d' % i

    def _add(self, name, shape):
        self.shapes[self.scope + '/' + name] = tuple(shape)

    def variable_names(self):
        return list(self.shapes)

    def set_weights(self, weights, strict=True):
        for name, shape in self.shapes.items():
            if name not in weights:
                if strict and '_gate/' not in name:
                    raise KeyError("missing variable %s" % name)
                continue
            a = np.asarray(weights[name], dtype=np.float32)
            if tuple(a.shape) != shape:
                raise ValueError("variable %s has shape %s, expected %s" % (name, a.shape, shape))
            self.host[name] = np.ascontiguousarray(a)
        self._dev_vars = None

    def get_weights(self):
        return {k: v.copy() for k, v in self.host.items()}

    @property
    def vars(self):
        """The variables on the device (uploaded on first use; the product path has no CPU fallback)."""
        if self._dev_vars is None:
            self._dev_vars = {k: torch.from_numpy(v).cuda() for k, v in self.host.items()}
        return self._dev_vars

    def forward(self, inputs):
        """inputs [B, T] -> pooled [B, T - input_size + 1, outputs] (fp32 CUDA tensor)."""
        lib = _lib.load()
        x = _cuda_f32(inputs)
        if x.ndim != 2:
            raise ValueError("inputs must be [batch, time]")
        B, T = x.shape
        if T < self.input_size:
            raise ValueError("clips must be at least input_size = %d samples long" % self.input_size)
        v, sc, st = self.vars, self.scope + '/', _stream()
        K, R, S, L = self.K, self.R, self.S, len(self.dilations)
        h = torch.empty(B, T, R, dtype=torch.float32, device="cuda")
        _lib.check(lib.srwn_dilated_causal_conv1d(x.data_ptr(), v[sc + 'causal_conv_Kernel'].data_ptr(), v[sc + 'causal_conv_Bias'].data_ptr(),
                                                  h.data_ptr(), B, T, 1, R, K, 1, st))
        total = torch.empty(B, T, S, dtype=torch.float32, device="cuda")
        skip = torch.empty_like(total)
        h2 = torch.empty_like(h)
        for i, d in enumerate(self.dilations):
            n = 'dilated_conv_%d' % i
            dst = total if i == 0 else skip
            _lib.check(lib.srwn_residual_dilation_layer(
                h.data_ptr(), v[sc + '%s_filter/%s_Kernel' % (n, n)].data_ptr(), v[sc + '%s_filter/%s_Bias' % (n, n)].data_ptr(),
                v[sc + self._layer(2 * i) + '/kernel'].data_ptr(), v[sc + self._layer(2 * i) + '/bias'].data_ptr(),
                v[sc + self._layer(2 * i + 1) + '/kernel'].data_ptr(), v[sc + self._layer(2 * i + 1) + '/bias'].data_ptr(),
                h2.data_ptr(), dst.data_ptr(), B, T, R, S, K, d, st))
            if i > 0:
                _lib.check(lib.srwn_axpy(total.data_ptr(), skip.data_ptr(), 1.0, total.numel(), st))      # tf.reduce_sum(skip_layers, axis=0)
            h, h2 = h2, h
        _lib.check(lib.srwn_relu(total.data_ptr(), total.numel(), st))
        t1 = skip if L > 0 else torch.empty_like(total)
        _lib.check(lib.srwn_dilated_causal_conv1d(total.data_ptr(), v[sc + self._layer(2 * L) + '/kernel'].data_ptr(),
                                                  v[sc + self._layer(2 * L) + '/bias'].data_ptr(), t1.data_ptr(), B, T, S, S, 1, 1, st))
        _lib.check(lib.srwn_relu(t1.data_ptr(), t1.numel(), st))
        t2 = torch.empty(B, T, self.outputs, dtype=torch.float32, device="cuda")
        _lib.check(lib.srwn_dilated_causal_conv1d(t1.data_ptr(), v[sc + self._layer(2 * L + 1) + '/kernel'].data_ptr(),
                                                  v[sc + self._layer(2 * L + 1) + '/bias'].data_ptr(), t2.data_ptr(), B, T, S, self.outputs, 1, 1, st))
        out_len = T - self.input_size + 1
        pooled = torch.empty(B, out_len, self.outputs, dtype=torch.float32, device="cuda")
        _lib.check(lib.srwn_avg_pool_time(t2.data_ptr(), pooled.data_ptr(), B, T, self.outputs, self.input_size, st))
        return pooled


def _no_train(cls):
    raise NotImplementedError("%s.train: this build has no backward pass through the skip path of the residual stack "
                              "(only the student's distillation step trains on the device); predict / loss / checkpoints work" % cls)


class WaveNet(object):
    """model.py:8-72.  ``predict(inputs)`` = softmax of the pooled logits [B, 1, output_channels]; ``loss(inputs, targets)`` =
    mean softmax cross-entropy against ``targets`` [B, output_size] (model.py:24-29)."""

    def __init__(self, input_size, output_size, dilations, filter_width=2, dilation_channels=32, skip_channels=256,
                 output_channels=256, name='WaveNet', learning_rate=0.001):
        self.input_size, self.output_size, self.dilations = input_size, output_size, dilations
        self.filter_width, self.dilation_channels, self.skip_channels = filter_width, dilation_channels, skip_channels
        self.output_channels, self.learning_rate = output_channels, learning_rate
        self._net = _BlockStack(name, input_size, output_channels, dilations, filter_width, dilation_channels, skip_channels)
        self.network_params = self._net.variable_names()

    def set_weights(self, weights, strict=True):
        self._net.set_weights(weights, strict)

    def get_weights(self):
        return self._net.get_weights()

    def get_logits(self, inputs):
        return self._net.forward(inputs)

    def predict(self, inputs):
        lg = self._net.forward(inputs)
        out = torch.empty_like(lg)
        _lib.check(_lib.load().srwn_softmax(lg.data_ptr(), out.data_ptr(), lg.shape[0] * lg.shape[1], lg.shape[2], _stream()))
        return out.cpu().numpy()

    def loss(self, inputs, targets):
        """tf.reduce_mean(softmax_cross_entropy_with_logits_v2(logits, expand_dims(targets, 1))) -- a few numbers, on the host."""
        lg = self._net.forward(inputs).cpu().numpy().astype(np.float64)
        y = np.asarray(targets, dtype=np.float64)[:, None, :]
        m = lg.max(-1, keepdims=True)
        logp = lg - m - np.log(np.exp(lg - m).sum(-1, keepdims=True))
        return float(np.mean(-(y * logp).sum(-1)))

    def train(self, inputs, targets):
        _no_train("WaveNet")


class SiameseWaveNet(object):
    """model.py:660-798.  Both branches share the variables under ``<name>/siamese``; methods keep the reference's explicit
    ``sess`` first argument (ignored: there is no TF session)."""

    def __init__(self, input_size, output_dimensions, dilations, margin=5.0, filter_width=2, dilation_channels=32,
                 skip_channels=256, name='SiameseWaveNet', learning_rate=0.001):
        self.input_size, self.output_dimensions, self.dilations, self.margin = input_size, output_dimensions, dilations, margin
        self.filter_width, self.dilation_channels, self.skip_channels = filter_width, dilation_channels, skip_channels
        self.learning_rate = learning_rate
        self._net = _BlockStack(name + '/siamese', input_size, output_dimensions, dilations, filter_width, dilation_channels, skip_channels)
        self.network_params = self._net.variable_names()
        self.last_checkpoint_time = time.time()

    def set_weights(self, weights, strict=True):
        self._net.set_weights(weights, strict)

    def get_weights(self):
        return self._net.get_weights()

    def get_embedding(self, sess, inputs):
        return self._net.forward(inputs).cpu().numpy()

    def _distance(self, inputs_left, inputs_right):
        el, er = self._net.forward(inputs_left), self._net.forward(inputs_right)
        if el.shape[1] != 1:
            raise ValueError("distance needs clips of exactly input_size samples (tf.squeeze(embedding, 1), model.py:731)")
        B, D = el.shape[0], el.shape[2]
        d = torch.empty(B, dtype=torch.float32, device="cuda")
        _lib.check(_lib.load().srwn_pair_distance(el.data_ptr(), er.data_ptr(), d.data_ptr(), B, D, _stream()))
        return d

    def get_distance(self, sess, inputs_left, inputs_right):
        return self._distance(inputs_left, inputs_right).cpu().numpy()

    def loss(self, sess, inputs_left, inputs_right, labels):
        """Contrastive loss (model.py:745-749; label 1 = same, 0 = different) and the distances."""
        d = self._distance(inputs_left, inputs_right).cpu().numpy().astype(np.float64)
        y = np.asarray(labels, dtype=np.float64)
        losses = y * 0.5 * d ** 2 + (1 - y) * 0.5 * np.maximum(0.0, float(self.margin) - d) ** 2
        return float(losses.mean()), d.astype(np.float32)

    def train(self, sess, inputs_left, inputs_right, labels):
        _no_train("SiameseWaveNet")

    def save(self, sess, logdir, global_step, force=False):
        """TF1 tensor-bundle checkpoint of the network variables, throttled to one per minute like the reference (model.py:767-775)."""
        if not (force or time.time() - self.last_checkpoint_time > 60):
            return False
        from . import tf_checkpoint
        os.makedirs(logdir, exist_ok=True)
        path = os.path.join(logdir, 'model.ckpt-%d' % global_step)
        tf_checkpoint.write_checkpoint(path, self.get_weights())
        with open(os.path.join(logdir, 'checkpoint'), 'w') as f:
            f.write('model_checkpoint_path: "%s"\n' % os.path.basename(path))
        self.last_checkpoint_time = time.time()
        return True

    def load(self, sess, logdir):
        from . import tf_checkpoint
        if logdir is None or not os.path.exists(logdir):
            return None
        path = tf_checkpoint.latest_checkpoint(logdir)
        if path is None:
            return None
        try:
            self.set_weights(tf_checkpoint.read_checkpoint(path))
        except (KeyError, FileNotFoundError):
            print('Could not find checkpoint at %s' % path)
            return False
        print('Restoring previous session')
        return True
