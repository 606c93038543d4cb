"""Python-facing mirror of the reference's ``model.py`` for the hot path: same class names,
constructor arguments and method names/argument meaning as ``WaveNetAutoEncoder``
(model.py:75-285) and ``ParallelWaveNet`` (model.py:290-656).  Each former ``sess.run`` is one
call into libsrwn.so (include/srwn.h).  Like the reference's ``feed_dict`` boundary, methods take
NumPy arrays (or torch tensors) and return NumPy arrays; CUDA tensors in -> CUDA tensors out,
with no host copies (used for device-resident benchmarking).

The teacher encoder (``encode`` / ``reconstruct``, SURVEY.md 8(f)-1) runs through its own handle
(``srwn_encoder_*``); teacher training (``train``) raises NotImplementedError.
"""
import ctypes
import os
import time

import numpy as np
import torch

from . import _lib, synth, tf_checkpoint


def _as_i32_array(values):
    arr = (ctypes.c_int32 * len(values))(*[int(v) for v in values])
    return arr


def _f32(a):
    """NumPy array or tensor -> contiguous fp32 tensor; host data stays on the host."""
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    return t.float().contiguous()


def _cuda_f32(a):
    """NumPy array or tensor -> contiguous fp32 CUDA tensor (a tensor that already is one is returned as it is)."""
    return _f32(a).cuda()


class _Workspace(object):
    """Caller-side device workspace of a library call: grows to the largest size asked of it and is never shrunk."""

    def __init__(self):
        self._buf = None

    def get(self, query, *args):
        """(pointer, bytes) of at least the size ``query(*args, &n)`` reports."""
        n = ctypes.c_size_t()
        _lib.check(query(*args, ctypes.byref(n)))
        if self._buf is None or self._buf.numel() < n.value:
            self._buf = None             # release the old buffer before the larger one is allocated
            self._buf = torch.empty(max(n.value, 256), dtype=torch.uint8, device="cuda")
        return self._buf.data_ptr(), self._buf.numel()


class _Handle(object):
    """One libsrwn handle: its lifetime, weight upload and commit, workspace and profiling switch.  The decoder and the
    encoder handle (include/srwn.h) differ only in the names of the entry points they pass in: create, destroy,
    set_weight, commit and set_profiling."""

    def __init__(self, what, cfg, entry_points):
        lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("the SR-WaveNet %s needs a CUDA device (no CPU fallback)" % what)
        create, self._destroy, self._set_weight, self._commit, self._set_profiling = (getattr(lib, n) for n in entry_points)
        h = ctypes.c_void_p()
        _lib.check(create(ctypes.byref(cfg), ctypes.byref(h)))
        self.lib, self.h = lib, h
        self._ws = _Workspace()

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self._destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_weights(self, weights):
        for name, arr in weights.items():
            a = np.ascontiguousarray(arr, dtype=np.float32)
            shape = (ctypes.c_int64 * a.ndim)(*a.shape)
            _lib.check(self._set_weight(self.h, name.encode(), a.ctypes.data_as(ctypes.c_void_p), shape, a.ndim))
        _lib.check(self._commit(self.h, _stream()))

    def set_profiling(self, enable):
        _lib.check(self._set_profiling(self.h, int(bool(enable))))


class _Engine(_Handle):
    """Owns one libsrwn handle plus the caller-side workspace and pinned staging buffers."""

    def __init__(self, kind, dilations, filter_width, dilation_channels, skip_channels, cond_channels,
                 pool_stride, num_mixtures=0, num_flows=0):
        self._dil = _as_i32_array(dilations)
        cfg = _lib.Config(kind, len(dilations), self._dil, filter_width, dilation_channels, skip_channels,
                          cond_channels, pool_stride, num_mixtures, num_flows)
        _Handle.__init__(self, "hot path", cfg, ("srwn_create", "srwn_destroy", "srwn_set_weight",
                                                 "srwn_commit_weights", "srwn_set_profiling"))
        self.kind = kind
        self.cond_channels = cond_channels
        self.pool_stride = pool_stride
        self._pinned = {}

    def check_encoding(self, e, B, T):
        """The library reads ``cond_channels`` floats for each of the T / pool_stride frames of each of the B rows and
        knows nothing else of the encoding's shape, so it is checked here, before any launch."""
        if e.ndim != 3 or e.shape[0] != B or e.shape[2] != self.cond_channels:
            raise ValueError("encoding must be [B, T/pool_stride, %d]" % self.cond_channels)
        if e.shape[1] * self.pool_stride != T:
            raise ValueError("T=%d must equal pool_stride * frames = %d (model.py:183)"
                             % (T, e.shape[1] * self.pool_stride))

    def get_weight(self, name, shape):
        out = np.empty(shape, dtype=np.float32)
        _lib.check(self.lib.srwn_get_weight(self.h, name.encode(), out.ctypes.data_as(ctypes.c_void_p), out.size))
        return out

    def last_kernel_ms(self):
        """(elapsed ms, launches, kernel name) of the dominant kernel(s) of the last call."""
        ms, n, name = ctypes.c_float(), ctypes.c_int32(), ctypes.c_char_p()
        _lib.check(self.lib.srwn_last_kernel_ms(self.h, ctypes.byref(ms), ctypes.byref(n), ctypes.byref(name)))
        return ms.value, n.value, name.value.decode()

    def random_uniform(self, shape, seed, stream_id, lo, hi):
        """U(lo, hi) draws on the device (Philox, csrc/philox.cuh) for the sampler's noise (ops.py:187, 196)."""
        out = torch.empty(shape, dtype=torch.float32, device="cuda")
        _lib.check(self.lib.srwn_random_uniform(out.data_ptr(), out.numel(), seed, stream_id, lo, hi, _stream()))
        return out

    def set_team_size(self, ctas_per_team):
        """CTAs per team of the fused kernel (0 = chosen per (B, T)); results do not depend on it."""
        _lib.check(self.lib.srwn_set_team_size(self.h, int(ctas_per_team)))

    def last_partition(self):
        """(teams, CTAs per team) of the last fused call."""
        t, g = ctypes.c_int32(), ctypes.c_int32()
        _lib.check(self.lib.srwn_last_partition(self.h, ctypes.byref(t), ctypes.byref(g)))
        return t.value, g.value

    def check_async(self, op, B, T, precision):
        """Synchronises and raises if the last fused launch aborted on the device."""
        ws, wsn = self.workspace(op, B, T, precision)
        _lib.check(self.lib.srwn_check_async_error(self.h, op, B, T, precision, ws, wsn,
                                                   torch.cuda.current_stream().cuda_stream))

    def workspace(self, op, B, T, precision):
        return self._ws.get(self.lib.srwn_workspace_bytes, self.h, op, B, T, precision)

    def to_device(self, a, key):
        """NumPy / CPU tensor -> CUDA fp32 tensor through a persistent pinned staging buffer."""
        t = _f32(a)
        if t.is_cuda:
            return t, True
        if not t.is_pinned():
            buf, ev = self._pinned.get(key, (None, None))
            if buf is None or buf.shape != t.shape:
                buf, ev = torch.empty(t.shape, dtype=torch.float32, pin_memory=True), torch.cuda.Event()
                self._pinned[key] = (buf, ev)
            else:
                ev.synchronize()        # the previous H2D copy out of this staging buffer may still be queued
            buf.copy_(t)
            d = buf.to("cuda", non_blocking=True)
            ev.record()
            return d, False
        return t.to("cuda", non_blocking=True), False

    def to_host(self, t, on_device):
        if on_device:
            return t
        key = ("out", tuple(t.shape), t.dtype)
        buf = self._pinned.get(key)
        if buf is None:
            buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            self._pinned[key] = buf
        buf.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return buf.numpy().copy()

    def finish(self, t, on_dev, op, B, T, precision):
        """Result hand-over of a call ``op`` over [B, T] at ``precision``.  Host boundary (NumPy in -> NumPy out): the copy
        synchronises anyway, so a fused launch that aborted on the device raises here instead of returning partial data.
        Device-resident results are not synchronised; an abort then refuses the NEXT call on the handle (pinned abort
        words, include/srwn.h)."""
        out = self.to_host(t, on_dev)
        if not on_dev and (precision != _lib.FP32 or op == _lib.OP_STUDENT_STREAM):    # a stream call checks its t0 in both
            self.check_async(op, B, T, precision)
        return out


class _EncoderEngine(_Handle):
    """Owns one libsrwn encoder handle (include/srwn.h, srwn_encoder_*) and its workspace."""

    def __init__(self, n_layers, filter_width, encoder_channels, skip_channels, latent_channels, pool_stride):
        cfg = _lib.EncoderConfig(n_layers, filter_width, encoder_channels, skip_channels, latent_channels,
                                 pool_stride)
        _Handle.__init__(self, "encoder", cfg, ("srwn_encoder_create", "srwn_encoder_destroy", "srwn_encoder_set_weight",
                                                "srwn_encoder_commit", "srwn_encoder_set_profiling"))
        self.latent_channels, self.pool_stride = latent_channels, pool_stride

    def supports(self, prec):
        return bool(self.lib.srwn_encoder_supports(self.h, prec))

    def last_ms(self):
        ms = ctypes.c_float()
        _lib.check(self.lib.srwn_encoder_last_ms(self.h, ctypes.byref(ms)))
        return ms.value

    def encode(self, x, prec, check=True):
        """x: CUDA fp32 [B,T] -> CUDA fp32 [B, T // P, latent]."""
        B, T = x.shape
        ws, wsn = self._ws.get(self.lib.srwn_encoder_workspace_bytes, self.h, B, T, prec)
        out = torch.empty(B, T // self.pool_stride, self.latent_channels, dtype=torch.float32, device="cuda")
        _lib.check(self.lib.srwn_teacher_encode(self.h, x.data_ptr(), out.data_ptr(), B, T, prec, ws, wsn, _stream()))
        if check and prec != _lib.FP32:
            _lib.check(self.lib.srwn_encoder_check_async_error(self.h, B, T, prec, ws, wsn, _stream()))
        return out


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _with_conditions(encoding, conditions, condition_size):
    """model.py:161-167 / 495-500: tile the global condition over frames and concatenate."""
    if condition_size > 0:
        if conditions is None:
            raise ValueError("condition_size > 0 needs `conditions`")
        if isinstance(encoding, torch.Tensor):
            c = torch.as_tensor(conditions, dtype=torch.float32, device=encoding.device)
            return torch.cat([encoding, c[:, None, :].expand(-1, encoding.shape[1], -1)], dim=2)
        c = np.asarray(conditions, dtype=np.float32)
        return np.concatenate([encoding, np.tile(c[:, None, :], [1, encoding.shape[1], 1])], axis=2)
    return encoding


class _Model(object):
    """What the teacher and the student share: Glorot-initialised weights with zero biases, the host copy of the weights
    that ``get_weights`` returns, the precisions the engine offers, and the stand-in for tf.train.Saver
    (model.py:217-239).  ``save`` writes ``<logdir>/model.ckpt-<step>.npz`` (name-keyed,
    TF variable names) plus the ``checkpoint`` state file, throttled to once per 60 s unless ``force``; with
    ``checkpoint_format = "tf"`` it writes a TensorFlow tensor bundle (``.index`` + ``.data-00000-of-00001``) instead.
    ``load`` restores whichever of the two the state file points to, so a checkpoint directory written by the
    reference's Saver loads as it is (``tf_checkpoint.py``; optimizer slots and other variables the graph does not have
    are ignored)."""

    checkpoint_format = "npz"

    def _init_weights(self, w):
        for k in w:                      # TF initialises biases to zero (ops.py:18, tf.layers default)
            if k.endswith('Bias') or k.endswith('/bias'):
                w[k][...] = 0
        self._weights = {}
        self.set_weights(w)

    def _mirror_weights(self, weights):
        self._weights.update({k: np.array(v, dtype=np.float32) for k, v in weights.items()})

    def available_precisions(self):
        op = _lib.OP_TEACHER_LOGITS if self._eng.kind == _lib.TEACHER else _lib.OP_STUDENT_FORWARD
        return ["fp32", "fp16"] if self._eng.lib.srwn_supports(self._eng.h, op, _lib.FP16) else ["fp32"]

    def _save(self, logdir, global_step, force):
        if force or time.time() - self.last_checkpoint_time > 60:
            if not os.path.isdir(logdir):
                os.makedirs(logdir)
            path = os.path.join(logdir, 'model.ckpt-%d' % global_step)
            if self.checkpoint_format == "tf":
                tf_checkpoint.write_checkpoint(path, self.get_weights())
            else:
                np.savez(path + '.npz', **self.get_weights())
            if isinstance(self, WaveNetAutoEncoder):      # tf.train.Saver.save also exports the meta-graph the student imports
                from . import tf_meta
                tf_meta.write_meta(path + '.meta', *tf_meta.teacher_meta_skeleton(self.name))
            with open(os.path.join(logdir, 'checkpoint'), 'w') as f:
                f.write('model_checkpoint_path: "%s"\n' % os.path.basename(path))
            self.last_checkpoint_time = time.time()
            return True
        return False

    def _load(self, logdir):
        if logdir is not None and os.path.exists(logdir):
            path = tf_checkpoint.latest_checkpoint(logdir)
            if path is not None:
                if os.path.exists(path + '.npz'):
                    with np.load(path + '.npz') as z:
                        self.set_weights({k: z[k] for k in z.files})
                elif os.path.exists(path + '.index'):
                    known = self.get_weights()
                    found = {k: v for k, v in tf_checkpoint.read_checkpoint(path).items()
                             if k in known and tuple(v.shape) == tuple(known[k].shape)}
                    if not found:
                        print('No variable of this graph in %s' % path)
                        return False
                    self.set_weights(found)
                else:
                    print('Could not find checkpoint at %s' % path)
                    return False
                print('Restoring previous session')
                return True
        return None


class WaveNetAutoEncoder(_Model):
    """model.py:75-285: decoder (the hot path) and encoder; constructor signature kept verbatim."""

    def __init__(self, input_size, condition_size, num_mixtures, dilations, filter_width=2,
                 encoder_channels=128, dilation_channels=32, skip_channels=256, latent_channels=16,
                 pool_stride=512, name='WaveNetAutoEncoder', learning_rate=0.001):
        self.input_size = input_size
        self.condition_size = condition_size
        self.num_mixtures = num_mixtures
        self.dilations = list(dilations)
        self.filter_width = filter_width
        self.encoder_channels = encoder_channels
        self.dilation_channels = dilation_channels
        self.skip_channels = skip_channels
        self.latent_channels = latent_channels
        self.pool_stride = pool_stride
        self.name = name
        self.learning_rate = learning_rate
        self.precision = "fp32"
        self.seed = int.from_bytes(os.urandom(7), "little")      # the reference's RNG is unseeded (SURVEY F10); set for reproducible draws
        self._noise_calls = 0
        self.last_checkpoint_time = time.time()
        self.createNetwork()

    # -- graph construction stand-ins ------------------------------------------------------
    def createNetwork(self):
        """model.py:202-215: the reference builds placeholders + encoder + two decoder instances;
        here it creates the decoder engine and Glorot-initialised variables."""
        self._eng = _Engine(_lib.TEACHER, self.dilations, self.filter_width, self.dilation_channels,
                            self.skip_channels, self.latent_channels + self.condition_size,
                            self.pool_stride, num_mixtures=self.num_mixtures)
        w = synth.make_teacher_weights(self.dilations, self.filter_width, self.dilation_channels,
                                       self.skip_channels, self.latent_channels + self.condition_size,
                                       self.num_mixtures, seed=None, dead_vars=True)
        self._enc_eng = _EncoderEngine(len(self.dilations), self.filter_width, self.encoder_channels,
                                       self.skip_channels, self.latent_channels, self.pool_stride)
        we = synth.make_encoder_weights(len(self.dilations), self.filter_width, self.encoder_channels,
                                        self.skip_channels, self.latent_channels, seed=None, gain=1.0)
        w.update(we)
        self._init_weights(w)

    def createEncoder(self, h, reuse=False, precision=None):
        """model.py:137-155 -> encoding [B, T/pool_stride, latent].  h [B,T,1] or [B,T]."""
        h2 = h[..., 0] if getattr(h, "ndim", 2) == 3 else h
        return self.encode(h2, precision=precision)

    def createDecoder(self, truth, encoding, conditions, reuse=False, u1=None, u2=None, precision=None):
        """model.py:158-200 -> (logits [B,T,4M], out [B,T]).  truth [B,T,1] or [B,T]."""
        from . import ops
        truth2 = truth[..., 0] if getattr(truth, "ndim", 2) == 3 else truth
        logits = self.get_logits(truth2, encoding, conditions, precision=precision)
        out = ops.sample_from_discretized_mix_logistic(logits, self.num_mixtures, u1, u2)
        out = out[..., 0]
        if not isinstance(logits, torch.Tensor):
            out = out.cpu().numpy()
        return logits, out

    # -- weights -----------------------------------------------------------------------------
    def set_weights(self, weights):
        """name -> ndarray with TF variable names (``WaveNetAutoEncoder/Decoder/...`` and
        ``WaveNetAutoEncoder/Encoder/...``); either half may be given alone."""
        dec = {k: v for k, v in weights.items() if '/Encoder/' not in k}
        enc = {k: v for k, v in weights.items() if '/Encoder/' in k}
        if dec:
            self._eng.set_weights(dec)
        if enc:
            self._enc_eng.set_weights(enc)
        self._mirror_weights(weights)

    def get_weights(self):
        return dict(self._weights)

    def load(self, logdir):
        return self._load(logdir)

    def save(self, logdir, global_step, force=False):
        return self._save(logdir, global_step, force)

    @classmethod
    def from_checkpoint(cls, logdir, dilations, latent_channels, pool_stride, condition_size=0, filter_width=2,
                        dilation_channels=32, input_size=0):
        """A teacher built from a checkpoint directory alone (what ParallelWaveNet(teacher=<dir>) needs,
        model.py:323-334): mixtures, skip and encoder widths come from the stored variable shapes."""
        path = tf_checkpoint.latest_checkpoint(logdir)
        if path is None:
            raise IOError("no teacher checkpoint under %s (expected the files WaveNetAutoEncoder.save writes)" % logdir)
        L = len(dilations)
        k_head2 = '%sconv1d_%d/kernel' % (synth.TEACHER_PREFIX, 3 * L + 1)
        k_enc0 = '%snc_conv_NC/conv1d/kernel' % synth.ENCODER_PREFIX
        if os.path.exists(path + '.npz'):
            with np.load(path + '.npz') as z:
                head2, enc0 = z[k_head2].shape, z[k_enc0].shape
        else:                                              # a tf.train.Saver checkpoint (tensor bundle)
            shapes = {n: sh for n, sh, _ in tf_checkpoint.list_variables(path)}
            head2, enc0 = shapes[k_head2], shapes[k_enc0]
        t = cls(input_size=input_size, condition_size=condition_size, num_mixtures=head2[2] // 4, dilations=dilations,
                filter_width=filter_width, encoder_channels=enc0[2], dilation_channels=dilation_channels,
                skip_channels=head2[1], latent_channels=latent_channels, pool_stride=pool_stride)
        if not t.load(logdir):
            raise IOError("could not restore the teacher from %s" % logdir)
        if os.path.exists(path + '.meta'):
            # the part of tf.train.import_meta_graph(..., input_map=...) + get_collection(...)[0] (model.py:326-341) that can
            # fail: the placeholders the student re-wires and the collections it reads must exist in the teacher's graph
            from . import tf_meta
            t.meta_collections = tf_meta.check_teacher_contract(tf_meta.read_meta(path + '.meta'), t.name)
        return t

    # -- sess.run wrappers -------------------------------------------------------------------
    def train(self, inputs, conditions=None):
        raise NotImplementedError("teacher training (model.py:242-248) is outside the hot path")

    def encode(self, inputs, conditions=None, precision=None):
        """model.py:250-255 -> encoding [B, T/pool_stride, latent] (``conditions`` does not enter the
        encoder graph, model.py:212).  A ragged tail T % pool_stride is dropped like the VALID pooling
        of model.py:154 does.  The 16-bit tensor-core path needs T % 128 == 0; other lengths run fp32."""
        eng = self._enc_eng
        x, on_dev = self._eng.to_device(inputs, "x")
        prec = self._prec(precision)
        if prec != _lib.FP32 and (not eng.supports(prec) or x.shape[1] % 128 != 0):
            prec = _lib.FP32
        return self._eng.to_host(eng.encode(x, prec), on_dev)

    def reconstruct(self, inputs, conditions=None, u1=None, u2=None, precision=None):
        """model.py:257-262 -> [B,T]: encoder, then the decoder teacher-forced on the same audio, then
        parallel sampling from the logits (``self.out``)."""
        x, on_dev = self._eng.to_device(inputs, "x")
        enc = self.encode(x, precision=precision)
        out = self.reconstruct_with_encoding(x, enc, conditions, u1=u1, u2=u2, precision=precision)
        return out if on_dev else out.cpu().numpy()

    def _prec(self, precision):
        return _lib.PRECISIONS[precision or self.precision]

    def get_logits(self, inputs, encoding, conditions=None, precision=None):
        """model.py:279-285 -> logits [B,T,4M]."""
        eng = self._eng
        enc = _with_conditions(encoding, conditions, self.condition_size)
        x, on_dev = eng.to_device(inputs, "x")
        e, _ = eng.to_device(enc, "enc")
        B, T = x.shape
        eng.check_encoding(e, B, T)
        prec = self._prec(precision)
        ws, wsn = eng.workspace(_lib.OP_TEACHER_LOGITS, B, T, prec)
        logits = torch.empty(B, T, 4 * self.num_mixtures, dtype=torch.float32, device="cuda")
        _lib.check(eng.lib.srwn_teacher_logits(eng.h, x.data_ptr(), e.data_ptr(), logits.data_ptr(), B, T,
                                               prec, ws, wsn, _stream()))
        return eng.finish(logits, on_dev, _lib.OP_TEACHER_LOGITS, B, T, prec)

    def nll(self, inputs, encoding, conditions=None, scored=None, sum_all=True, precision=None):
        """``loss_encoding`` of model.py:114-115: teacher-forced mixture-of-logistics negative
        log-likelihood.  ``scored`` (default: ``inputs``) is the audio whose likelihood is taken
        (model.py:374 scores the student's output against logits of the real audio).
        Returns a Python float (sum_all=True, ops.py:172) or [B,T,1] (ops.py:175)."""
        eng = self._eng
        enc = _with_conditions(encoding, conditions, self.condition_size)
        x, on_dev = eng.to_device(inputs, "x")
        e, _ = eng.to_device(enc, "enc")
        xs = x if scored is None else eng.to_device(scored, "xs")[0]
        B, T = x.shape
        eng.check_encoding(e, B, T)
        prec = self._prec(precision)
        ws, wsn = eng.workspace(_lib.OP_TEACHER_NLL, B, T, prec)
        if sum_all:
            out = torch.empty(1, dtype=torch.float32, device="cuda")
            _lib.check(eng.lib.srwn_teacher_nll(eng.h, x.data_ptr(), e.data_ptr(), xs.data_ptr(), None,
                                                out.data_ptr(), None, B, T, prec, ws, wsn, _stream()))
            return out if on_dev else float(eng.finish(out, False, _lib.OP_TEACHER_NLL, B, T, prec)[0])
        out = torch.empty(B, T, 1, dtype=torch.float32, device="cuda")
        _lib.check(eng.lib.srwn_teacher_nll(eng.h, x.data_ptr(), e.data_ptr(), xs.data_ptr(), out.data_ptr(),
                                            None, None, B, T, prec, ws, wsn, _stream()))
        return eng.finish(out, on_dev, _lib.OP_TEACHER_NLL, B, T, prec)

    def nll_stream(self, batches, precision=None, depth=2):
        """Scores a sequence of host batches: ``batches`` yields ``(inputs [B,T], encoding [B,T/P,C])`` (NumPy arrays or CPU
        tensors, pinned or not); yields one float per batch, in order -- the value ``nll(inputs, encoding)`` returns.
        Throughput path of a scoring service: the upload of batch i+1 runs on a copy stream while batch i is scored, and the
        4-byte result of batch i is read back while batch i+1 runs, so a step costs max(copy, kernel) instead of their sum.
        ``depth`` device-side input slots (>= 2)."""
        eng = self._eng
        prec = self._prec(precision)
        depth = max(2, int(depth))
        compute = torch.cuda.current_stream()
        copy = getattr(self, "_copy_stream", None) or torch.cuda.Stream()
        self._copy_stream = copy
        slots = [dict(x=None, e=None, px=None, pe=None, up=torch.cuda.Event(), used=torch.cuda.Event(), done=torch.cuda.Event(),
                      out=torch.empty(1, dtype=torch.float32, device="cuda"), host=torch.empty(1, dtype=torch.float32, pin_memory=True))
                 for _ in range(depth)]

        def upload(slot, batch):
            x, e = _f32(batch[0]), _f32(_with_conditions(batch[1], None, self.condition_size))
            if slot["x"] is None or slot["x"].shape != x.shape or slot["e"].shape != e.shape:
                slot["x"] = torch.empty(x.shape, dtype=torch.float32, device="cuda")
                slot["e"] = torch.empty(e.shape, dtype=torch.float32, device="cuda")
                slot["px"] = torch.empty(x.shape, dtype=torch.float32, pin_memory=True)
                slot["pe"] = torch.empty(e.shape, dtype=torch.float32, pin_memory=True)
            slot["used"].synchronize() if slot.get("busy") else None      # the kernel that read this slot last has finished
            src_x, src_e = x, e
            if not x.is_pinned():
                slot["px"].copy_(x); src_x = slot["px"]
            if not e.is_pinned():
                slot["pe"].copy_(e); src_e = slot["pe"]
            with torch.cuda.stream(copy):
                slot["x"].copy_(src_x, non_blocking=True)
                slot["e"].copy_(src_e, non_blocking=True)
                slot["up"].record(copy)

        def launch(slot):
            B, T = slot["x"].shape
            eng.check_encoding(slot["e"], B, T)
            ws, wsn = eng.workspace(_lib.OP_TEACHER_NLL, B, T, prec)
            compute.wait_event(slot["up"])
            _lib.check(eng.lib.srwn_teacher_nll(eng.h, slot["x"].data_ptr(), slot["e"].data_ptr(), slot["x"].data_ptr(), None,
                                                slot["out"].data_ptr(), None, B, T, prec, ws, wsn, compute.cuda_stream))
            slot["used"].record(compute)
            slot["host"].copy_(slot["out"], non_blocking=True)
            slot["done"].record(compute)
            slot["busy"], slot["shape"] = True, (B, T)

        def collect(slot):
            slot["done"].synchronize()
            if prec != _lib.FP32:                      # abort words of that launch, without draining the launches behind it
                _lib.check(eng.lib.srwn_peek_async_error(eng.h))
            return float(slot["host"][0])

        it = iter(batches)
        pending = []                                  # slots launched, oldest first
        i = 0
        try:
            first = next(it)
        except StopIteration:
            return
        try:
            upload(slots[0], first)
            nxt = 0
            while nxt is not None:
                cur = slots[nxt]
                launch(cur)
                pending.append(cur)
                i += 1
                try:
                    batch = next(it)
                    if len(pending) == depth:         # every slot is in flight: hand the oldest result out before reusing its slot
                        yield collect(pending.pop(0))
                    nxt = i % depth
                    upload(slots[nxt], batch)
                except StopIteration:
                    nxt = None
            while pending:
                yield collect(pending.pop(0))
        finally:
            # the slots' device buffers go back to the allocator when this frame dies: nothing on the copy stream (or, when
            # the consumer stopped early or an error came up, on the compute stream) may still be using them
            copy.synchronize()
            if pending:
                compute.synchronize()

    def reconstruct_with_encoding(self, inputs, encoding, conditions=None, u1=None, u2=None,
                                  precision=None):
        """model.py:264-270 -> [B,T]: one teacher-forced pass + parallel sampling from the logits
        (``out_from_encoding``).  ``u1``/``u2`` inject the sampler's uniforms (ops.py:187,196)."""
        _, out = self.createDecoder(inputs, encoding, conditions, reuse=True, u1=u1, u2=u2,
                                    precision=precision)
        return out

    def generation_state(self, batch_size, precision="fp16"):
        """A fresh (reset) state for resumable generation of ``batch_size`` utterances: pass it to ``generate(state=...)``
        to continue a previous call instead of starting from silence."""
        return GenerationState(self._eng, batch_size, precision)

    def generate(self, encoding, conditions=None, u1=None, u2=None, num_samples=None,
                 return_logits=False, zero_last=False, precision="fp32", state=None, prefix=None):
        """Autoregressive generation, the queue-based restatement of teacher.py:153-170:
        x[t] = clip(MoL_sample(logits_t)) with logits_t from x[<t] and encoding[t // pool_stride].
        ``zero_last=True`` reproduces teacher.py:170, which zeroes the final sample of this call.
        ``precision``: "fp32" (parity-grade FFMA kernel) or "fp16" (tensor-core kernel, fp16 operands
        and queue state, fp32 accumulate / residual stream).

        ``state`` (from ``generation_state``): continue where the last call on that state stopped and advance it by
        this call's T; ``encoding``, ``u1`` and ``u2`` then cover this call's samples only.  ``prefix`` [B, n], n <= T:
        the first n samples of this call are these (real audio, teacher-forced through the queues) instead of draws;
        without ``state`` it primes a fresh state used for this call alone.  Splitting a generation into calls gives
        bit for bit the audio of one call only with injected ``u1``/``u2``: noise drawn on the device comes from a new
        Philox stream per call."""
        eng = self._eng
        enc = _with_conditions(encoding, conditions, self.condition_size)
        e, on_dev = eng.to_device(enc, "enc")
        B = e.shape[0]
        T = num_samples if num_samples is not None else e.shape[1] * self.pool_stride
        eng.check_encoding(e, B, T)
        if prefix is not None:
            xp = eng.to_device(prefix, "prefix")[0]
            if xp.ndim != 2 or xp.shape[0] != B or xp.shape[1] > T:
                raise ValueError("prefix must be [B=%d, n] with n <= T=%d, got %s" % (B, T, tuple(xp.shape)))
            if state is None:
                state = self.generation_state(B, precision)
        if state is not None and (state.batch_size != B or state.precision != precision):
            raise ValueError("state was made for batch_size=%d, precision=%r; this call has %d, %r"
                             % (state.batch_size, state.precision, B, precision))
        d1, d2 = self._draw_uniforms(B, T) if u1 is None or u2 is None else (None, None)
        u1 = d1 if u1 is None else eng.to_device(u1, "u1")[0]
        u2 = d2 if u2 is None else eng.to_device(u2, "u2")[0]
        prec = _lib.PRECISIONS[precision]
        if not eng.lib.srwn_supports(eng.h, _lib.OP_TEACHER_GENERATE, prec):
            raise RuntimeError("generate(precision=%r) is not supported for this configuration" % precision)
        ws, wsn = eng.workspace(_lib.OP_TEACHER_GENERATE, B, T, prec)
        x = torch.empty(B, T, dtype=torch.float32, device="cuda")
        logits = torch.empty(B, T, 4 * self.num_mixtures, dtype=torch.float32, device="cuda") \
            if return_logits else None
        lg_ptr = logits.data_ptr() if return_logits else None
        if state is None:
            _lib.check(eng.lib.srwn_teacher_generate(eng.h, e.data_ptr(), u1.data_ptr(), u2.data_ptr(),
                                                     x.data_ptr(), lg_ptr, B, T, prec, ws, wsn, _stream()))
        else:
            n = 0 if prefix is None else int(xp.shape[1])
            _lib.check(eng.lib.srwn_teacher_generate_resume(eng.h, state.data_ptr(), e.data_ptr(), u1.data_ptr(),
                                                            u2.data_ptr(), xp.data_ptr() if n else None, n, x.data_ptr(),
                                                            lg_ptr, B, T, prec, ws, wsn, _stream()))
        # not eng.finish: the generation kernel's abort flag lives in the workspace and is not sticky, so no later call
        # would see it; device-resident results are checked here too
        if prec != _lib.FP32:
            eng.check_async(_lib.OP_TEACHER_GENERATE, B, T, prec)
        if zero_last:
            x[:, T - 1:] = 0            # teacher.py:170
        if return_logits:
            return eng.to_host(x, on_dev), eng.to_host(logits, on_dev)
        return eng.to_host(x, on_dev)

    def prefill(self, state, audio, encoding, conditions=None):
        """Prime ``state`` with real audio in one parallel pass: afterwards it is, byte for byte, the state that
        ``generate(state=state, prefix=audio)`` over the same n samples leaves, and ``state.position()`` has advanced by
        n.  ``audio`` [B, n] (n a multiple of pool_stride) continues from the state's position; ``encoding`` [B, n/P, C]
        are its frames.  Only the last sum(dilations) + 2 samples reach the state, so a long prime costs no more than
        that window.  Produces no audio or logits (``nll`` scores a prime)."""
        eng = self._eng
        if not isinstance(state, GenerationState) or state._eng is not eng:
            raise ValueError("state must come from this model's generation_state()")
        enc = _with_conditions(encoding, conditions, self.condition_size)
        e = eng.to_device(enc, "enc")[0]
        x = eng.to_device(audio, "prefill")[0]
        B = state.batch_size
        if x.ndim != 2 or x.shape[0] != B or x.shape[1] < 1:
            raise ValueError("audio must be [B=%d, n] with n >= 1, got %s" % (B, tuple(x.shape)))
        n = int(x.shape[1])
        eng.check_encoding(e, B, n)
        prec = _lib.PRECISIONS.get(state.precision)
        if prec is None or not eng.lib.srwn_supports(eng.h, _lib.OP_TEACHER_PREFILL, prec):
            raise ValueError("prefill(precision=%r) is not supported for this configuration" % state.precision)
        ws, wsn = eng.workspace(_lib.OP_TEACHER_PREFILL, B, n, prec)
        _lib.check(eng.lib.srwn_generate_state_prefill(eng.h, state.data_ptr(), x.data_ptr(), e.data_ptr(), n, B, prec,
                                                       ws, wsn, _stream()))

    def generate_requests(self, requests, slots, chunk, precision="fp16"):
        """Continuous batching: generate many utterances of different lengths through one state of ``slots`` utterances,
        refilling the slot of each finished utterance with the next request.  A generator of ``(index, audio)``, yielded
        as each request finishes.

        A request is a dict (or just its encoding): ``encoding`` [F, latent_channels] its frames; ``conditions``
        [condition_size] when the model has them; optionally ``prime`` [n0] real samples that start the utterance (n0 a
        multiple of pool_stride, the frames cover the prime and the continuation) and ``u1`` [F*P - n0, M], ``u2``
        [F*P - n0] the sampler's uniforms for its generated samples (otherwise drawn on the device).  Its audio is the
        F*P - n0 samples after the prime, a CUDA tensor when ``encoding`` is one, else a NumPy array.

        Before each ``generate`` call of ``chunk`` samples (a multiple of pool_stride) free slots are filled in arrival
        order: primed requests through ``prefill`` of a side state (one per prime length), the others from a reset
        state, both moved in with ``GenerationState.splice``.  Each call takes every slot's frames and uniforms at that
        slot's own offset (idle slots get zeros); what a request generates past its end is dropped.  With injected
        uniforms a request's audio is bit for bit that of generating it alone (B = 1, the same prime through prefill)."""
        P, M, cs = self.pool_stride, self.num_mixtures, self.condition_size
        slots, chunk = int(slots), int(chunk)
        if slots < 1 or chunk < P or chunk % P:
            raise ValueError("slots must be positive and chunk a positive multiple of pool_stride=%d" % P)

        reqs = []
        for i, r in enumerate(requests):
            r = r if isinstance(r, dict) else {"encoding": r}
            e = _cuda_f32(r["encoding"])
            if e.ndim != 2 or e.shape[1] != self.latent_channels:
                raise ValueError("request %d: encoding must be [F, %d]" % (i, self.latent_channels))
            prime = _cuda_f32(r["prime"]).reshape(-1) if r.get("prime") is not None else None
            n0 = 0 if prime is None else int(prime.shape[0])
            need = e.shape[0] * P - n0
            if n0 % P or need < 0:
                raise ValueError("request %d: the prime (%d samples) must be a multiple of %d within the %d frames"
                                 % (i, n0, P, e.shape[0]))
            c = None
            if cs:
                if r.get("conditions") is None:
                    raise ValueError("request %d: condition_size > 0 needs `conditions`" % i)
                c = _cuda_f32(r["conditions"]).reshape(-1)
                if c.shape[0] != cs:
                    raise ValueError("request %d: conditions must be [%d]" % (i, cs))
            inj = r.get("u1") is not None or r.get("u2") is not None
            if inj:
                if r.get("u1") is None or r.get("u2") is None:
                    raise ValueError("request %d: inject both u1 and u2, or neither" % i)
                u1, u2 = _cuda_f32(r["u1"]), _cuda_f32(r["u2"]).reshape(-1)
                if tuple(u1.shape) != (need, M) or u2.shape[0] != need:
                    raise ValueError("request %d: u1 must be [%d, %d] and u2 [%d]" % (i, need, M, need))
            reqs.append({"enc": e, "prime": prime, "n0": n0, "need": need, "cond": c,
                         "u1": u1 if inj else None, "u2": u2 if inj else None,
                         "on_dev": isinstance(r["encoding"], torch.Tensor) and r["encoding"].is_cuda})
        N = len(reqs)
        if N == 0:
            return

        # every request's generation frames, uniforms and output in flat device buffers, each with one sentinel row
        # (zeros to read, a sink to write) that idle slots and samples past a request's end point at
        def flat(parts, tail_shape):
            return torch.cat([p for p in parts if p is not None and p.shape[0]] +
                             [torch.zeros((1,) + tail_shape, device="cuda")])
        fbase, ubase, obase = np.zeros(N, np.int64), np.full(N, -1, np.int64), np.zeros(N, np.int64)
        nf = nu = no = 0
        for i, r in enumerate(reqs):
            fbase[i], obase[i] = nf, no
            nf += r["need"] // P
            no += r["need"]
            if r["u1"] is not None:
                ubase[i] = nu
                nu += r["need"]
        enc_all = flat([r["enc"][r["n0"] // P:] for r in reqs], (self.latent_channels,))
        cond_all = torch.stack([r["cond"] for r in reqs] + [torch.zeros(cs, device="cuda")]) if cs else None
        u1_all = flat([r["u1"] for r in reqs], (M,))
        u2_all = flat([r["u2"] for r in reqs], ())
        out_all = torch.empty(no + 1, dtype=torch.float32, device="cuda")
        need_np = np.array([r["need"] for r in reqs], np.int64)

        main = self.generation_state(slots, precision)
        silence = self.generation_state(1, precision)           # reset, never generated on: the source of fresh slots
        slot_req = np.full(slots, -1, np.int64)                  # request in each slot, -1 idle
        slot_pos = np.zeros(slots, np.int64)                     # samples it has generated
        ar_f = torch.arange(chunk // P, device="cuda")
        ar_s = torch.arange(chunk, device="cuda")
        nxt = 0
        while True:
            # fill the free slots from the queue
            fresh, primed = [], {}
            while nxt < N and (slot_req < 0).any():
                if reqs[nxt]["need"] == 0:
                    yield nxt, self._request_audio(out_all[:0], reqs[nxt]["on_dev"])
                    nxt += 1
                    continue
                s = int(np.flatnonzero(slot_req < 0)[0])
                slot_req[s], slot_pos[s] = nxt, 0
                if reqs[nxt]["n0"]:
                    primed.setdefault(reqs[nxt]["n0"], []).append(s)
                else:
                    fresh.append(s)
                nxt += 1
            if fresh:
                main.splice(fresh, silence, [0] * len(fresh))
            for n0, rows in primed.items():
                rs = [reqs[slot_req[s]] for s in rows]
                side = self.generation_state(len(rows), precision)
                self.prefill(side, torch.stack([r["prime"] for r in rs]),
                             torch.stack([r["enc"][:n0 // P] for r in rs]),
                             conditions=torch.stack([r["cond"] for r in rs]) if cs else None)
                main.splice(rows, side)
            active = slot_req >= 0
            if not active.any():
                return
            # gather every slot's frames and uniforms at its own offset (sentinel rows for idle slots and past the end)
            rq = np.where(active, slot_req, 0)
            left = torch.from_numpy(np.where(active, need_np[rq] - slot_pos, 0)).cuda()
            pos = torch.from_numpy(slot_pos).cuda()
            fb = torch.from_numpy(fbase[rq] + slot_pos // P).cuda()
            ub = torch.from_numpy(np.where(active, ubase[rq], -1) + slot_pos).cuda()
            ob = torch.from_numpy(obase[rq] + slot_pos).cuda()
            inj = torch.from_numpy(active & (ubase[rq] >= 0)).cuda()
            fvalid = ar_f[None, :] * P < left[:, None]
            svalid = ar_s[None, :] < left[:, None]
            fidx = torch.where(fvalid, fb[:, None] + ar_f[None, :], enc_all.shape[0] - 1)
            uidx = torch.where(svalid & inj[:, None], ub[:, None] + ar_s[None, :], u2_all.shape[0] - 1)
            oidx = torch.where(svalid, ob[:, None] + ar_s[None, :], out_all.shape[0] - 1)
            enc_c = enc_all[fidx]
            u1_c, u2_c = u1_all[uidx], u2_all[uidx]
            drawn = np.flatnonzero(active & (ubase[rq] < 0))
            if drawn.size:                                         # uniforms of requests without injected ones
                d1, d2 = self._draw_uniforms(slots, chunk)
                dr = torch.from_numpy(drawn).cuda()
                u1_c[dr], u2_c[dr] = d1[dr], d2[dr]
            cond_c = cond_all[torch.from_numpy(np.where(active, slot_req, N)).cuda()] if cs else None
            x = self.generate(enc_c, conditions=cond_c, u1=u1_c, u2=u2_c, precision=precision, state=main)
            out_all[oidx.reshape(-1)] = x.reshape(-1)
            # hand out the requests that have finished and free their slots
            slot_pos[active] += chunk
            for s in np.flatnonzero(active & (slot_pos >= need_np[rq])):
                i = int(slot_req[s])
                slot_req[s] = -1
                yield i, self._request_audio(out_all[obase[i]:obase[i] + need_np[i]], reqs[i]["on_dev"])

    def _draw_uniforms(self, rows, T):
        """The sampler's two U(1e-5, 1 - 1e-5) draws (ops.py:187, 196), [rows, T, M] and [rows, T], on the device from
        Philox streams 2k and 2k + 1 of ``seed``, k counting the calls that draw: a seeded model repeats its noise."""
        self._noise_calls += 1
        lo, hi = 1e-5, 1.0 - 1e-5
        return (self._eng.random_uniform((rows, T, self.num_mixtures), self.seed, 2 * self._noise_calls, lo, hi),
                self._eng.random_uniform((rows, T), self.seed, 2 * self._noise_calls + 1, lo, hi))

    @staticmethod
    def _request_audio(x, on_dev):
        return x.clone() if on_dev else x.cpu().numpy()


class GenerationState(object):
    """Device buffer that carries autoregressive generation from one ``generate`` call to the next: the dilation queues,
    the last two samples and the position of each utterance (include/srwn.h, srwn_generate_state_*).  Created reset."""

    def __init__(self, eng, batch_size, precision="fp16"):
        self._eng = eng
        self.batch_size, self.precision = int(batch_size), precision
        self._prec = _lib.PRECISIONS[precision]
        n = ctypes.c_size_t()
        _lib.check(eng.lib.srwn_generate_state_bytes(eng.h, self.batch_size, self._prec, ctypes.byref(n)))
        self.buffer = torch.empty(n.value, dtype=torch.uint8, device="cuda")
        self.reset()

    def reset(self):
        """Back to silence at position 0 (the zero padding of ops.py:9)."""
        _lib.check(self._eng.lib.srwn_generate_state_reset(self._eng.h, self.buffer.data_ptr(), self.batch_size,
                                                           self._prec, _stream()))

    def position(self):
        """Samples generated through this state since the last reset (reads the device header: synchronises)."""
        return int(self.buffer[:8].view(torch.int64).item())

    def splice(self, rows, src, src_rows=None):
        """Utterance ``src_rows[i]`` of ``src`` (default: utterance i) replaces utterance ``rows[i]`` of this state
        (include/srwn.h, srwn_generate_state_splice).  ``src`` is another state of the same model and precision, at any
        position: each layer's queue is rotated to this state's phase, so generating here continues the utterance bit for
        bit as generating on ``src`` would.  This state's position, its other utterances and ``src`` are unchanged."""
        if not isinstance(src, GenerationState) or src._eng is not self._eng:
            raise ValueError("src must be a state of this state's model")
        if src is self or src.buffer.data_ptr() == self.buffer.data_ptr():
            raise ValueError("src and this state are the same state")
        if src.precision != self.precision:
            raise ValueError("src has precision %r, this state %r" % (src.precision, self.precision))
        rows = [int(r) for r in rows]
        src_rows = list(range(len(rows))) if src_rows is None else [int(r) for r in src_rows]
        if len(src_rows) != len(rows):
            raise ValueError("%d destination rows but %d source rows" % (len(rows), len(src_rows)))
        if any(r < 0 or r >= self.batch_size for r in rows) or any(r < 0 or r >= src.batch_size for r in src_rows):
            raise ValueError("rows must be in [0, %d) and src_rows in [0, %d)" % (self.batch_size, src.batch_size))
        if len(set(rows)) != len(rows):
            raise ValueError("a destination row is named twice")
        n = len(rows)
        dst_a, src_a = (ctypes.c_int32 * max(n, 1))(*rows), (ctypes.c_int32 * max(n, 1))(*src_rows)
        _lib.check(self._eng.lib.srwn_generate_state_splice(self._eng.h, self.data_ptr(), self.batch_size, dst_a,
                                                           src.data_ptr(), src.batch_size, src_a, n, self._prec,
                                                           _stream()))

    def data_ptr(self):
        return self.buffer.data_ptr()


class SynthesisState(object):
    """Device buffer that carries the student's flows from one ``generate`` call to the next: per flow the last H inputs,
    the last H / pool_stride frames and the position (include/srwn.h, srwn_student_state_*).  Created reset.  The host
    keeps its own copy of the position, which each call passes to the library (it sets the call's shape)."""

    def __init__(self, eng, batch_size, precision="fp16"):
        self._eng = eng
        self.batch_size, self.precision = int(batch_size), precision
        self._prec = _lib.PRECISIONS[precision]
        n = ctypes.c_size_t()
        _lib.check(eng.lib.srwn_student_state_bytes(eng.h, self.batch_size, self._prec, ctypes.byref(n)))
        self.buffer = torch.empty(n.value, dtype=torch.uint8, device="cuda")
        self.reset()

    def reset(self):
        """Back to the start of an utterance: position 0, silence before it."""
        _lib.check(self._eng.lib.srwn_student_state_reset(self._eng.h, self.buffer.data_ptr(), self.batch_size,
                                                          self._prec, _stream()))
        self._t0 = 0

    def position(self):
        """Samples synthesized through this state since the last reset (reads the device header: synchronises)."""
        return int(self.buffer[:8].view(torch.int64).item())

    def data_ptr(self):
        return self.buffer.data_ptr()


class ParallelWaveNet(_Model):
    """model.py:290-656.  ``teacher`` is a checkpoint directory in the reference; here it may also
    be a ``WaveNetAutoEncoder`` instance or None.  Methods keep the explicit ``sess`` first argument
    (ignored)."""

    def __init__(self, input_size, condition_size, dilations, teacher, num_flows=2, filter_width=2,
                 dilation_channels=32, skip_channels=256, latent_channels=16, pool_stride=512,
                 name='ParallelWaveNet', alpha=1.0, beta=1.0, gamma=1.0, learning_rate=0.001):
        self.input_size = input_size
        self.condition_size = condition_size
        self.dilations = list(dilations)
        self.teacher = teacher
        if isinstance(teacher, str):
            # model.py:326-331 imports the teacher's meta-graph from this directory; here the checkpoint written by
            # WaveNetAutoEncoder.save names every variable, and the constructor arguments the graph would carry
            # (mixtures, skip / encoder channels) are read off the variable shapes
            self.teacher = WaveNetAutoEncoder.from_checkpoint(teacher, dilations, latent_channels=latent_channels,
                                                              pool_stride=pool_stride, condition_size=condition_size,
                                                              filter_width=filter_width,
                                                              dilation_channels=dilation_channels, input_size=input_size)
        self.num_flows = num_flows
        self.filter_width = filter_width
        self.dilation_channels = dilation_channels
        self.skip_channels = skip_channels
        self.latent_channels = latent_channels
        self.pool_stride = pool_stride
        self.name = name
        self.alpha, self.beta, self.gamma = alpha, beta, gamma
        self.learning_rate = learning_rate
        self.precision = "fp32"
        self.seed = int.from_bytes(os.urandom(7), "little")      # key of the on-device logistic noise (generate(sess, None, ...))
        self._noise_calls = 0
        self.last_checkpoint_time = time.time()
        self.createNetwork()

    def createNetwork(self):
        """model.py:489-535."""
        self._eng = _Engine(_lib.STUDENT, self.dilations, self.filter_width, self.dilation_channels,
                            self.skip_channels, self.latent_channels + self.condition_size,
                            self.pool_stride, num_flows=self.num_flows)
        self._stft_ws = _Workspace()      # the power loss's STFT calls take no handle: their workspace is kept here
        w = synth.make_student_weights(self.dilations, self.num_flows, self.filter_width,
                                       self.dilation_channels, self.skip_channels,
                                       self.latent_channels + self.condition_size, seed=None)
        self._init_weights(w)

    def _flow_model(self, scope):
        """A one-flow network holding the variables of ``scope`` ('Flow<i>'): model.py:457-486 builds each flow as its own
        sub-graph; here it is the same kernels run for a single stack."""
        f = int(str(scope).replace('Flow', ''))
        if not 0 <= f < self.num_flows:
            raise ValueError("scope must be 'Flow0' .. 'Flow%d'" % (self.num_flows - 1))
        cache = self.__dict__.setdefault("_flow_models", {})
        if f not in cache:
            m = ParallelWaveNet(self.input_size, self.condition_size, self.dilations, None, num_flows=1,
                                filter_width=self.filter_width, dilation_channels=self.dilation_channels,
                                skip_channels=self.skip_channels, latent_channels=self.latent_channels,
                                pool_stride=self.pool_stride)
            cache[f] = m
        src, dst = synth.student_prefix(f), synth.student_prefix(0)
        cache[f].set_weights({dst + k[len(src):]: v for k, v in self.get_weights().items() if k.startswith(src)})
        return cache[f]

    def createFlow(self, inputs, encoding, scope, precision=None):
        """model.py:457-486 -> (scale, mean, out), each [B,T,1]: out = inputs * scale + mean with
        scale = exp(params[..., 0]), mean = params[..., 1] (no clamp on the log-scale)."""
        x = inputs[..., 0] if getattr(inputs, "ndim", 2) == 3 else inputs
        r = self._flow_model(scope).forward_all(x, encoding, precision=precision)
        return r["s_tot"][..., None], r["mu_tot"][..., None], r["x_last"][..., None]

    def createPartialFlow(self, inputs, encoding, scope, precision=None):
        """model.py:415-454 -> params [B,T,2] = (log scale, mean) of one flow."""
        scale, mean, _ = self.createFlow(inputs, encoding, scope, precision=precision)
        log = torch.log if isinstance(scale, torch.Tensor) else np.log
        cat = torch.cat if isinstance(scale, torch.Tensor) else np.concatenate
        return cat([log(scale), mean], -1)

    def set_weights(self, weights):
        """name -> ndarray with TF variable names (``ParallelWaveNet/Flow{f}/Flow{f}/...``)."""
        self._eng.set_weights(weights)
        self._mirror_weights(weights)

    def get_weights(self):
        if getattr(self, "_packed_stale", False):        # trained on the device since the last read-back
            self.sync_weights()
        return dict(self._weights)

    def load(self, sess, logdir):
        if isinstance(self.teacher, str):
            pass   # the reference restores the imported teacher meta-graph here (model.py:543-544)
        return self._load(logdir)

    def save(self, sess, logdir, global_step, force=False):
        return self._save(logdir, global_step, force)

    def synthesis_state(self, batch_size, precision="fp16"):
        """A fresh (reset) state for synthesizing ``batch_size`` utterances in chunks: pass it to ``generate(state=...)``
        or ``forward_all(state=...)`` to continue the previous call on it."""
        return SynthesisState(self._eng, batch_size, precision)

    def _forward(self, inputs, encoding, conditions, precision=None, want=("out",), state=None):
        eng = self._eng
        if state is not None:
            if not isinstance(state, SynthesisState) or state._eng is not eng:
                raise ValueError("state must come from this model's synthesis_state()")
            precision = precision or state.precision
        enc = _with_conditions(encoding, conditions, self.condition_size)
        e, on_dev = eng.to_device(enc, "enc")
        if inputs is None:          # student.py:104 / :172 draws the logistic noise on the host; here it is drawn on the device
            B, T = e.shape[0], e.shape[1] * self.pool_stride
            z = None
        else:
            z, on_dev = eng.to_device(inputs, "z")
            B, T = z.shape
        eng.check_encoding(e, B, T)
        prec = _lib.PRECISIONS[precision or self.precision]
        if state is not None and (state.batch_size != B or state.precision != precision):
            raise ValueError("state was made for batch_size=%d, precision=%r; this call has %d, %r"
                             % (state.batch_size, state.precision, B, precision))
        if prec != _lib.FP32 and getattr(self, "_packed_stale", False):
            self.sync_weights()
        op = _lib.OP_STUDENT_FORWARD if state is None else _lib.OP_STUDENT_STREAM
        ws, wsn = eng.workspace(op, B, T, prec)
        bufs = {k: torch.empty(B, T, dtype=torch.float32, device="cuda") for k in set(want) | {"out"}}
        g = lambda k: bufs[k].data_ptr() if k in bufs else None
        if state is not None:               # this call's T samples continue the state (device noise: a new Philox stream)
            if z is None:
                self._noise_calls += 1
            _lib.check(eng.lib.srwn_student_forward_resume(eng.h, state.data_ptr(), state._t0,
                                                           None if z is None else z.data_ptr(), self.seed,
                                                           self._noise_calls, e.data_ptr(), g("out"), g("s_tot"),
                                                           g("mu_tot"), g("x_last"), g("z"), B, T, prec, ws, wsn,
                                                           _stream()))
            state._t0 += T
        elif z is None:
            self._noise_calls += 1
            _lib.check(eng.lib.srwn_student_sample(eng.h, self.seed, self._noise_calls, e.data_ptr(), g("out"), g("s_tot"),
                                                   g("mu_tot"), g("x_last"), g("z"), B, T, prec, ws, wsn, _stream()))
        else:
            bufs.pop("z", None)
            _lib.check(eng.lib.srwn_student_forward(eng.h, z.data_ptr(), e.data_ptr(), g("out"), g("s_tot"),
                                                    g("mu_tot"), g("x_last"), B, T, prec, ws, wsn, _stream()))
        return bufs, (on_dev, op, B, T, prec)

    def generate(self, sess, inputs, encoding, conditions=None, precision=None, state=None):
        """model.py:570-576 -> out [B,T,1] = clip(z*s_tot + mu_tot, -1, 1).  ``inputs=None`` draws the logistic noise of
        student.py:172 on the device (inside the fused flow kernel on the fp16 path): nothing but the encoding is uploaded.

        ``state`` (from ``synthesis_state``): these T samples (a multiple of pool_stride) continue the clip where the last
        call on that state stopped, and the state advances by T; ``inputs`` and ``encoding`` then cover this call's
        samples only and the precision defaults to the state's.  With injected noise, any split of a clip into such calls
        gives bit for bit the audio of one call; noise drawn on the device comes from a new Philox stream per call
        (``forward_all`` returns it as ``z``)."""
        bufs, call = self._forward(inputs, encoding, conditions, precision, state=state)
        return self._eng.finish(bufs["out"][:, :, None], *call)

    def forward_all(self, inputs, encoding, conditions=None, precision=None, state=None):
        """out, s_tot, mu_tot (model.py:517-535) and the chained flow output, each [B,T]; with ``inputs=None`` also the
        noise ``z`` that was drawn.  ``state``: as in ``generate``."""
        want = ("out", "s_tot", "mu_tot", "x_last") + (("z",) if inputs is None else ())
        bufs, call = self._forward(inputs, encoding, conditions, precision, want=want, state=state)
        return {k: self._eng.finish(v, *call) for k, v in bufs.items()}

    def _entropies(self, inputs, encoding, conditions):
        bufs, _ = self._forward(inputs, encoding, conditions, want=("s_tot",))
        B, T = bufs["s_tot"].shape
        per = torch.empty(B, dtype=torch.float64, device="cuda")
        _lib.check(self._eng.lib.srwn_entropy(bufs["s_tot"].data_ptr(), per.data_ptr(), B, T, _stream()))
        return per.cpu().numpy()

    def getEntropy_fast(self, sess, inputs, encoding, conditions=None):
        """model.py:595-600: reduce_sum(log(s_tot) + 2) over the whole batch (model.py:356)."""
        return float(self._entropies(inputs, encoding, conditions).sum())

    def getEntropy(self, sess, inputs, encoding, conditions=None):
        """model.py:578-593: per-example entropies."""
        return self._entropies(inputs, encoding, conditions)

    # ---- distillation (model.py:316-401, 603-642) -------------------------------------------------
    def _teacher_logits(self, truth, enc, teacher_logits, teacher_precision):
        """stop_gradient(teacher decoder teacher-forced on the REAL audio) (model.py:326-334, F5)."""
        if teacher_logits is not None:
            return self._eng.to_device(teacher_logits, "tlogits")[0]
        if not isinstance(self.teacher, WaveNetAutoEncoder):
            raise RuntimeError("train needs `teacher` to be a WaveNetAutoEncoder (or pass teacher_logits=)")
        prec = teacher_precision or ("fp16" if "fp16" in self.teacher.available_precisions() else "fp32")
        return self.teacher.get_logits(truth, enc, precision=prec)

    def loss_and_grads(self, inputs, truth, encoding, conditions=None, teacher_logits=None,
                       teacher_precision=None, batch_norm=None):
        """One forward + backward of the distillation graph (model.py:356-384) on the device.
        Returns (loss, power_loss, entropy, flat_grads) with flat_grads a CUDA fp32 tensor laid out like the
        library's weight arena (see ``grad_of``).  ``batch_norm`` overrides the divisor B of model.py:379
        (the global batch under data parallelism)."""
        eng = self._eng
        enc = _with_conditions(encoding, conditions, self.condition_size)
        z, _ = eng.to_device(inputs, "z")
        x, _ = eng.to_device(truth, "truth")
        e, _ = eng.to_device(enc, "enc")
        B, T = z.shape
        eng.check_encoding(e, B, T)
        if x.shape != z.shape:
            raise ValueError("truth must be [B,T] like inputs")
        tl = self._teacher_logits(x, e, teacher_logits, teacher_precision).contiguous()
        M = tl.shape[2] // 4
        ws, wsn = eng.workspace(_lib.OP_STUDENT_TRAIN, B, T, _lib.FP32)
        out = torch.empty(B, T, dtype=torch.float32, device="cuda")
        s_tot, mu_tot = torch.empty_like(out), torch.empty_like(out)
        _lib.check(eng.lib.srwn_student_forward_train(eng.h, z.data_ptr(), e.data_ptr(), out.data_ptr(),
                                                      s_tot.data_ptr(), mu_tot.data_ptr(), B, T, ws, wsn, _stream()))
        norm = float(batch_norm or B)
        # cross-entropy against the teacher's mixture (model.py:374-375): value + d/d out
        d_ce, nll = torch.empty_like(out), torch.empty_like(out)
        _lib.check(eng.lib.srwn_mol_loss_grad(out.data_ptr(), tl.data_ptr(), d_ce.data_ptr(), nll.data_ptr(), B, T, M, _stream()))
        # spectral power loss (model.py:360-371) and its gradient: FFT kernels of csrc/stft_loss.cu
        power, d_pow = self._power_loss(x, out)
        # entropy (model.py:356), clip mask (model.py:535) and the loss gradients the backward pass starts from
        d_pre, d_s = torch.empty_like(out), torch.empty_like(out)
        sums = torch.empty(_lib.DISTILL_SUMS_LEN, dtype=torch.float64, device="cuda")
        _lib.check(eng.lib.srwn_distill_loss_grad(z.data_ptr(), s_tot.data_ptr(), mu_tot.data_ptr(), nll.data_ptr(),
                                                  d_ce.data_ptr(), d_pow.data_ptr(), float(self.alpha), float(self.beta),
                                                  1.0 / norm, d_pre.data_ptr(), d_s.data_ptr(), sums.data_ptr(), B, T,
                                                  _stream()))
        entropy = sums[1]
        # one bucket [flat gradient | loss | power_loss]: what a data-parallel step all-reduces in a single call
        n = ctypes.c_int64()
        _lib.check(eng.lib.srwn_param_count(eng.h, ctypes.byref(n)))
        bucket = torch.empty(n.value + 2, dtype=torch.float32, device="cuda")
        grads, tail = bucket[:n.value], bucket[n.value:]
        _lib.check(eng.lib.srwn_distill_finish(sums.data_ptr(), power.data_ptr(), float(self.alpha), float(self.beta),
                                               1.0 / norm, tail.data_ptr(), _stream()))        # model.py:374-379
        _lib.check(eng.lib.srwn_student_backward(eng.h, z.data_ptr(), e.data_ptr(), d_pre.data_ptr(), d_s.data_ptr(),
                                                 grads.data_ptr(), B, T, ws, wsn, _stream()))
        self._bucket = bucket
        return tail[0], tail[1], entropy, grads

    def _power_loss(self, truth, out, frame_length=512, frame_step=256):
        """gamma * || mean_t |STFT(truth)|^2 - mean_t |STFT(out)|^2 ||^2 (model.py:360-371) and d/d out, on the device.
        Returns (power_loss: float64 CUDA tensor [1], d_out [B,T] fp32)."""
        eng = self._eng
        B, T = out.shape
        ws, wsn = self._stft_ws.get(eng.lib.srwn_stft_workspace_bytes, B, T, frame_length, frame_step)
        p = torch.empty(1, dtype=torch.float64, device="cuda")
        g = torch.empty_like(out)
        _lib.check(eng.lib.srwn_stft_power_loss(truth.data_ptr(), out.data_ptr(), float(self.gamma), p.data_ptr(),
                                                g.data_ptr(), B, T, frame_length, frame_step, ws, wsn, _stream()))
        return p, g

    def grad_of(self, flat_grads, name):
        """View of one variable's gradient inside ``flat_grads`` (TF variable name)."""
        off, cnt = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(self._eng.lib.srwn_weight_offset(self._eng.h, name.encode(), ctypes.byref(off), ctypes.byref(cnt)))
        return flat_grads[off.value:off.value + cnt.value]

    def apply_gradients(self, flat_grads, clip_norm=1.0, beta1=0.9, beta2=0.999, epsilon=1e-8):
        """tf.clip_by_global_norm(grads, 1.0) + AdamOptimizer(learning_rate).apply_gradients (model.py:382-401).
        Under torch.distributed the caller all-reduces ``flat_grads`` first (``train_fast`` does)."""
        eng = self._eng
        if not hasattr(self, "_adam"):
            self._adam = dict(m=torch.zeros_like(flat_grads), v=torch.zeros_like(flat_grads),
                              scratch=torch.zeros(4, dtype=torch.float32, device="cuda"), step=0)
        a = self._adam
        a["step"] += 1
        _lib.check(eng.lib.srwn_adam_step(eng.h, flat_grads.data_ptr(), a["m"].data_ptr(), a["v"].data_ptr(),
                                          a["scratch"].data_ptr(), float(clip_norm), float(self.learning_rate),
                                          float(beta1), float(beta2), float(epsilon), a["step"], _stream()))
        self._packed_stale = True

    def sync_weights(self):
        """Re-packs the 16-bit operand images from the (trained) device weights and refreshes ``get_weights``."""
        eng = self._eng
        _lib.check(eng.lib.srwn_commit_weights(eng.h, _stream()))
        for k, v in list(self._weights.items()):
            try:
                self._weights[k] = eng.get_weight(k, v.shape)
            except _lib.SrwnError:
                pass      # dead variables (gate conv, student skip conv) are not stored
        self._packed_stale = False

    def _sync_replicas(self, local_B):
        """Data parallelism: every rank must hold the same weights and optimizer state, or the shared gradient moves
        different parameters and the replicas drift apart.  On the first distributed step rank 0's weight arena and Adam
        state are broadcast; the global batch is the sum of the ranks' local batches (recomputed when the local one
        changes).  Returns (world, global batch)."""
        from . import shard
        if not shard.is_distributed():
            return 1, local_B
        import torch.distributed as dist
        st = self.__dict__.setdefault("_dp", {})
        if st.get("local_B") != local_B:
            st["local_B"], st["global_B"] = local_B, shard.global_batch(local_B)
        if not st.get("synced"):
            eng = self._eng
            n = ctypes.c_int64()
            _lib.check(eng.lib.srwn_param_count(eng.h, ctypes.byref(n)))
            w = torch.empty(n.value, dtype=torch.float32, device="cuda")
            _lib.check(eng.lib.srwn_weights_flat(eng.h, w.data_ptr(), n.value, 0, _stream()))      # device arena -> w
            state = [w]
            if hasattr(self, "_adam"):
                step = torch.tensor([float(self._adam["step"])], device="cuda")
                state += [self._adam["m"], self._adam["v"], step]
            shard.broadcast_from_rank0(state)
            _lib.check(eng.lib.srwn_weights_flat(eng.h, w.data_ptr(), n.value, 1, _stream()))      # w -> device arena
            if hasattr(self, "_adam"):
                self._adam["step"] = int(step.item())
            self._packed_stale = True
            st["synced"] = True
        return dist.get_world_size(), st["global_B"]

    def train_fast(self, sess, inputs, truth, encoding, conditions=None, teacher_logits=None, teacher_precision=None):
        """model.py:634-642: one optimisation step, returns (loss, power_loss).  With torch.distributed
        initialised, ranks hold batch shards: the loss is normalised by the global batch, the bucket
        [flat gradient | loss | power_loss] is summed with ONE all-reduce before the global-norm clip (SURVEY.md 8(e)),
        and every rank applies the same Adam update to the same weights (``_sync_replicas``).  CUDA tensors in ->
        0-d CUDA tensors out with no host synchronisation inside the step; NumPy in -> Python floats."""
        B = int(inputs.shape[0])
        world, global_B = self._sync_replicas(B)
        on_dev = isinstance(inputs, torch.Tensor) and inputs.is_cuda
        loss, power, _, grads = self.loss_and_grads(inputs, truth, encoding, conditions, teacher_logits,
                                                    teacher_precision, batch_norm=global_B)
        if world > 1:
            from . import shard
            ev = self.__dict__.get("_coll_events")       # bench.py: CUDA events around the collective
            if ev:
                ev[0].record()
            shard.all_reduce_sum(self._bucket)
            if ev:
                ev[1].record()
        self.apply_gradients(grads)
        if on_dev:
            return loss, power
        lp = self._eng.to_host(self._bucket[-2:], False)
        return float(lp[0]), float(lp[1])

    def train(self, sess, inputs, truth, encoding, conditions=None, teacher_logits=None, teacher_precision=None):
        """model.py:603-632, literally: one evaluation of the graph per EXAMPLE of ``inputs`` -- its noise row fed as a
        batch of one, broadcast against the whole ``encoding`` / ``truth`` batch, the loss divided by shape(inputs)[0] = 1
        (model.py:379), gradients clipped per example (``self.grads`` are the clipped ones, model.py:385-392) -- then the
        clipped gradients, losses and power losses are averaged and one Adam update is applied without further clipping.
        Returns (mean loss, mean power loss)."""
        eng = self._eng
        z_all, _ = eng.to_device(inputs, "z_all")
        x, _ = eng.to_device(truth, "truth")
        e, _ = eng.to_device(_with_conditions(encoding, conditions, self.condition_size), "enc")
        N, Be = z_all.shape[0], e.shape[0]
        mean = None
        scratch = torch.zeros(1, dtype=torch.float32, device="cuda")
        for i in range(N):
            zi = z_all[i:i + 1].expand(Be, -1).contiguous()          # [1,T] against [Be, ...]: TF broadcasts the batch axis
            self.loss_and_grads(zi, x, e, None, teacher_logits, teacher_precision, batch_norm=1)
            b = self._bucket
            _lib.check(eng.lib.srwn_clip_by_global_norm(b.data_ptr(), b.numel() - 2, 1.0, scratch.data_ptr(), _stream()))
            if mean is None:
                mean = torch.zeros_like(b)
            _lib.check(eng.lib.srwn_axpy(mean.data_ptr(), b.data_ptr(), 1.0 / N, b.numel(), _stream()))
        self.apply_gradients(mean[:-2], clip_norm=0.0)
        lp = eng.to_host(mean[-2:], False)
        return float(lp[0]), float(lp[1])

    def _need_teacher(self):
        if not isinstance(self.teacher, WaveNetAutoEncoder):
            raise RuntimeError("this call evaluates the imported teacher graph (model.py:326-334): construct "
                               "ParallelWaveNet with teacher=<WaveNetAutoEncoder instance>")
        return self.teacher

    def encode(self, sess, inputs, conditions=None, precision=None):
        """model.py:644-649: the imported teacher's ``Encoding_output`` on ``inputs``."""
        return self._need_teacher().encode(inputs, conditions, precision=precision)

    def reconstruct(self, sess, inputs, conditions=None, **kw):
        """model.py:651-656: the imported teacher's ``Out_e`` (encoder + teacher-forced decoder + sampling)."""
        return self._need_teacher().reconstruct(inputs, conditions, **kw)
