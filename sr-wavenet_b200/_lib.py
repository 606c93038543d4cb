"""ctypes binding of libsrwn.so (include/srwn.h).  No torch types cross this boundary:
tensors are passed as raw device pointers (``tensor.data_ptr()``) and the stream as the
``cudaStream_t`` integer.  There is no fallback: if the library is missing, ``load()`` raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SRWN_LIB") or os.path.join(_HERE, "libsrwn.so")   # SRWN_LIB: tuning builds (tools/exp_build.sh <source.cu> <name> [flags])

ABI_VERSION = 7      # SRWN_ABI_VERSION in include/srwn.h
OK, ERR_INVALID, ERR_CUDA, ERR_WEIGHTS, ERR_UNSUPPORTED, ERR_WORKSPACE = range(6)
TEACHER, STUDENT = 0, 1
FP32, BF16, FP16 = 0, 1, 2
OP_TEACHER_LOGITS, OP_TEACHER_NLL, OP_TEACHER_GENERATE, OP_STUDENT_FORWARD, OP_STUDENT_TRAIN, OP_TEACHER_PREFILL, \
    OP_STUDENT_STREAM = range(7)
DISTILL_SUMS_LEN = 1024   # SRWN_DISTILL_SUMS_LEN
PRECISIONS = {"fp32": FP32, "fp16": FP16}      # BF16 is refused by the library (include/srwn.h)


class SrwnError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libsrwn error %d: %s" % (code, msg))
        self.code = code


class Config(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("n_layers", ctypes.c_int32),
                ("dilations", ctypes.POINTER(ctypes.c_int32)), ("filter_width", ctypes.c_int32),
                ("dilation_channels", ctypes.c_int32), ("skip_channels", ctypes.c_int32),
                ("cond_channels", ctypes.c_int32), ("pool_stride", ctypes.c_int32),
                ("num_mixtures", ctypes.c_int32), ("num_flows", ctypes.c_int32)]


class EncoderConfig(ctypes.Structure):
    _fields_ = [("n_layers", ctypes.c_int32), ("filter_width", ctypes.c_int32),
                ("encoder_channels", ctypes.c_int32), ("skip_channels", ctypes.c_int32),
                ("latent_channels", ctypes.c_int32), ("pool_stride", ctypes.c_int32)]


_vp, _i32, _i64, _sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
_fp = ctypes.c_void_p   # device float* (raw address)

# name -> (restype, argtypes); every symbol include/srwn.h declares
SIGNATURES = {
    "srwn_abi_version": (ctypes.c_int, []),
    "srwn_last_error": (ctypes.c_char_p, []),
    "srwn_launch_count": (_i64, []),
    "srwn_create": (ctypes.c_int, [ctypes.POINTER(Config), ctypes.POINTER(_vp)]),
    "srwn_destroy": (ctypes.c_int, [_vp]),
    "srwn_set_weight": (ctypes.c_int, [_vp, ctypes.c_char_p, _vp, ctypes.POINTER(_i64), _i32]),
    "srwn_get_weight": (ctypes.c_int, [_vp, ctypes.c_char_p, _vp, _i64]),
    "srwn_commit_weights": (ctypes.c_int, [_vp, _vp]),
    "srwn_set_profiling": (ctypes.c_int, [_vp, _i32]),
    "srwn_set_team_size": (ctypes.c_int, [_vp, _i32]),
    "srwn_set_wait_limit": (ctypes.c_int, [_vp, _i64]),
    "srwn_last_partition": (ctypes.c_int, [_vp, ctypes.POINTER(_i32), ctypes.POINTER(_i32)]),
    "srwn_last_kernel_ms": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(_i32),
                                           ctypes.POINTER(ctypes.c_char_p)]),
    "srwn_check_async_error": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_peek_async_error": (ctypes.c_int, [_vp]),
    "srwn_supports": (ctypes.c_int, [_vp, _i32, _i32]),
    "srwn_workspace_bytes": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, ctypes.POINTER(_sz)]),
    "srwn_teacher_logits": (ctypes.c_int, [_vp, _fp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_teacher_nll": (ctypes.c_int, [_vp, _fp, _fp, _fp, _fp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_teacher_generate": (ctypes.c_int, [_vp, _fp, _fp, _fp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_generate_state_bytes": (ctypes.c_int, [_vp, _i32, _i32, ctypes.POINTER(_sz)]),
    "srwn_generate_state_reset": (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp]),
    "srwn_teacher_generate_resume": (ctypes.c_int, [_vp, _vp, _fp, _fp, _fp, _fp, _i32, _fp, _fp, _i32, _i32, _i32,
                                                    _vp, _sz, _vp]),
    "srwn_generate_state_prefill": (ctypes.c_int, [_vp, _vp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_generate_state_splice": (ctypes.c_int, [_vp, _vp, _i32, ctypes.POINTER(_i32), _vp, _i32, ctypes.POINTER(_i32),
                                                  _i32, _i32, _vp]),
    "srwn_student_forward": (ctypes.c_int, [_vp, _fp, _fp, _fp, _fp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_student_sample": (ctypes.c_int, [_vp, ctypes.c_uint64, ctypes.c_uint64, _fp, _fp, _fp, _fp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_student_state_bytes": (ctypes.c_int, [_vp, _i32, _i32, ctypes.POINTER(_sz)]),
    "srwn_student_state_reset": (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp]),
    "srwn_student_forward_resume": (ctypes.c_int, [_vp, _vp, _i64, _fp, ctypes.c_uint64, ctypes.c_uint64, _fp, _fp, _fp, _fp,
                                                   _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_random_logistic": (ctypes.c_int, [_fp, _i64, ctypes.c_uint64, ctypes.c_uint64, _vp]),
    "srwn_random_uniform": (ctypes.c_int, [_fp, _i64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_float, ctypes.c_float, _vp]),
    "srwn_weights_flat": (ctypes.c_int, [_vp, _fp, _i64, _i32, _vp]),
    "srwn_distill_finish": (ctypes.c_int, [_vp, _vp, ctypes.c_float, ctypes.c_float, ctypes.c_float, _fp, _vp]),
    "srwn_clip_by_global_norm": (ctypes.c_int, [_fp, _i64, ctypes.c_float, _fp, _vp]),
    "srwn_axpy": (ctypes.c_int, [_fp, _fp, ctypes.c_float, _i64, _vp]),
    "srwn_entropy": (ctypes.c_int, [_fp, _vp, _i32, _i32, _vp]),
    "srwn_param_count": (ctypes.c_int, [_vp, ctypes.POINTER(_i64)]),
    "srwn_weight_offset": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    "srwn_student_forward_train": (ctypes.c_int, [_vp, _fp, _fp, _fp, _fp, _fp, _i32, _i32, _vp, _sz, _vp]),
    "srwn_student_backward": (ctypes.c_int, [_vp, _fp, _fp, _fp, _fp, _fp, _i32, _i32, _vp, _sz, _vp]),
    "srwn_mol_loss_grad": (ctypes.c_int, [_fp, _fp, _fp, _fp, _i32, _i32, _i32, _vp]),
    "srwn_adam_step": (ctypes.c_int, [_vp, _fp, _fp, _fp, _fp, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                      ctypes.c_float, ctypes.c_float, _i32, _vp]),
    "srwn_stft_workspace_bytes": (ctypes.c_int, [_i32, _i32, _i32, _i32, ctypes.POINTER(_sz)]),
    "srwn_stft_power": (ctypes.c_int, [_fp, _fp, _i32, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_stft_power_loss": (ctypes.c_int, [_fp, _fp, ctypes.c_float, _vp, _fp, _i32, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_distill_loss_grad": (ctypes.c_int, [_fp, _fp, _fp, _fp, _fp, _fp, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                              _fp, _fp, _vp, _i32, _i32, _vp]),
    "srwn_encoder_create": (ctypes.c_int, [ctypes.POINTER(EncoderConfig), ctypes.POINTER(_vp)]),
    "srwn_encoder_destroy": (ctypes.c_int, [_vp]),
    "srwn_encoder_set_weight": (ctypes.c_int, [_vp, ctypes.c_char_p, _vp, ctypes.POINTER(_i64), _i32]),
    "srwn_encoder_commit": (ctypes.c_int, [_vp, _vp]),
    "srwn_encoder_supports": (ctypes.c_int, [_vp, _i32]),
    "srwn_encoder_workspace_bytes": (ctypes.c_int, [_vp, _i32, _i32, _i32, ctypes.POINTER(_sz)]),
    "srwn_teacher_encode": (ctypes.c_int, [_vp, _fp, _fp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_encoder_check_async_error": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _sz, _vp]),
    "srwn_encoder_set_profiling": (ctypes.c_int, [_vp, _i32]),
    "srwn_encoder_last_ms": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_float)]),
    "srwn_dilated_causal_conv1d": (ctypes.c_int, [_fp, _fp, _fp, _fp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "srwn_residual_dilation_layer": (ctypes.c_int, [_fp] * 9 + [_i32] * 6 + [_vp]),
    "srwn_conv1d_same": (ctypes.c_int, [_fp, _fp, _fp, _fp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "srwn_log_softmax": (ctypes.c_int, [_fp, _fp, _i64, _i32, _i32, _vp]),
    "srwn_right_shift": (ctypes.c_int, [_fp, _fp, _i32, _i32, _i32, _i32, _vp]),
    "srwn_resize_nearest": (ctypes.c_int, [_fp, _fp, _i32, _i32, _i32, _i32, _vp]),
    "srwn_relu": (ctypes.c_int, [_fp, _i64, _vp]),
    "srwn_avg_pool_time": (ctypes.c_int, [_fp, _fp, _i32, _i32, _i32, _i32, _vp]),
    "srwn_softmax": (ctypes.c_int, [_fp, _fp, _i64, _i32, _vp]),
    "srwn_pair_distance": (ctypes.c_int, [_fp, _fp, _fp, _i32, _i32, _vp]),
    "srwn_mol_loss": (ctypes.c_int, [_fp, _fp, _fp, _fp, _i32, _i32, _i32, _vp]),
    "srwn_mol_sample": (ctypes.c_int, [_fp, _fp, _fp, _fp, _vp, _i32, _i32, _i32, _vp]),
}

_lib = None


def load():
    """Loads libsrwn.so (built in-tree by ``__graft_entry__.build()``).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libsrwn.so not found at %s: build it with `python __graft_entry__.py` "
            "(there is no CPU or PyTorch fallback for the hot path)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.srwn_abi_version() != ABI_VERSION:
        raise RuntimeError("libsrwn.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != OK:
        raise SrwnError(rc, load().srwn_last_error().decode("utf-8", "replace"))


def launch_count():
    return int(load().srwn_launch_count())
