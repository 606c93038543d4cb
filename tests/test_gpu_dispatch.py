"""-m gpu: one rule says which op runs at which precision on which handle (csrc/api.cu).  srwn_supports, srwn_workspace_bytes,
the op's entry points and the state calls must agree on it: an (op, precision) the rule refuses is refused by each of them
with the same code and before any launch, and one it accepts runs in exactly the workspace srwn_workspace_bytes reports.

The handles cover every refusal the rule has: the wrong handle kind, SRWN_BF16, a value that is no precision, SRWN_FP16
where the fused kernel (a dilation past 512) or the generation kernel (32 layers) does not cover the configuration, an op
that runs in fp32 only, an unknown op, and the batch limit of the fused kernel."""
import ctypes

import pytest
import torch

from sr_wavenet_b200 import synth, _lib

pytestmark = pytest.mark.gpu

P, M, F = 128, 5, 2
B, T = 2, 2 * P
PRECISIONS = [_lib.FP32, _lib.BF16, _lib.FP16, 7]
FUSED_OPS = [_lib.OP_TEACHER_LOGITS, _lib.OP_TEACHER_NLL, _lib.OP_STUDENT_FORWARD, _lib.OP_STUDENT_STREAM]
HANDLES = {
    "teacher": ("teacher", synth.DEFAULT_DILATIONS),
    "teacher_fused_refuses": ("teacher", [1, 2, 513]),
    "teacher_generation_refuses": ("teacher", [1 << (i % 10) for i in range(32)]),
    "student": ("student", synth.DEFAULT_DILATIONS),
    "student_fused_refuses": ("student", [1, 2, 513]),
}


@pytest.fixture(scope="module")
def models(lib):
    import sr_wavenet_b200 as srwn
    out = {}
    for name, (kind, dil) in HANDLES.items():
        if kind == "teacher":
            m = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=M, dilations=dil, skip_channels=128,
                                        latent_channels=32, pool_stride=P)
            m.set_weights(synth.make_teacher_weights(dil, num_mixtures=M))
        else:
            m = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=dil, teacher=None, num_flows=F,
                                     skip_channels=128, latent_channels=32, pool_stride=P)
            m.set_weights(synth.make_student_weights(dil, num_flows=F))
        out[name] = m
    return out


class Inputs(object):
    """Device inputs and outputs of every entry point for b utterances of T samples."""

    def __init__(self, b):
        dev = lambda a: torch.from_numpy(a).cuda()
        self.x = dev(synth.synthetic_audio(b, T))
        self.enc = dev(synth.synthetic_encoding(b, T // P))
        self.z = dev(synth.logistic_noise(b, T))
        u1, u2 = synth.sampler_uniforms(b, T, num_mixtures=M)
        self.u1, self.u2 = dev(u1), dev(u2)
        self.out = torch.empty(b, T, 4 * M, device="cuda")
        self.row = [torch.empty(b, T, device="cuda") for _ in range(3)]


def workspace_query(lib, h, op, b, prec):
    n = ctypes.c_size_t()
    return lib.srwn_workspace_bytes(h, op, b, T, prec, ctypes.byref(n)), n.value


def state_calls(lib, op):
    """(bytes, reset) of the state the op runs on, or None."""
    if op in (_lib.OP_TEACHER_GENERATE, _lib.OP_TEACHER_PREFILL):
        return lib.srwn_generate_state_bytes, lib.srwn_generate_state_reset
    if op == _lib.OP_STUDENT_STREAM:
        return lib.srwn_student_state_bytes, lib.srwn_student_state_reset
    return None


def reset_state(lib, h, op, b, prec):
    query, reset = state_calls(lib, op)
    n = ctypes.c_size_t()
    _lib.check(query(h, b, prec, ctypes.byref(n)))
    state = torch.empty(n.value, dtype=torch.uint8, device="cuda")
    _lib.check(reset(h, state.data_ptr(), b, prec, torch.cuda.current_stream().cuda_stream))
    return state


def entry_points(lib, h, op, b, prec, io, state, ws, wsn):
    """Every call of `op` at `prec`, each a thunk returning the library's code."""
    st = torch.cuda.current_stream().cuda_stream
    x, enc, z, u1, u2, out = io.x.data_ptr(), io.enc.data_ptr(), io.z.data_ptr(), io.u1.data_ptr(), io.u2.data_ptr(), \
        io.out.data_ptr()
    r0, r1, r2 = (r.data_ptr() for r in io.row)
    s = state.data_ptr() if state is not None else None
    if op == _lib.OP_TEACHER_LOGITS:
        return [lambda: lib.srwn_teacher_logits(h, x, enc, out, b, T, prec, ws, wsn, st)]
    if op == _lib.OP_TEACHER_NLL:
        return [lambda: lib.srwn_teacher_nll(h, x, enc, x, r0, None, None, b, T, prec, ws, wsn, st)]
    if op == _lib.OP_TEACHER_GENERATE:
        return [lambda: lib.srwn_teacher_generate(h, enc, u1, u2, r0, None, b, T, prec, ws, wsn, st),
                lambda: lib.srwn_teacher_generate_resume(h, s, enc, u1, u2, None, 0, r0, None, b, T, prec, ws, wsn, st)]
    if op == _lib.OP_STUDENT_FORWARD:
        return [lambda: lib.srwn_student_forward(h, z, enc, r0, r1, r2, None, b, T, prec, ws, wsn, st),
                lambda: lib.srwn_student_sample(h, 1, 2, enc, r0, r1, r2, None, None, b, T, prec, ws, wsn, st)]
    if op == _lib.OP_STUDENT_TRAIN:           # no precision argument: the training calls run in fp32
        if prec != _lib.FP32:
            return []
        return [lambda: lib.srwn_student_forward_train(h, z, enc, r0, r1, r2, b, T, ws, wsn, st)]
    if op == _lib.OP_TEACHER_PREFILL:
        return [lambda: lib.srwn_generate_state_prefill(h, s, x, enc, T, b, prec, ws, wsn, st)]
    if op == _lib.OP_STUDENT_STREAM:
        return [lambda: lib.srwn_student_forward_resume(h, s, 0, z, 0, 0, enc, r0, r1, r2, None, None, b, T, prec, ws, wsn,
                                                        st)]
    return []


def supports_quietly(lib, h, op, prec):
    """srwn_supports, checking that it leaves the last error as it was."""
    n = ctypes.c_size_t()
    assert lib.srwn_workspace_bytes(h, 99, B, T, _lib.FP32, ctypes.byref(n)) == _lib.ERR_INVALID
    before = lib.srwn_last_error()
    ok = lib.srwn_supports(h, op, prec)
    assert lib.srwn_last_error() == before
    assert ok in (0, 1)
    return ok


@pytest.mark.parametrize("name", list(HANDLES))
def test_supports_workspace_and_calls_agree(models, name):
    lib, h = _lib.load(), models[name]._eng.h
    io = Inputs(B)
    dummy = torch.zeros(16 << 20, dtype=torch.uint8, device="cuda")   # a state that is never reset (refused calls)
    st = torch.cuda.current_stream().cuda_stream
    for op in (-1, 7):
        assert supports_quietly(lib, h, op, _lib.FP32) == 0
        assert workspace_query(lib, h, op, B, _lib.FP32)[0] == _lib.ERR_INVALID
    accepted = 0
    for op in range(7):
        for prec in PRECISIONS:
            what = "%s op %d precision %d" % (name, op, prec)
            ok = supports_quietly(lib, h, op, prec)
            rc, nbytes = workspace_query(lib, h, op, B, prec)
            assert ok == (rc == _lib.OK), what
            calls = state_calls(lib, op)
            if not ok:
                n0 = _lib.launch_count()
                for call in entry_points(lib, h, op, B, prec, io, dummy, None, 0):
                    assert call() == rc, what + ": " + lib.srwn_last_error().decode()
                if calls is not None:
                    n = ctypes.c_size_t()
                    assert calls[0](h, B, prec, ctypes.byref(n)) == rc, what
                    assert calls[1](h, dummy.data_ptr(), B, prec, st) == rc, what
                assert _lib.launch_count() == n0, what
                continue
            accepted += 1
            state = reset_state(lib, h, op, B, prec) if calls is not None else None
            ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            for call in entry_points(lib, h, op, B, prec, io, state, ws.data_ptr(), nbytes):
                if state is not None:
                    _lib.check(calls[1](h, state.data_ptr(), B, prec, st))
                _lib.check(call())
                _lib.check(lib.srwn_check_async_error(h, op, B, T, prec, ws.data_ptr(), nbytes, st))
    assert accepted >= 3


@pytest.mark.parametrize("name", list(HANDLES))
def test_batch_limit_agrees(models, name):
    """One utterance past 8 per SM: the query and every call refuse with the same code, naming the limit, before any launch
    (the calls get no workspace, so a call that skipped the limit would report the workspace instead)."""
    lib, h = _lib.load(), models[name]._eng.h
    limit = 8 * torch.cuda.get_device_properties(0).multi_processor_count
    io = None
    for op in FUSED_OPS:
        if not lib.srwn_supports(h, op, _lib.FP16):
            continue
        io = io or Inputs(limit + 1)
        state = reset_state(lib, h, op, limit + 1, _lib.FP16) if state_calls(lib, op) is not None else None
        rc, _ = workspace_query(lib, h, op, limit + 1, _lib.FP16)
        assert rc == _lib.ERR_UNSUPPORTED and str(limit) in lib.srwn_last_error().decode()
        n0 = _lib.launch_count()
        for call in entry_points(lib, h, op, limit + 1, _lib.FP16, io, state, None, 0):
            assert call() == rc
            assert str(limit) in lib.srwn_last_error().decode()
        assert _lib.launch_count() == n0


def test_encoder_workspace_refuses_what_encode_refuses(models):
    eng = models["teacher"]._enc_eng
    eng.set_weights(synth.make_encoder_weights())
    lib, e = _lib.load(), eng.h
    x, out = torch.zeros(B, T, device="cuda"), torch.zeros(B, T // P, 32, device="cuda")
    n = ctypes.c_size_t()
    assert lib.srwn_encoder_supports(e, _lib.FP16) == 1
    for prec in (_lib.BF16, 7):
        assert lib.srwn_encoder_supports(e, prec) == 0
        rc = lib.srwn_encoder_workspace_bytes(e, B, T, prec, ctypes.byref(n))
        assert rc == _lib.ERR_UNSUPPORTED
        assert lib.srwn_teacher_encode(e, x.data_ptr(), out.data_ptr(), B, T, prec, None, 0, None) == rc
    for prec in (_lib.FP32, _lib.FP16):
        _lib.check(lib.srwn_encoder_workspace_bytes(e, B, T, prec, ctypes.byref(n)))
