"""-m gpu: the fp32-grade residual stack (csrc/stack_f32.cu) is one runner for inference and for the forward of the
distillation step, and its launch sites opt in to large dynamic shared memory on every call, whichever device runs it."""
import numpy as np
import pytest
import torch

from sr_wavenet_b200 import synth, _lib

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def srwn(lib):
    import sr_wavenet_b200
    assert torch.cuda.is_available()
    return sr_wavenet_b200


def _student(srwn, dil, F, C, P, seed=11):
    s = srwn.ParallelWaveNet(input_size=0, condition_size=0, dilations=dil, teacher=None, num_flows=F,
                             skip_channels=128, latent_channels=C, pool_stride=P, alpha=0.25, beta=1.0, gamma=1.0)
    s.set_weights(synth.make_student_weights(dil, num_flows=F, latent_channels=C, seed=seed))
    return s


def _inputs(B, T, P, C, M, seed=5):
    rng = np.random.default_rng(seed)
    z = rng.logistic(0, 1, size=(B, T)).astype(np.float32)
    truth = synth.synthetic_audio(B, T)
    enc = rng.normal(0, 1, size=(B, T // P, C)).astype(np.float32)
    tl = (rng.normal(0, 1, size=(B, T, 4 * M)) * 0.5).astype(np.float32)
    return z, truth, enc, tl


@pytest.mark.parametrize("cfg", ["default", "many_tiles"])
def test_training_forward_equals_inference_forward(srwn, cfg):
    """srwn_student_forward_train keeps every layer input but computes what srwn_student_forward computes at SRWN_FP32,
    bit for bit: the distillation step differentiates the inference network.  many_tiles: 2 x 16384 samples are 256
    tiles of 128 steps over one CTA per SM, so CTAs walk more than one tile."""
    if cfg == "default":
        dil, F, C, P, B, T = synth.DEFAULT_DILATIONS, 4, 32, 128, 1, 1280
    else:
        dil, F, C, P, B, T = synth.DEFAULT_DILATIONS, 2, 32, 128, 2, 16384
    s = _student(srwn, dil, F, C, P)
    eng, st = s._eng, torch.cuda.current_stream().cuda_stream
    z_np, _, enc_np, _ = _inputs(B, T, P, C, 3)
    z, enc = torch.from_numpy(z_np).cuda(), torch.from_numpy(enc_np).cuda()

    def run(train):
        out, s_tot, mu_tot = (torch.full((B, T), float("nan"), device="cuda") for _ in range(3))
        if train:
            ws, wsn = eng.workspace(_lib.OP_STUDENT_TRAIN, B, T, _lib.FP32)
            _lib.check(eng.lib.srwn_student_forward_train(eng.h, z.data_ptr(), enc.data_ptr(), out.data_ptr(), s_tot.data_ptr(),
                                                          mu_tot.data_ptr(), B, T, ws, wsn, st))
        else:
            ws, wsn = eng.workspace(_lib.OP_STUDENT_FORWARD, B, T, _lib.FP32)
            _lib.check(eng.lib.srwn_student_forward(eng.h, z.data_ptr(), enc.data_ptr(), out.data_ptr(), s_tot.data_ptr(),
                                                    mu_tot.data_ptr(), None, B, T, _lib.FP32, ws, wsn, st))
        return out, s_tot, mu_tot

    s._eng.set_profiling(True)
    try:
        train = run(True)
        with pytest.raises(RuntimeError):      # the training forward is not profiled: no profiled call yet
            s._eng.last_kernel_ms()
        ref = run(False)
        assert s._eng.last_kernel_ms()[1:] == (len(dil), "k_fwd_layer (3xTF32)")
        run(True)
        assert s._eng.last_kernel_ms()[1:] == (len(dil), "k_fwd_layer (3xTF32)")
    finally:
        s._eng.set_profiling(False)
    for name, a, b in zip(("out", "s_tot", "mu_tot"), train, ref):
        assert torch.isfinite(b).all(), name
        assert torch.equal(a, b), name


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_two_devices_in_one_process(srwn):
    """The same student and the same encoder on cuda:0 and then on cuda:1 of one process: every kernel that needs more
    than 48 KB of dynamic shared memory is set up on the device that launches it, and the results agree bit for bit."""
    dil, F, C, P, M, B, T = [1, 2, 4, 8], 2, 8, 128, 3, 2, 1024
    z, truth, enc, tl = _inputs(B, T, P, C, M)
    x = synth.synthetic_audio(3, 1280, seed=77)
    grads, encodings = [], []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            s = _student(srwn, dil, F, C, P)
            _, _, _, flat = s.loss_and_grads(z, truth, enc, teacher_logits=tl)
            assert flat.device == torch.device("cuda", dev)
            grads.append(flat.cpu())
            t = srwn.WaveNetAutoEncoder(input_size=1280, condition_size=0, num_mixtures=5, dilations=synth.DEFAULT_DILATIONS,
                                        skip_channels=128, latent_channels=32, pool_stride=128)
            t.set_weights(synth.make_encoder_weights(len(synth.DEFAULT_DILATIONS), seed=44))
            encodings.append(t.encode(x, precision="fp16"))
            torch.cuda.synchronize()
            del s, t
    assert torch.isfinite(grads[0]).all() and grads[0].abs().max() > 0
    assert torch.equal(grads[0], grads[1])
    assert np.array_equal(encodings[0], encodings[1])
