"""-m gpu: the team wavefront of the fused kernel (csrc/fused.cu).  A piece of the (utterance, chunk) line is walked
by a team of G CTAs that hand the per-layer history rings from CTA to CTA through global memory and flags; the result
must not depend on G (G = 1 is the one-CTA-per-piece schedule with no hand-off), on the partition, or on the batch order."""
import numpy as np
import pytest
import torch

from conftest import f64
from oracle import srwn_oracle as orc
from sr_wavenet_b200 import synth, _lib

pytestmark = pytest.mark.gpu
DIL = synth.DEFAULT_DILATIONS


@pytest.fixture(scope="module")
def srwn(lib):
    import sr_wavenet_b200
    assert torch.cuda.is_available()
    return sr_wavenet_b200


@pytest.mark.parametrize("B,T", [(1, 64000), (3, 20096), (5, 8192)])
def test_teacher_is_bit_identical_for_every_team_size(srwn, B, T):
    t = srwn.WaveNetAutoEncoder(input_size=T, condition_size=0, num_mixtures=5, dilations=DIL, skip_channels=128,
                                latent_channels=32, pool_stride=128)
    w = synth.make_teacher_weights(DIL)
    t.set_weights(w)
    x = torch.from_numpy(synth.synthetic_audio(B, T, seed=21)).cuda()
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // 128, seed=22)).cuda()
    ref = None
    seen = []
    for G in (1, 2, 3, 4, 7, 8, 16, 18, 0):
        t._eng.set_team_size(G)
        lg = t.get_logits(x, enc, precision="fp16")
        nll = t.nll(x, enc, sum_all=False, precision="fp16")
        t._eng.check_async(_lib.OP_TEACHER_NLL, B, T, _lib.FP16)
        seen.append((G,) + t._eng.last_partition())
        if ref is None:
            ref = (lg.clone(), nll.clone())
        else:
            assert torch.equal(lg, ref[0]) and torch.equal(nll, ref[1]), "team size %d changes the result" % G
    print("teacher %dx%d partitions (requested G, teams, G):" % (B, T), seen)
    # and the result is the oracle's (one utterance)
    o = orc.teacher_decoder_logits(f64(w), x[:1].cpu().numpy().astype(np.float64), enc[:1].cpu().numpy().astype(np.float64), DIL, 128)
    assert np.abs(ref[0][:1].cpu().numpy() - o).max() <= 1e-2


def test_student_is_bit_identical_for_every_team_size(srwn):
    B, T = 2, 32000
    s = srwn.ParallelWaveNet(input_size=T, condition_size=0, dilations=DIL, teacher=None, num_flows=4, skip_channels=128,
                             latent_channels=32, pool_stride=128)
    s.set_weights(synth.make_student_weights(DIL, 4))
    z = torch.from_numpy(synth.logistic_noise(B, T, seed=5)).cuda()
    enc = torch.from_numpy(synth.synthetic_encoding(B, T // 128, seed=6)).cuda()
    ref = None
    for G in (1, 2, 4, 9, 18, 0):
        s._eng.set_team_size(G)
        r = s.forward_all(z, enc, precision="fp16")
        s._eng.check_async(_lib.OP_STUDENT_FORWARD, B, T, _lib.FP16)
        if ref is None:
            ref = {k: v.clone() for k, v in r.items()}
        else:
            for k in ref:
                assert torch.equal(r[k], ref[k]), (G, k)
    assert all(torch.isfinite(v).all() for v in ref.values())


def test_small_batches_run_near_the_large_batch_rate(srwn):
    """The point of the hand-off: 4 x 64000 (the 8-GPU share of configs[1]) no longer pays the receptive-field warm-up
    per CTA.  Kernel time per sample within 25 % of the 32 x 64000 rate (it was 1.6x before)."""
    t = srwn.WaveNetAutoEncoder(input_size=64000, condition_size=0, num_mixtures=5, dilations=DIL, skip_channels=128,
                                latent_channels=32, pool_stride=128)
    t.set_weights(synth.make_teacher_weights(DIL))
    t._eng.set_profiling(True)
    rate = {}
    for B in (32, 4):
        x = torch.from_numpy(synth.synthetic_audio(B, 64000)).cuda()
        enc = torch.from_numpy(synth.synthetic_encoding(B, 500)).cuda()
        best = 1e9
        for _ in range(4):
            t.nll(x, enc, precision="fp16")
            best = min(best, t._eng.last_kernel_ms()[0])
        t._eng.check_async(_lib.OP_TEACHER_NLL, B, 64000, _lib.FP16)
        rate[B] = B * 64000 / best / 1e3
        print("teacher %dx64000: %.3f ms per launch = %.1f M samples/s, partition %s" % (B, best, rate[B], t._eng.last_partition()))
    assert rate[4] >= 0.65 * rate[32]
