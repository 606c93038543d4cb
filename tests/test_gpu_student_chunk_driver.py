"""-m gpu: ``student.py --test --chunk S`` synthesizes each clip in calls of S samples through one synthesis state and
writes the same audio as the one-call run with the same host noise."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_student_driver_chunked_test_writes_the_same_wav(lib, tmp_path):
    import sr_wavenet_b200 as srwn
    import student as drv
    from scipy.io import wavfile
    assert torch.cuda.is_available()
    tdir, sdir = str(tmp_path / "teacher"), str(tmp_path / "student")
    srwn.WaveNetAutoEncoder(input_size=4096, condition_size=0, num_mixtures=5, dilations=drv.DILATIONS, latent_channels=32,
                            skip_channels=128, pool_stride=128).save(tdir, 1, force=True)
    srwn.ParallelWaveNet(input_size=4096, condition_size=0, dilations=drv.DILATIONS, teacher=tdir, num_flows=4,
                         skip_channels=128, latent_channels=32, pool_stride=128).save(None, sdir, 1, force=True)
    common = ["--teacher", tdir, "--student", sdir, "--num-samples", "4096", "--batch-size", "2", "--test", "--clips", "2",
              "--seed", "7"]
    one, chunked = str(tmp_path / "one"), str(tmp_path / "chunked")
    drv.main(common + ["--out-dir", one])
    res = drv.main(common + ["--out-dir", chunked, "--chunk", "2048"])
    assert res["output_shape"] == (2, 4096, 1)
    for step in range(2):
        name = "student_wav_%d.wav" % step
        ra, a = wavfile.read(os.path.join(one, name))
        rb, b = wavfile.read(os.path.join(chunked, name))
        assert ra == rb and a.shape == (4096,)
        np.testing.assert_array_equal(a, b)
    with pytest.raises(SystemExit):
        drv.main(common + ["--out-dir", chunked, "--chunk", "100"])
