"""CPU side of the WaveNet / SiameseWaveNet heads (model.py:8-72, 660-798): the variable names and shapes this build creates
are the ones the reference's graph creates (checked against the fixture, and against the reference itself when
SRWN_REFERENCE_DIR names a checkout of it), and the committed fixture is what the reference's source produces today."""
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN

HERE = os.path.dirname(os.path.abspath(__file__))


def _fixture():
    with np.load(os.path.join(GOLDEN, "reference_heads.npz")) as z:
        return {k: z[k] for k in z.files}


def _cfg(g):
    return {k[4:]: g[k] for k in g if k.startswith("cfg_")}


def _build(g):
    from sr_wavenet_b200.heads import WaveNet, SiameseWaveNet
    c = _cfg(g)
    dil = [int(d) for d in c["dilations"]]
    wn = WaveNet(int(c["input_size"]), int(c["output_channels"]), dil, int(c["filter_width"]), int(c["dilation_channels"]),
                 int(c["skip_channels"]), int(c["output_channels"]))
    si = SiameseWaveNet(int(c["input_size"]), int(c["output_dimensions"]), dil, float(c["margin"]), int(c["filter_width"]),
                        int(c["dilation_channels"]), int(c["skip_channels"]))
    return wn, si


def test_variable_names_and_shapes_match_the_reference_graph():
    g = _fixture()
    wn, si = _build(g)
    for net, tag in ((wn, "wn"), (si, "si")):
        assert sorted(net.network_params) == [str(n) for n in g[tag + "_names"]]
        shapes = net._net.shapes
        for n in net.network_params:
            assert tuple(g["%s_w/%s" % (tag, n)].shape) == shapes[n], n
    assert len(wn.network_params) == 2 + 8 * 5 + 4            # front conv, (filter, gate, residual, skip) x (kernel, bias) per block, two 1x1 convs


def test_train_is_refused_loudly():
    g = _fixture()
    wn, si = _build(g)
    with pytest.raises(NotImplementedError):
        wn.train(g["wn_x"], g["wn_targets"])
    with pytest.raises(NotImplementedError):
        si.train(None, g["si_xl"], g["si_xr"], g["si_labels"])


def test_fixture_is_what_the_reference_produces():
    import refshim
    if not refshim.available():
        pytest.skip("SRWN_REFERENCE_DIR does not name a reference checkout")
    sys.path.insert(0, GOLDEN)
    import make_reference_heads_golden as mk
    fresh, g = mk.compute(), _fixture()
    assert sorted(fresh) == sorted(g)
    for k in g:
        if g[k].dtype.kind in "US":
            assert list(fresh[k]) == list(g[k])
        else:
            np.testing.assert_allclose(fresh[k], g[k], rtol=1e-12, atol=1e-14, err_msg=k)
