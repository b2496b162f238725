"""Pin of the oracle restatements against outputs of the UNMODIFIED reference, frozen into
tests/golden/reference_outputs.json by oracle/make_golden_outputs.py: arrays compared exactly are stored as cases.digest,
scalars and arrays compared within a tolerance as values."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import cases, ref_torch, spec_np


def t(x):
    return torch.from_numpy(np.ascontiguousarray(x))


@pytest.fixture(scope="module")
def ref():
    return json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))


def test_layers_live(ref):
    ref = ref["layers"]
    shape = (10, 14, 12)
    src = cases.smooth_volume(1, shape)
    flow = cases.smooth_field(2, 3, shape, scale=5.0)
    lab = cases.label_volume(3, shape)
    assert cases.digest(spec_np.warp(src, flow)) == ref["warp"]
    assert cases.digest(spec_np.warp(lab, flow, mode="nearest")) == ref["warp_nearest"]
    assert cases.digest(spec_np.vecint(flow, 5)) == ref["vecint5"]
    for vr in (2, 0.5):
        r = ref_torch.resize_transform(t(flow), vr).numpy()
        assert cases.digest(r) == ref["resize_%s" % vr]         # r is the reference's output
        np.testing.assert_allclose(spec_np.resize_flow(flow, vr), r, rtol=0, atol=5e-6 * np.abs(flow).max())


def test_losses_live(ref):
    ref = ref["losses"]
    I, J = cases.volume_pair(7, (16, 20, 18))
    assert abs(ref["ncc"] - spec_np.ncc_loss(I, J)) < 2e-6
    assert ref["ncc"] == ref_torch.ncc_loss(t(I), t(J)).item()
    f = cases.smooth_field(8, 3, (8, 10, 12), scale=2.0)
    assert abs(ref["grad_l2"] - spec_np.grad_loss(f, "l2", 2)) < 1e-6
    assert abs(ref["mse"] - spec_np.mse_loss(I, J)) < 1e-7


def test_network_live(ref):
    ref = ref["network"]
    kw = dict(inshape=(16, 16, 32), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]], bidir=True)
    cfg = dict(ref["config"], inshape=kw["inshape"])
    assert cfg["nb_unet_features"] == kw["nb_unet_features"] and cfg["bidir"]
    sd = ref_torch.init_state_dict(cfg, seed=5, flow_std=2e-2)
    s, g = cases.volume_pair(9, kw["inshape"])
    with torch.no_grad():
        b = ref_torch.vxm_forward(sd, cfg, t(s), t(g))
    assert [cases.digest(x.numpy()) for x in b] == ref["outputs"]


def test_eval_helpers_live(ref):
    """Next rows N2 / N3: Dice overlap and Jacobian determinant restatements vs reference py/utils.py:265-287, :473-516
    (pystrum's volsize2ndgrid, absent where the outputs were frozen, was supplied as its documented np.meshgrid(indexing='ij'))."""
    ref = ref["eval_helpers"]
    rng = np.random.RandomState(5)
    a, b = rng.randint(0, 5, size=(9, 10, 11)), rng.randint(0, 6, size=(9, 10, 11))
    assert np.array_equal(np.array(ref["dice"]), spec_np.dice_overlap(a, b))
    assert np.array_equal(np.array(ref["dice_labels"]), spec_np.dice_overlap(a, b, [1, 3, 7], True))
    for shape in ((7, 9), (6, 7, 8)):
        disp = cases.smooth_field(11, len(shape), shape, scale=3.0)[0]        # (nd, *vol)
        disp = np.moveaxis(disp, 0, -1).astype(np.float64)
        np.testing.assert_allclose(spec_np.jacobian_determinant(disp), np.array(ref["jacdet_%dd" % len(shape)]), rtol=0, atol=1e-12)
