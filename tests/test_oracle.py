"""CPU tests: the oracle restatements (oracle/spec_np.py, oracle/ref_torch.py) against the golden
vectors frozen from the unmodified reference (oracle/make_golden.py), plus closed-form known answers
(SURVEY.md section 8(c) iv)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import cases, ref_torch, spec_np

from conftest import GOLDEN


def t(x):
    return torch.from_numpy(np.ascontiguousarray(x))


def test_warp_spec_matches_reference_bitwise(golden):
    g = golden("layers")
    assert np.array_equal(spec_np.warp(g["src"], g["flow"]), g["warp_lin"])
    assert np.array_equal(spec_np.warp(g["lab"], g["flow"], mode="nearest"), g["warp_near"])
    assert np.array_equal(spec_np.warp(g["lab"][:1], g["tie_flow"], mode="nearest"), g["warp_near_tie"])
    assert np.array_equal(spec_np.warp(g["src"][:1], g["tie_flow"]), g["warp_lin_tie"])
    assert np.array_equal(spec_np.warp(g["lab2"], g["flow2"], mode="nearest"), g["warp2_near"])
    np.testing.assert_allclose(spec_np.warp(g["src2"], g["flow2"]), g["warp2_lin"], rtol=0, atol=5e-7)


def test_warp_torch_restatement(golden):
    g = golden("layers")
    assert np.array_equal(ref_torch.spatial_transform(t(g["src"]), t(g["flow"])).numpy(), g["warp_lin"])
    assert np.array_equal(ref_torch.spatial_transform(t(g["lab"]), t(g["flow"]), "nearest").numpy(), g["warp_near"])
    assert np.array_equal(ref_torch.spatial_transform(t(g["src2"]), t(g["flow2"])).numpy(), g["warp2_lin"])


def test_vecint(golden):
    g = golden("layers")
    for n in (0, 1, 4, 7):
        assert np.array_equal(spec_np.vecint(g["vel"], n), g["vecint_%d" % n])
        assert np.array_equal(ref_torch.vec_int(t(g["vel"]), n).numpy(), g["vecint_%d" % n])
    np.testing.assert_allclose(spec_np.vecint(g["vel2"], 5), g["vecint2_5"], rtol=0, atol=2e-6)


def test_resize(golden):
    g = golden("layers")
    for key, x, vr in (("resize_down", "flow", 2), ("resize_up", "flow", 0.5), ("resize_one", "flow", 1),
                       ("resize_down_odd", "odd", 2), ("resize_up_odd", "odd", 0.5),
                       ("resize2_down", "flow2", 2), ("resize2_up", "flow2", 0.5)):
        o = spec_np.resize_flow(g[x], vr)
        assert o.shape == g[key].shape, key
        np.testing.assert_allclose(o, g[key], rtol=0, atol=4e-6 * max(1.0, np.abs(g[key]).max()), err_msg=key)
        assert np.array_equal(ref_torch.resize_transform(t(g[x]), vr).numpy(), g[key]), key


def test_losses(golden):
    g = golden("losses")
    assert abs(spec_np.ncc_loss(g["I"], g["J"]) - g["ncc"]) < 2e-6
    assert abs(spec_np.ncc_loss(g["I"], g["J"], [5, 5, 5]) - g["ncc5"]) < 2e-6
    assert abs(spec_np.ncc_loss(g["I2"], g["J2"]) - g["ncc2"]) < 2e-6
    gr = spec_np.ncc_grad_pred(g["I"], g["J"])
    assert np.abs(gr - g["ncc_grad"]).max() < 1e-3 * np.abs(g["ncc_grad"]).max()
    assert abs(ref_torch.ncc_loss(t(g["I"]), t(g["J"])).item() - g["ncc"]) < 1e-7
    assert abs(spec_np.mse_loss(g["I"], g["J"]) - g["mse"]) < 1e-7
    assert abs(spec_np.grad_loss(g["gflow"], "l2", 2) - g["grad_l2"]) < 1e-6 * abs(g["grad_l2"])
    assert abs(spec_np.grad_loss(g["gflow"], "l1") - g["grad_l1"]) < 1e-6 * abs(g["grad_l1"])
    assert abs(ref_torch.grad_loss(t(g["gflow"]), "l2", 2).item() - g["grad_l2"]) < 1e-6 * abs(g["grad_l2"])
    assert abs(spec_np.dice_loss(g["dice_true"], g["dice_pred"]) - g["dice"]) < 1e-6
    assert abs(ref_torch.dice_loss(t(g["dice_true"]), t(g["dice_pred"])).item() - g["dice"]) < 1e-6


VARIANTS = {
    "default3d": dict(inshape=(32, 32, 48)),
    "small3d": dict(inshape=(16, 32, 16), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]]),
    "nodiffeo3d": dict(inshape=(16, 16, 16), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]], int_steps=0),
    "bidir_full3d": dict(inshape=(16, 16, 16), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]], bidir=True,
                         int_downsize=1),
    "halfres3d": dict(inshape=(16, 16, 32), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]], unet_half_res=True),
    "intfeat3d": dict(inshape=(16, 16, 16), nb_unet_features=4, nb_unet_levels=3, unet_feat_mult=2,
                      nb_unet_conv_per_level=2),
    "config1_2d": dict(inshape=(64, 64), int_steps=0),
    "diffeo2d": dict(inshape=(32, 48), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]], int_steps=5),
}
DEFAULTS = dict(nb_unet_features=None, nb_unet_levels=None, unet_feat_mult=1, nb_unet_conv_per_level=1, int_steps=7,
                int_downsize=2, bidir=False, use_probs=False, src_feats=1, trg_feats=1, unet_half_res=False)


def full_cfg(kw):
    c = dict(DEFAULTS)
    c.update(kw)
    return c


@pytest.fixture
def golden_threads():
    """torch's CPU convolutions split their sums by thread count, so their bits depend on it: bit-exact comparisons with
    the vectors oracle/make_golden.py froze run with the 8 threads it used, whatever the machine's core count."""
    prev = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(prev)


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_vxmdense_restatement_against_reference(golden, golden_threads, name):
    """ref_torch.vxm_forward (functional restatement) == reference VxmDense.forward, all ctor variants."""
    g = golden("vxmdense")
    cfg = full_cfg(VARIANTS[name])
    sd = ref_torch.init_state_dict(cfg, seed=1234, flow_std=2e-2)
    s, tr = cases.volume_pair(91, cfg["inshape"], sigma=1.5)
    with torch.no_grad():
        out = ref_torch.vxm_forward(sd, cfg, t(s), t(tr))
        reg = ref_torch.vxm_forward(sd, cfg, t(s), t(tr), registration=True)
    for i, y in enumerate(out):
        assert np.array_equal(y.numpy(), g["%s/train%d" % (name, i)]), (name, i)
    assert np.array_equal(reg[1].numpy(), g["%s/reg_flow" % name])


def test_known_answers():
    shape = (8, 10, 12)
    src = cases.smooth_volume(3, shape)
    lab = cases.label_volume(4, shape)
    zero = np.zeros((1, 3) + shape, np.float32)
    # zero flow = identity; only to ~1 ulp for linear: the reference's normalise/unnormalise round trip
    # (layers.py:37, GridSampler.h:27-31) is not exact for every index
    np.testing.assert_allclose(spec_np.warp(src, zero), src, rtol=0, atol=2e-6)
    assert np.array_equal(spec_np.warp(lab, zero, "nearest"), lab)
    sh = zero.copy()
    sh[:, 2] = 2.0                                                            # integer shift along W, zero fill
    out = spec_np.warp(src, sh)
    np.testing.assert_allclose(out[..., :-2], src[..., 2:], rtol=0, atol=2e-6)
    assert np.abs(out[..., -2:]).max() < 2e-6
    outn = spec_np.warp(lab, sh, "nearest")
    assert np.array_equal(outn[..., :-2], lab[..., 2:]) and not outn[..., -2:].any()
    v = cases.smooth_field(5, 3, shape, scale=2.0)
    assert np.array_equal(spec_np.vecint(v, 0), v)                            # VecInt(0) = identity
    assert np.array_equal(spec_np.resize_flow(v, 1), v)                       # ResizeTransform(1) = identity
    ramp = np.zeros((1, 3) + shape, np.float32)
    ramp[:, 0] = np.arange(shape[0], dtype=np.float32)[:, None, None] * 0.5   # slope .5 along D only
    assert abs(spec_np.grad_loss(ramp, "l2") - 0.25 / 9) < 1e-7   # 1 of 3 channels, 1 of 3 axes
    a = (cases.label_volume(6, shape, 2) > 0).astype(np.float32)
    assert abs(spec_np.dice_loss(a, a) + 1) < 1e-6                            # Dice(x,x) = -1
    c = np.full((1, 3) + shape, 0.25, np.float32)                             # constant velocity -> constant in interior
    out = spec_np.vecint(c, 4)
    assert np.allclose(out[..., :4, :4, :4], 0.25, atol=1e-6)   # away from the high border, where zeros padding bleeds in


def test_digests_present():
    d = json.load(open(os.path.join(GOLDEN, "digests.json")))
    assert len(d["nearest_full_sha256"]) == 64


def test_adam_restatement():
    rng = np.random.default_rng(0)
    p = rng.standard_normal(100)
    m = np.zeros(100)
    v = np.zeros(100)
    tp = torch.tensor(p, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.Adam([tp], lr=1e-3)
    for step in range(1, 4):
        g = rng.standard_normal(100)
        tp.grad = torch.tensor(g)
        opt.step()
        p, m, v = spec_np.adam_step(p, g, m, v, step, lr=1e-3)
        np.testing.assert_allclose(tp.detach().numpy(), p, rtol=1e-12, atol=1e-14)


def test_eval_helpers_known_answers():
    """Oracle of the next rows N2 / N3 (Dice overlap, Jacobian determinant): closed-form cases."""
    from oracle import spec_np
    for shape in ((6, 7), (5, 6, 7)):
        nd = len(shape)
        grid = np.stack(np.meshgrid(*[np.arange(s, dtype=np.float64) for s in shape], indexing="ij"), -1)
        assert np.allclose(spec_np.jacobian_determinant(np.zeros(shape + (nd,))), 1.0)          # identity map
        assert np.allclose(spec_np.jacobian_determinant(0.1 * grid), 1.1 ** nd)                 # uniform dilation
        fold = -2.0 * grid                                                                       # x -> -x: orientation flips per axis
        assert np.allclose(spec_np.jacobian_determinant(fold), (-1.0) ** nd)
    a = np.array([[0, 1, 1], [2, 2, 0]])
    assert np.array_equal(spec_np.dice_overlap(a, a), [1.0, 1.0])
    b = np.array([[0, 1, 0], [2, 0, 0]])
    assert np.allclose(spec_np.dice_overlap(a, b), [2 * 1 / 3, 2 * 1 / 3])
    assert np.allclose(spec_np.dice_overlap(a, b, labels=[5]), [0.0])
