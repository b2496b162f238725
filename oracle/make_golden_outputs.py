"""Freeze what tests/test_oracle_vs_reference.py, tests/test_utils.py and tests/test_generators.py compare against the
UNMODIFIED reference into tests/golden/reference_outputs.json, so that those comparisons run without the reference tree.

TEST INFRASTRUCTURE ONLY; needs a reference checkout (see oracle/ref_import.py):
    python -m oracle.make_golden_outputs
Arrays the tests compare exactly are stored as cases.digest (shape + SHA-256), scalars and arrays compared within a
tolerance as values (JSON floats round-trip float64 exactly)."""
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import cases, ref_import, ref_torch  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")


def t(x):
    return torch.from_numpy(np.ascontiguousarray(x))


def layers(vxm_ref):
    shape = (10, 14, 12)
    src = cases.smooth_volume(1, shape)
    flow = cases.smooth_field(2, 3, shape, scale=5.0)
    lab = cases.label_volume(3, shape)
    out = dict(warp=cases.digest(vxm_ref.layers.SpatialTransformer(shape)(t(src), t(flow)).numpy()),
               warp_nearest=cases.digest(vxm_ref.layers.SpatialTransformer(shape, mode="nearest")(t(lab), t(flow)).numpy()),
               vecint5=cases.digest(vxm_ref.layers.VecInt(shape, 5)(t(flow)).numpy()))
    for vr in (2, 0.5):
        out["resize_%s" % vr] = cases.digest(vxm_ref.layers.ResizeTransform(vr, 3)(t(flow)).numpy())
    return out


def losses(vxm_ref):
    NCC = ref_import.reference_ncc_class(vxm_ref)
    I, J = cases.volume_pair(7, (16, 20, 18))
    f = cases.smooth_field(8, 3, (8, 10, 12), scale=2.0)
    return dict(ncc=NCC().loss(t(I), t(J)).item(), grad_l2=vxm_ref.losses.Grad("l2", loss_mult=2).loss(None, t(f)).item(),
                mse=vxm_ref.losses.MSE().loss(t(I), t(J)).item())


def network(vxm_ref):
    kw = dict(inshape=(16, 16, 32), nb_unet_features=[[4, 8, 8, 8], [8, 8, 8, 8, 8, 4, 4]], bidir=True)
    m = vxm_ref.networks.VxmDense(**kw)
    sd = ref_torch.init_state_dict(m.config, seed=5, flow_std=2e-2)
    m.load_state_dict(sd, strict=False)
    s, g = cases.volume_pair(9, kw["inshape"])
    with torch.no_grad():
        a = m(t(s), t(g))
    return dict(config=dict(m.config), outputs=[cases.digest(x.numpy()) for x in a])


def eval_helpers(vxm_ref):
    """Dice and Jacobian determinant of reference py/utils.py on the inputs of test_oracle_vs_reference (RandomState(5))
    and of test_utils (RandomState(2))."""
    nd_mod = sys.modules["pystrum.pynd.ndutils"]
    if not hasattr(nd_mod, "volsize2ndgrid"):   # pystrum, absent here, is stubbed at import: its documented meshgrid
        nd_mod.volsize2ndgrid = lambda volshape: np.meshgrid(*[np.arange(s) for s in volshape], indexing="ij")
    utils = vxm_ref.py.utils
    out = {}
    rng = np.random.RandomState(5)
    a, b = rng.randint(0, 5, size=(9, 10, 11)), rng.randint(0, 6, size=(9, 10, 11))
    out["dice"] = utils.dice(a, b).tolist()
    out["dice_labels"] = utils.dice(a, b, labels=[1, 3, 7], include_zero=True).tolist()
    for shape in ((7, 9), (6, 7, 8)):
        disp = np.moveaxis(cases.smooth_field(11, len(shape), shape, scale=3.0)[0], 0, -1).astype(np.float64)
        out["jacdet_%dd" % len(shape)] = utils.jacobian_determinant(disp).tolist()
    import test_utils
    rng = np.random.RandomState(2)
    a, b = rng.randint(0, 5, size=(9, 10, 11)), rng.randint(0, 5, size=(9, 10, 11))
    out["utils_dice"] = utils.dice(a, b).tolist()
    out["utils_jacdet"] = [utils.jacobian_determinant(d).tolist() for d in list(test_utils.fields())[:2]]
    return out


def generators(vxm_ref):
    import test_generators as tg
    with tempfile.TemporaryDirectory() as d:
        files = tg.make_dataset(d)
        return {name: tg.fingerprint(tg.run_case(vxm_ref.generators, files, case)) for name, case in sorted(tg.CASES.items())}


def main():
    vxm_ref = ref_import.import_reference()
    torch.set_num_threads(8)
    out = dict(layers=layers(vxm_ref), losses=losses(vxm_ref), network=network(vxm_ref), eval_helpers=eval_helpers(vxm_ref),
               generators=generators(vxm_ref))
    with open(OUT, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote", OUT, "%.1f KB" % (os.path.getsize(OUT) / 1024))


if __name__ == "__main__":
    main()
