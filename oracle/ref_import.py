"""Import the *unmodified* reference (voxelmorph @ /root/reference) on CPU.

TEST INFRASTRUCTURE ONLY: used by `oracle/make_golden*.py` to freeze the reference's
outputs into `tests/golden/`, against which the tests pin the restatements in
`oracle/spec_np.py` / `oracle/ref_torch.py` and the product package.  The tests never
import the reference.

The reference hard-imports three packages that are absent from this image and
irrelevant to the torch hot path (`neurite`, `skimage.measure`, `pystrum`):
reference voxelmorph/__init__.py:12, voxelmorph/py/utils.py:10,13.  They are stubbed
in `sys.modules`; no reference file is modified or copied.
"""
import inspect
import math
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("VXM_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "voxelmorph", "torch"))


def import_reference():
    """Return the reference `voxelmorph` module (torch backend)."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    os.environ["VXM_BACKEND"] = "pytorch"
    os.environ["NEURITE_BACKEND"] = "pytorch"
    if "voxelmorph" in sys.modules and getattr(sys.modules["voxelmorph"], "__file__", "").startswith(REFERENCE_ROOT):
        return sys.modules["voxelmorph"]
    if "voxelmorph" in sys.modules:
        raise RuntimeError("a different `voxelmorph` is already imported: %r" % sys.modules["voxelmorph"].__file__)
    ne = types.ModuleType("neurite")
    ne.__version__ = "0.2"
    sys.modules.setdefault("neurite", ne)
    sk = types.ModuleType("skimage")
    sk.measure = types.ModuleType("skimage.measure")
    sys.modules.setdefault("skimage", sk)
    sys.modules.setdefault("skimage.measure", sk.measure)
    for name in ("pystrum", "pystrum.pynd", "pystrum.pynd.ndutils"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["pystrum"].pynd = sys.modules["pystrum.pynd"]
    sys.modules["pystrum.pynd"].ndutils = sys.modules["pystrum.pynd.ndutils"]
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        import voxelmorph as vxm  # noqa
    finally:
        sys.path.remove(REFERENCE_ROOT)
    return vxm


def reference_ncc_class(vxm):
    """The reference NCC hard-codes `.to("cuda")` (voxelmorph/torch/losses.py:29).

    For the CPU oracle the class source is re-executed in memory with that token
    removed; nothing else changes.
    """
    import numpy as np
    import torch
    import torch.nn.functional as F
    src = inspect.getsource(vxm.losses.NCC).replace('.to("cuda")', "")
    ns = dict(torch=torch, F=F, np=np, math=math)
    exec(src, ns)
    return ns["NCC"]
