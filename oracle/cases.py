"""Deterministic synthetic inputs shared by oracle/make_golden.py, tests/ and bench.py.

TEST INFRASTRUCTURE ONLY.  Everything is generated with numpy's PCG64 streams and exact
float32 arithmetic (adds / multiplies only, no transcendental functions), so the same
arrays are reproduced bit for bit on the GPU box.
"""
import hashlib

import numpy as np

F32 = np.float32


def digest(a):
    """Shape and SHA-256 of the values of `a` (widened to float64, -0.0 folded into 0.0): two float arrays have the same
    digest exactly when np.array_equal holds, so a frozen digest stands for the array in an exact comparison."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64) + 0.0)
    return [list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()]


def _lerp_axis(x, out_n, axis):
    """Exact-arithmetic linear upsampling along one axis (align_corners), float32 ops only."""
    n = x.shape[axis]
    pos = (np.arange(out_n, dtype=np.float64) * (n - 1) / max(out_n - 1, 1))
    i0 = np.minimum(np.floor(pos).astype(np.int64), n - 1)
    i1 = np.minimum(i0 + 1, n - 1)
    lam = (pos - i0).astype(F32)
    sh = [1] * x.ndim
    sh[axis] = -1
    a = np.take(x, i0, axis=axis)
    b = np.take(x, i1, axis=axis)
    return (a + (b - a) * lam.reshape(sh)).astype(F32)


def smooth_field(seed, channels, shape, coarse=None, scale=1.0):
    """Smooth random field (1, channels, *shape): coarse uniform(-1,1) lattice, linearly upsampled."""
    rng = np.random.Generator(np.random.PCG64(seed))
    nd = len(shape)
    if coarse is None:
        coarse = [max(2, s // 16 + 2) for s in shape]
    lat = (rng.random((1, channels) + tuple(coarse), dtype=F32) * F32(2) - F32(1)) * F32(scale)
    out = lat.astype(F32)
    for a in range(nd):
        out = _lerp_axis(out, shape[a], a + 2)
    return out


def smooth_volume(seed, shape, noise=0.05):
    """Image-like volume in [0,1] (1,1,*shape): smooth structure plus a little white noise."""
    rng = np.random.Generator(np.random.PCG64(seed + 7919))
    base = smooth_field(seed, 1, shape, coarse=[max(3, s // 8 + 1) for s in shape], scale=1.0)
    vol = (base * F32(0.5) + F32(0.5)).astype(F32)
    vol = vol + (rng.random(vol.shape, dtype=F32) - F32(0.5)) * F32(noise)
    return np.clip(vol, 0, 1).astype(F32)


def label_volume(seed, shape, nlabels=30):
    """Blocky integer label map (1,1,*shape) float32: nearest-upsampled random coarse labels."""
    rng = np.random.Generator(np.random.PCG64(seed + 104729))
    coarse = [max(2, s // 6) for s in shape]
    lab = rng.integers(0, nlabels, size=(1, 1) + tuple(coarse)).astype(F32)
    for a, s in enumerate(shape):
        idx = (np.arange(s) * coarse[a]) // s
        lab = np.take(lab, idx, axis=a + 2)
    return lab


def volume_pair(seed, shape, sigma=3.0):
    """(source, target): target is the source volume resampled through a smooth displacement
    (pure numpy trilinear gather), so image losses and registration are non-degenerate."""
    from . import spec_np
    src = smooth_volume(seed, shape)
    flow = smooth_field(seed + 1, len(shape), shape, scale=sigma)
    trg = spec_np.warp(src, flow)
    return src, trg
