"""Explicit numpy restatement of the reference's VxmDense hot-path arithmetic.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Nothing here is imported by the
product package.  Every function cites the reference lines it restates; where the
arithmetic lives in PyTorch (a third-party dependency the reference does not pin —
reference setup.py:31-39 lists no torch requirement) the installed torch 2.11.0
ATen headers are cited as [torch] <header>:<line>.

Parity status: the reference ships no tests or golden vectors ("parity unpinned" by
the reference itself).  These restatements are pinned instead against outputs of
the unmodified reference run in the build container (oracle/make_golden.py ->
tests/golden/*.npz, oracle/make_golden_outputs.py -> tests/golden/reference_outputs.json,
checked in tests/test_oracle_vs_reference.py).

All arithmetic is float32 with one rounding per operation (numpy never contracts
to FMA), which is what makes the nearest-neighbour index sequence reproducible
bit for bit.
"""
import numpy as np

F32 = np.float32


# --------------------------------------------------------------------------------------
# SpatialTransformer  (reference voxelmorph/torch/layers.py:30-48)
# --------------------------------------------------------------------------------------

def _sample_coords(flow, div="true"):
    """Per-axis unnormalised sampling coordinate, replaying the reference's fp32 sequence.

    layers.py:32   loc = grid + flow
    layers.py:37   n   = 2 * (loc / (S-1) - 0.5)
    [torch] ATen/native/GridSampler.h:27-31 (align_corners=True)  w = ((n + 1) / 2) * (S-1)

    div='true'  : loc / (S-1) is a true fp32 division (torch CPU).
    div='recip' : loc * fl(1/(S-1)) — what torch's CUDA `tensor / python_scalar` computes
                  (ATen BinaryDivTrueKernel.cu folds a CPU-scalar divisor into a multiply).
    """
    flow = np.asarray(flow, dtype=F32)
    B, nd = flow.shape[:2]
    shape = flow.shape[2:]
    assert nd == len(shape)
    coords = []
    for i, S in enumerate(shape):
        idx = np.arange(S, dtype=F32).reshape([1] + [S if j == i else 1 for j in range(nd)])
        loc = (idx + flow[:, i]).astype(F32)
        sm1 = F32(S - 1)
        if div == "true":
            t = (loc / sm1).astype(F32)
        else:
            t = (loc * (F32(1.0) / sm1)).astype(F32)
        u = (t - F32(0.5)).astype(F32)
        n = (F32(2.0) * u).astype(F32)
        v = (n + F32(1.0)).astype(F32)
        w = ((v / F32(2.0)).astype(F32) * sm1).astype(F32)
        coords.append(w)
    return coords  # list over axes (D,H,W order), each (B, *shape) fp32


def warp(src, flow, mode="bilinear", div="true"):
    """out[b,c,p] = sample(src[b,c], p + flow[b,:,p]) with zeros padding.

    Bilinear weights / corner order follow [torch] aten/src/ATen/native/GridSampler.cpp
    grid_sampler_3d_cpu_impl (corner weights are products of (1 - frac)/(frac) formed as
    (ix_bse - ix) etc.; out-of-volume corners contribute 0).  Nearest:
    idx = nearbyint(coord) (round-half-even), value 0 when out of bounds
    ([torch] GridSampler.h:209-211 within_bounds_3d).
    """
    src = np.asarray(src, dtype=F32)
    coords = _sample_coords(flow, div)
    B, C = src.shape[:2]
    shape = src.shape[2:]
    nd = len(shape)
    out = np.zeros((B, C) + tuple(flow.shape[2:]), dtype=F32)
    bidx = np.arange(B).reshape([B] + [1] * nd)
    if mode == "nearest":
        idx = [np.rint(c).astype(np.int64) for c in coords]  # rint == nearbyint (half-to-even)
        ok = np.ones(idx[0].shape, dtype=bool)
        for i, S in enumerate(shape):
            ok &= (idx[i] >= 0) & (idx[i] < S)
        cl = [np.clip(idx[i], 0, shape[i] - 1) for i in range(nd)]
        for c in range(C):
            g = src[(bidx, c) + tuple(cl)]
            out[:, c] = np.where(ok, g, F32(0))
        return out
    assert mode == "bilinear"
    fl = [np.floor(c) for c in coords]
    i0 = [f.astype(np.int64) for f in fl]
    # weights: (i1 - x) for the low corner, (x - i0) for the high corner   (GridSampler.cpp)
    w_lo = [((fl[i] + F32(1.0)).astype(F32) - coords[i]).astype(F32) for i in range(nd)]
    w_hi = [(coords[i] - fl[i]).astype(F32) for i in range(nd)]
    # corner enumeration: ATen order t/b (axis 0) outermost, then n/s, then w/e fastest
    for c in range(C):
        acc = np.zeros(out.shape[:1] + out.shape[2:], dtype=F32)
        for corner in range(2 ** nd):
            bits = [(corner >> (nd - 1 - a)) & 1 for a in range(nd)]  # axis 0 is the slowest bit
            # weight product order: x-term * y-term * z-term  (last axis first)
            wgt = None
            for a in reversed(range(nd)):
                term = w_hi[a] if bits[a] else w_lo[a]
                wgt = term if wgt is None else (wgt * term).astype(F32)
            ii = [i0[a] + bits[a] for a in range(nd)]
            ok = np.ones(ii[0].shape, dtype=bool)
            for a in range(nd):
                ok &= (ii[a] >= 0) & (ii[a] < shape[a])
            cl = [np.clip(ii[a], 0, shape[a] - 1) for a in range(nd)]
            val = src[(bidx, c) + tuple(cl)]
            acc = np.where(ok, (acc + (val * wgt).astype(F32)).astype(F32), acc)
        out[:, c] = acc
    return out


def vecint(vec, nsteps):
    """Scaling and squaring (reference layers.py:61,64-68)."""
    assert nsteps >= 0
    vec = (np.asarray(vec, dtype=F32) * F32(1.0 / (2 ** nsteps))).astype(F32)
    for _ in range(nsteps):
        vec = (vec + warp(vec, vec)).astype(F32)
    return vec


# --------------------------------------------------------------------------------------
# ResizeTransform (reference layers.py:76-97; [torch] ATen/native/UpSample.h:271-296,442-475)
# --------------------------------------------------------------------------------------

def _lin_index(in_size, out_size):
    if out_size == in_size:
        o = np.arange(out_size)
        return o, o, np.ones(out_size, F32), np.zeros(out_size, F32)
    ratio = F32(in_size - 1) / F32(out_size - 1) if out_size > 1 else F32(0)
    real = (ratio * np.arange(out_size, dtype=F32)).astype(F32)
    i0 = np.minimum(real.astype(np.int64), in_size - 1)
    lam = np.minimum(np.maximum((real - i0.astype(F32)).astype(F32), F32(0)), F32(1))
    i1 = i0 + (i0 < in_size - 1)
    return i0, i1, (F32(1) - lam).astype(F32), lam


def interp_linear(x, out_shape):
    """N-D linear interpolation, align_corners=True (separable lerp, innermost axis first)."""
    x = np.asarray(x, dtype=F32)
    nd = x.ndim - 2
    y = x
    for a in reversed(range(nd)):
        ax = a + 2
        i0, i1, l0, l1 = _lin_index(y.shape[ax], out_shape[a])
        sh = [1] * y.ndim
        sh[ax] = -1
        y = (np.take(y, i0, axis=ax) * l0.reshape(sh) + np.take(y, i1, axis=ax) * l1.reshape(sh)).astype(F32)
    return y


def resize_flow(x, vel_resize):
    """factor = 1/vel_resize; <1: interpolate then scale; >1: scale then interpolate (layers.py:85-97)."""
    x = np.asarray(x, dtype=F32)
    factor = 1.0 / vel_resize
    if factor == 1:
        return x
    out_shape = [int(np.floor(s * factor)) for s in x.shape[2:]]
    if factor < 1:
        return (F32(factor) * interp_linear(x, out_shape)).astype(F32)
    return interp_linear((F32(factor) * x).astype(F32), out_shape)


# --------------------------------------------------------------------------------------
# Losses (reference voxelmorph/torch/losses.py)
# --------------------------------------------------------------------------------------

def box_sum(x, win):
    """Zero-padded box sum over the spatial axes of (B,1,*vol) (losses.py:29-55 ones-filter conv)."""
    x = np.asarray(x)
    nd = x.ndim - 2
    y = x
    for a in range(nd):
        ax = a + 2
        k = win[a]
        pad = k // 2
        pw = [(0, 0)] * y.ndim
        pw[ax] = (pad, pad)
        yp = np.pad(y, pw)
        cs = np.cumsum(yp.astype(np.float64), axis=ax)
        cs = np.concatenate([np.zeros_like(np.take(cs, [0], axis=ax)), cs], axis=ax)
        n = y.shape[ax]
        hi = np.take(cs, np.arange(k, k + n), axis=ax)
        lo = np.take(cs, np.arange(0, n), axis=ax)
        y = hi - lo
    return y


def ncc_cc_map(I, J, win=None, dtype=np.float64):
    """Local squared normalised cross-correlation map (losses.py:47-65).

    Computed in float64 by default: it is the yardstick the fp32 CUDA kernel and the fp32
    reference are both compared against (the variance terms are cancellations).
    """
    I = np.asarray(I, dtype=dtype)
    J = np.asarray(J, dtype=dtype)
    nd = I.ndim - 2
    win = [9] * nd if win is None else list(win)
    n = float(np.prod(win))
    Is, Js = box_sum(I, win), box_sum(J, win)
    I2s, J2s, IJs = box_sum(I * I, win), box_sum(J * J, win), box_sum(I * J, win)
    uI, uJ = Is / n, Js / n
    cross = IJs - uJ * Is - uI * Js + uI * uJ * n
    Ivar = I2s - 2 * uI * Is + uI * uI * n
    Jvar = J2s - 2 * uJ * Js + uJ * uJ * n
    cc = cross * cross / (Ivar * Jvar + 1e-5)
    return cc, dict(cross=cross, Ivar=Ivar, Jvar=Jvar, uI=uI, uJ=uJ)


def ncc_loss(y_true, y_pred, win=None):
    cc, _ = ncc_cc_map(y_true, y_pred, win)
    return -cc.mean()


def ncc_grad_pred(y_true, y_pred, win=None):
    """d(-mean cc)/d(y_pred), closed form (derived from losses.py:57-67; float64)."""
    I = np.asarray(y_true, dtype=np.float64)
    J = np.asarray(y_pred, dtype=np.float64)
    nd = I.ndim - 2
    win = [9] * nd if win is None else list(win)
    cc, t = ncc_cc_map(I, J, win)
    den = t["Ivar"] * t["Jvar"] + 1e-5
    A = 2 * t["cross"] / den
    Bq = -(t["cross"] ** 2) * t["Ivar"] / den ** 2
    g = I * box_sum(A, win) - box_sum(A * t["uI"], win) + 2 * J * box_sum(Bq, win) - 2 * box_sum(Bq * t["uJ"], win)
    return -g / cc.size


def grad_loss(y_pred, penalty="l2", loss_mult=None):
    """Forward-difference smoothness penalty (losses.py:102-135)."""
    y = np.asarray(y_pred, dtype=np.float64)
    nd = y.ndim - 2
    per_axis = []
    for a in range(nd):
        ax = a + 2
        d = np.diff(y, axis=ax)
        d = np.abs(d) if penalty == "l1" else d * d
        per_axis.append(d.reshape(d.shape[0], -1).mean(axis=1))
    g = sum(per_axis) / nd
    if loss_mult is not None:
        g = g * loss_mult
    return g.mean()


def mse_loss(y_true, y_pred):
    d = np.asarray(y_true, np.float64) - np.asarray(y_pred, np.float64)
    return (d * d).mean()


def dice_loss(y_true, y_pred):
    """losses.py:84-90."""
    a = np.asarray(y_true, np.float64)
    b = np.asarray(y_pred, np.float64)
    ax = tuple(range(2, a.ndim))
    top = 2 * (a * b).sum(axis=ax)
    bottom = np.maximum((a + b).sum(axis=ax), 1e-5)
    return -(top / bottom).mean()


# --------------------------------------------------------------------------------------
# U-Net pieces (reference voxelmorph/torch/networks.py:122-144,290-305)
# --------------------------------------------------------------------------------------

def conv_k3(x, w, b=None, leaky=None, dtype=np.float64):
    """3^n convolution, stride 1, zero pad 1 (nn.ConvNd as used at networks.py:211,299) + optional LeakyReLU."""
    x = np.asarray(x, dtype=dtype)
    w = np.asarray(w, dtype=dtype)
    nd = x.ndim - 2
    B, Cin = x.shape[:2]
    Cout = w.shape[0]
    xp = np.pad(x, [(0, 0), (0, 0)] + [(1, 1)] * nd)
    out = np.zeros((B, Cout) + x.shape[2:], dtype=dtype)
    for tap in np.ndindex(*w.shape[2:]):
        sl = tuple(slice(t, t + s) for t, s in zip(tap, x.shape[2:]))
        out += np.einsum("bi...,oi->bo...", xp[(slice(None), slice(None)) + sl], w[(slice(None), slice(None)) + tap])
    if b is not None:
        out += np.asarray(b, dtype=dtype).reshape([1, -1] + [1] * nd)
    if leaky is not None:
        out = np.where(out >= 0, out, out * leaky)
    return out


def maxpool2(x):
    """MaxPool(2) on every spatial axis (networks.py:83,130)."""
    x = np.asarray(x)
    nd = x.ndim - 2
    for a in range(nd):
        ax = a + 2
        n = x.shape[ax] // 2
        lo = np.take(x, np.arange(0, 2 * n, 2), axis=ax)
        hi = np.take(x, np.arange(1, 2 * n, 2), axis=ax)
        x = np.maximum(lo, hi)
    return x


def upsample2_nearest(x):
    """nn.Upsample(scale_factor=2, mode='nearest') (networks.py:84,137)."""
    x = np.asarray(x)
    for a in range(x.ndim - 2):
        x = np.repeat(x, 2, axis=a + 2)
    return x


def adam_step(p, g, m, v, step, lr=1e-4, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam single-tensor update (scripts/torch/train.py:161,220), float64."""
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    denom = np.sqrt(v) / np.sqrt(bc2) + eps
    p = p - (lr / bc1) * m / denom
    return p, m, v


# --------------------------------------------------------------------------------------
# Evaluation helpers of the "next" rows N2 / N3  (reference voxelmorph/py/utils.py:265-287, :473-516)
# --------------------------------------------------------------------------------------

def dice_overlap(a1, a2, labels=None, include_zero=False):
    """Per-label Dice overlap of two label maps (py/utils.py:265-287, used by scripts/tf/test.py:76-121).

    labels=None: every label present in either map, ascending; label 0 dropped unless include_zero.
    2|A∩B| / max(|A| + |B|, eps) with eps = np.finfo(float).eps, float64."""
    a1, a2 = np.asarray(a1), np.asarray(a2)
    if labels is None:
        labels = np.union1d(np.unique(a1), np.unique(a2))
    labels = np.asarray(labels)
    if not include_zero:
        labels = labels[labels != 0]
    out = np.zeros(len(labels), dtype=np.float64)
    for i, lab in enumerate(labels):
        m1, m2 = a1 == lab, a2 == lab
        out[i] = 2.0 * np.count_nonzero(m1 & m2) / max(float(np.count_nonzero(m1) + np.count_nonzero(m2)), np.finfo(float).eps)
    return out


def _central_diff(x, axis):
    """np.gradient along one axis with unit spacing: central differences inside, first-order one-sided at both ends."""
    x = np.moveaxis(np.asarray(x, dtype=np.float64), axis, 0)
    g = np.empty_like(x)
    if x.shape[0] == 1:
        raise ValueError("gradient needs at least 2 samples along every axis")
    g[1:-1] = (x[2:] - x[:-2]) / 2.0
    g[0] = x[1] - x[0]
    g[-1] = x[-1] - x[-2]
    return np.moveaxis(g, 0, axis)


def jacobian_determinant(disp):
    """det of the Jacobian of the map x -> x + disp(x) for a (*vol, nd) displacement field, nd in (2, 3)
    (py/utils.py:473-516; the identity grid comes from pystrum.pynd.ndutils.volsize2ndgrid == np.meshgrid(indexing='ij');
    spatial derivatives are np.gradient's).  Values <= 0 mark folds (scripts/torch/register.py:63-97 consumers)."""
    disp = np.asarray(disp, dtype=np.float64)
    vol = disp.shape[:-1]
    nd = len(vol)
    assert nd in (2, 3) and disp.shape[-1] == nd, "flow has to be 2D or 3D"
    grid = np.stack(np.meshgrid(*[np.arange(s) for s in vol], indexing="ij"), axis=-1)
    phi = disp + grid
    d = [_central_diff(phi, ax) for ax in range(nd)]       # d[a][..., c] = d phi_c / d x_a
    if nd == 2:
        return d[0][..., 0] * d[1][..., 1] - d[1][..., 0] * d[0][..., 1]
    dx, dy, dz = d
    return (dx[..., 0] * (dy[..., 1] * dz[..., 2] - dy[..., 2] * dz[..., 1])
            - dx[..., 1] * (dy[..., 0] * dz[..., 2] - dy[..., 2] * dz[..., 0])
            + dx[..., 2] * (dy[..., 0] * dz[..., 1] - dy[..., 1] * dz[..., 0]))
