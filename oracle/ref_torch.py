"""Functional torch restatement of the reference VxmDense train / register step.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): the checker for the end-to-end parity
tests, the autograd oracle for the backward kernels, and the timed CPU baseline
(`bench.py --impl reference`, `cpu_baseline`).  It is deliberately *not* structured like
the reference's nn.Module tree: it is a set of pure functions over a flat
`{state_dict key: tensor}` mapping, so it consumes the very same checkpoint the product
model (or the reference) produces.

The arithmetic the reference reaches through torch (F.grid_sample, F.interpolate,
nn.Conv3d, MaxPool, Upsample, Adam — third-party, torch 2.11.0 in this image, not
pinned by the reference's setup.py) is called here through the same torch entry points;
the explicit formulas are restated separately in oracle/spec_np.py and the two are
cross-checked in tests/.

Pinned against the unmodified reference by tests/golden (oracle/make_golden.py and
oracle/make_golden_outputs.py, checked in tests/test_oracle_vs_reference.py).
"""
import math

import torch
import torch.nn.functional as F


# ---- layers (reference voxelmorph/torch/layers.py) ------------------------------------

def identity_grid(shape, device=None, dtype=torch.float32):
    """(1, nd, *shape) voxel-index grid, ij indexing (layers.py:17-22)."""
    axes = [torch.arange(0, s, device=device, dtype=dtype) for s in shape]
    return torch.stack(torch.meshgrid(*axes, indexing="ij")).unsqueeze(0)


def spatial_transform(src, flow, mode="bilinear"):
    """layers.py:30-48: sample src at (p + flow[p]); zeros padding; align_corners=True."""
    shape = flow.shape[2:]
    nd = len(shape)
    loc = identity_grid(shape, flow.device, flow.dtype) + flow
    comps = []
    for i in range(nd):
        comps.append(2 * (loc[:, i] / (shape[i] - 1) - 0.5))
    # grid_sample wants channels-last with x (last spatial axis) first
    grid = torch.stack(comps[::-1], dim=-1)
    return F.grid_sample(src, grid, align_corners=True, mode=mode)


def vec_int(vec, nsteps):
    """layers.py:61-68."""
    vec = vec * (1.0 / (2 ** nsteps))
    for _ in range(nsteps):
        vec = vec + spatial_transform(vec, vec)
    return vec


def resize_transform(x, vel_resize):
    """layers.py:76-97."""
    factor = 1.0 / vel_resize
    mode = {1: "linear", 2: "bilinear", 3: "trilinear"}[x.dim() - 2]
    if factor < 1:
        x = F.interpolate(x, align_corners=True, scale_factor=factor, mode=mode)
        x = factor * x
    elif factor > 1:
        x = factor * x
        x = F.interpolate(x, align_corners=True, scale_factor=factor, mode=mode)
    return x


# ---- network (reference voxelmorph/torch/networks.py) ---------------------------------

DEFAULT_FEATURES = ((16, 32, 32, 32), (32, 32, 32, 32, 32, 16, 16))  # py/utils.py:16-21


class _RoundBf16(torch.autograd.Function):
    """bf16 storage emulation with a straight-through gradient (used to mirror the tensor-core engine, which keeps
    activations and weight operands in bf16 and accumulates in fp32)."""

    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


_EMULATE_BF16 = [False]


def emulate_bf16(flag):
    """Test switch: round conv operands / activations to bf16 exactly where the tensor-core engine stores bf16."""
    _EMULATE_BF16[0] = bool(flag)


def _conv(x, sd, prefix, leaky):
    nd = x.dim() - 2
    fn = (F.conv1d, F.conv2d, F.conv3d)[nd - 1]
    w = sd[prefix + ".weight"]
    if _EMULATE_BF16[0]:
        x, w = _RoundBf16.apply(x), _RoundBf16.apply(w)
    y = fn(x, w, sd[prefix + ".bias"], stride=1, padding=1)
    y = F.leaky_relu(y, 0.2) if leaky else y
    if _EMULATE_BF16[0] and leaky:
        y = _RoundBf16.apply(y)          # activations are stored in bf16; the flow head output stays fp32
    return y


def unet_plan(cfg):
    """Resolve the Unet feature plan exactly as networks.py:56-85 does (default / list / int forms)."""
    import numpy as np
    nb_features = cfg.get("nb_unet_features")
    nb_levels = cfg.get("nb_unet_levels")
    feat_mult = cfg.get("unet_feat_mult", 1)
    ncpl = cfg.get("nb_unet_conv_per_level", 1)
    if nb_features is None:
        nb_features = DEFAULT_FEATURES
    if isinstance(nb_features, int):
        feats = np.round(nb_features * feat_mult ** np.arange(nb_levels)).astype(int)
        nb_features = [np.repeat(feats[:-1], ncpl), np.repeat(np.flip(feats), ncpl)]
    enc_nf, dec_nf = nb_features
    n_dec = len(enc_nf)
    return dict(enc=list(enc_nf), dec=list(dec_nf[:n_dec]), final=list(dec_nf[n_dec:]),
                levels=int(n_dec / ncpl) + 1, ncpl=ncpl)


def unet_forward(x, sd, cfg, prefix="unet_model"):
    """networks.py:122-144."""
    plan = unet_plan(cfg)
    nd = x.dim() - 2
    pool = (F.max_pool1d, F.max_pool2d, F.max_pool3d)[nd - 1]
    half_res = cfg.get("unet_half_res", False)
    L, ncpl = plan["levels"], plan["ncpl"]
    skips = [x]
    for level in range(L - 1):
        for c in range(ncpl):
            x = _conv(x, sd, "%s.encoder.%d.%d.main" % (prefix, level, c), True)
        skips.append(x)
        x = pool(x, 2)
    for level in range(L - 1):
        for c in range(ncpl):
            x = _conv(x, sd, "%s.decoder.%d.%d.main" % (prefix, level, c), True)
        if not half_res or level < L - 2:
            x = F.interpolate(x, scale_factor=2, mode="nearest")
            x = torch.cat([x, skips.pop()], dim=1)
    for i in range(len(plan["final"])):
        x = _conv(x, sd, "%s.remaining.%d.main" % (prefix, i), True)
    return x


def vxm_forward(sd, cfg, source, target, registration=False, unet_autocast=None):
    """networks.py:244-287.  `cfg` is the checkpoint's config dict (modelio.py:17-34).
    `unet_autocast` (bench.py's GPU eager baseline only): run the U-Net + flow head under torch.autocast with that dtype
    (what a user gets from wrapping the reference model's U-Net in autocast); everything after the flow head stays fp32."""
    int_steps = cfg.get("int_steps", 7)
    int_downsize = cfg.get("int_downsize", 2)
    bidir = cfg.get("bidir", False)
    half_res = cfg.get("unet_half_res", False)
    if unet_autocast is not None:
        with torch.autocast(source.device.type, dtype=unet_autocast):
            x = unet_forward(torch.cat([source, target], dim=1), sd, cfg)
            flow = _conv(x, sd, "flow", False)
        flow = flow.float()
    else:
        x = unet_forward(torch.cat([source, target], dim=1), sd, cfg)
        flow = _conv(x, sd, "flow", False)
    pos = flow
    if (not half_res) and int_steps > 0 and int_downsize > 1:
        pos = resize_transform(pos, int_downsize)
    preint = pos
    neg = -pos if bidir else None
    if int_steps > 0:
        pos = vec_int(pos, int_steps)
        neg = vec_int(neg, int_steps) if bidir else None
        if int_downsize > 1:
            pos = resize_transform(pos, 1 / int_downsize)
            neg = resize_transform(neg, 1 / int_downsize) if bidir else None
    y_source = spatial_transform(source, pos)
    y_target = spatial_transform(target, neg) if bidir else None
    if registration:
        return y_source, pos
    return (y_source, y_target, preint) if bidir else (y_source, preint)


def init_state_dict(cfg, seed=0, flow_std=1e-5, dtype=torch.float32):
    """Random parameters with the reference's key names / shapes / init families
    (ConvNd default kaiming-uniform(a=sqrt 5); flow ~ N(0, flow_std), zero bias: networks.py:210-215).
    Values are NOT bit-identical to a reference-constructed model; parity tests copy one
    state_dict into both sides."""
    g = torch.Generator().manual_seed(seed)
    nd = len(cfg["inshape"])
    plan = unet_plan(cfg)
    half_res = cfg.get("unet_half_res", False)
    infeats = cfg.get("src_feats", 1) + cfg.get("trg_feats", 1)
    sd = {}

    def add_conv(prefix, cin, cout):
        fan_in = cin * 3 ** nd
        bound = 1.0 / math.sqrt(fan_in)
        sd[prefix + ".weight"] = ((torch.rand((cout, cin) + (3,) * nd, generator=g, dtype=dtype) * 2 - 1) * bound)
        sd[prefix + ".bias"] = ((torch.rand((cout,), generator=g, dtype=dtype) * 2 - 1) * bound)

    L, ncpl = plan["levels"], plan["ncpl"]
    prev = infeats
    enc_hist = [prev]
    for level in range(L - 1):
        for c in range(ncpl):
            nf = int(plan["enc"][level * ncpl + c])
            add_conv("unet_model.encoder.%d.%d.main" % (level, c), prev, nf)
            prev = nf
        enc_hist.append(prev)
    enc_hist = enc_hist[::-1]
    for level in range(L - 1):
        for c in range(ncpl):
            nf = int(plan["dec"][level * ncpl + c])
            add_conv("unet_model.decoder.%d.%d.main" % (level, c), prev, nf)
            prev = nf
        if not half_res or level < L - 2:
            prev += enc_hist[level]
    for i, nf in enumerate(plan["final"]):
        add_conv("unet_model.remaining.%d.main" % i, prev, int(nf))
        prev = int(nf)
    sd["flow.weight"] = torch.randn((nd, prev) + (3,) * nd, generator=g, dtype=dtype) * flow_std
    sd["flow.bias"] = torch.zeros((nd,), dtype=dtype)
    return sd


# ---- losses (reference voxelmorph/torch/losses.py) ------------------------------------

def ncc_loss(y_true, y_pred, win=None):
    """losses.py:15-67 (device-agnostic: the ones filter lives on the inputs' device)."""
    nd = y_true.dim() - 2
    win = [9] * nd if win is None else list(win)
    filt = torch.ones([1, 1, *win], dtype=y_true.dtype, device=y_true.device)
    pad = math.floor(win[0] / 2)
    conv = (F.conv1d, F.conv2d, F.conv3d)[nd - 1]

    def S(t):
        return conv(t, filt, stride=1, padding=pad)

    I, J = y_true, y_pred
    I_sum, J_sum, I2_sum, J2_sum, IJ_sum = S(I), S(J), S(I * I), S(J * J), S(I * J)
    n = float(math.prod(win))
    u_I, u_J = I_sum / n, J_sum / n
    cross = IJ_sum - u_J * I_sum - u_I * J_sum + u_I * u_J * n
    I_var = I2_sum - 2 * u_I * I_sum + u_I * u_I * n
    J_var = J2_sum - 2 * u_J * J_sum + u_J * u_J * n
    cc = cross * cross / (I_var * J_var + 1e-5)
    return -cc.mean()


def mse_loss(y_true, y_pred):
    return ((y_true - y_pred) ** 2).mean()


def dice_loss(y_true, y_pred):
    ax = list(range(2, y_pred.dim()))
    top = 2 * (y_true * y_pred).sum(dim=ax)
    bottom = torch.clamp((y_true + y_pred).sum(dim=ax), min=1e-5)
    return -(top / bottom).mean()


def grad_loss(y_pred, penalty="l2", loss_mult=None):
    nd = y_pred.dim() - 2
    terms = []
    for a in range(nd):
        ax = a + 2
        n = y_pred.shape[ax]
        d = y_pred.narrow(ax, 1, n - 1) - y_pred.narrow(ax, 0, n - 1)
        d = d.abs() if penalty == "l1" else d * d
        terms.append(d.flatten(1).mean(dim=-1))
    g = sum(terms) / nd
    if loss_mult is not None:
        g = g * loss_mult
    return g.mean()


# ---- one full training step (scripts/torch/train.py:199-220) ---------------------------

def train_step(sd, cfg, opt, source, target, image_loss="ncc", lam=0.01, unet_autocast=None, sync=True):
    """fwd + loss + bwd + Adam (tensors on any device).  `sd` values must be leaf tensors with
    requires_grad=True and `opt` a torch.optim.Adam over them.  Returns the loss value (a tensor when sync=False)."""
    int_downsize = cfg.get("int_downsize", 2)
    y_source, preint = vxm_forward(sd, cfg, source, target, unet_autocast=unet_autocast)
    il = ncc_loss(target, y_source) if image_loss == "ncc" else mse_loss(target, y_source)
    loss = il + lam * grad_loss(preint, "l2", loss_mult=int_downsize)
    opt.zero_grad()
    loss.backward()
    opt.step()
    return float(loss.detach()) if sync else loss.detach()
