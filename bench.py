#!/usr/bin/env python
"""bench.py — BASELINE.json metric: 3-D vol-pairs/sec (160x192x224) for one diffeomorphic VxmDense TRAINING step
(forward + NCC/Grad losses + backward + gradient allreduce + Adam) at N GPUs, one volume pair per GPU per step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is obtained.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FULL = (160, 192, 224)
# first-step loss vs the fp32 CPU oracle, per convolution engine (measured on B200 at 160x192x224: bf16 1.8e-7, bf16x3 2.7e-7;
# the moved image is within 1e-4 in every mode, the flow field is what bf16 operands cost: 6e-3 vs 1.4e-5 for bf16x3)
PARITY_TOL = {"bf16": 1e-5, "bf16x3": 1e-5, "f32": 1e-5}
METRIC = "vol-pairs/sec (3D 160x192x224 VxmDense int_steps=7 train step, NCC+Grad, Adam)"
UNIT = "vol-pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--shape", type=int, nargs=3, default=list(FULL), help="debug only; the metric is quoted at 160 192 224")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--engine", default=None, choices=["f32", "bf16"], help="convolution engine (default: bf16 tensor-core engine)")
    ap.add_argument("--no-graph", action="store_true", help="time eager kernel launches instead of the captured CUDA graph")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel roofline legs")
    ap.add_argument("--config", type=int, default=2, choices=[2, 5], help="BASELINE.json config: 2 = the headline (default; config 3 is "
                    "the same under torchrun), 5 = semi-supervised: + Dice on the linearly warped 30-label one-hot segmentation")
    ap.add_argument("--no-parity", action="store_true", help="skip the first-step loss check against the CPU oracle and the bf16x3 parity-mode leg")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the reference-torch-on-GPU (eager ATen / cuDNN) baseline leg")
    ap.add_argument("--no-c4", action="store_true", help="skip the BASELINE config 4 sweep (256^3 warp / VecInt GB/s)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (its loss) and left behind "
                    "(the trained parameters) to DIR/<name>.npy, float32, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 training step (--impl b200)")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------
# conv FLOPs of the default U-Net per training step (SURVEY.md section 8(d))
# ------------------------------------------------------------------------------------------------
def conv_flops_per_step(shape):
    import numpy as np
    V = float(np.prod(shape))
    layers = [  # (cin, cout, voxel fraction, has_dgrad)
        (2, 16, 1, False), (16, 32, 1 / 8, True), (32, 32, 1 / 64, True), (32, 32, 1 / 512, True),
        (32, 32, 1 / 4096, True), (64, 32, 1 / 512, True), (64, 32, 1 / 64, True), (64, 32, 1 / 8, True),
        (48, 32, 1, True), (32, 16, 1, True), (16, 16, 1, True), (16, 3, 1, True)]
    fwd = sum(2 * 27 * ci * co * V * f for ci, co, f, _ in layers)
    bwd = sum(2 * 27 * ci * co * V * f * (2 if dg else 1) for ci, co, f, dg in layers)
    return fwd, fwd + bwd


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, during the timed region)
# ------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Summary of the samples taken in [t0, t1] (host clock).  The sampler is started before the warm-up so that it is
        already streaming; when the timed region is shorter than the sampling period the nearest sample taken under the
        same load (warm-up steps run back to back with the timed ones) is used and `window` says so."""
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.06)   # let the sample that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        rows, window = list(self.rows), "timed region"
        if t0 is not None:
            inside = [r for r in rows if t0 <= r[0] <= t1 + 0.06]
            if inside:
                rows = inside
            elif rows:
                rows = [min(rows, key=lambda r: abs(r[0] - 0.5 * (t0 + t1)))]
                window = "nearest sample under load (timed region shorter than the 50 ms sampling period)"
        for _, r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), power_w_max=max(pw), samples=len(sm),
                    reasons=sorted(reasons), window=window)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's torch CPU path on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_step_time(shape, steps, warmup, budget_s, min_full=1):
    """Time the oracle restatement of the reference training step (oracle/ref_torch.py: same torch CPU operators
    the reference calls) on all host cores.  Returns (sec per FULL-SIZE pair, cores, sample description)."""
    import numpy as np
    import torch
    from oracle import cases, ref_torch
    cores = os.cpu_count() or 1

    def make(shp):
        cfg = dict(inshape=tuple(shp), nb_unet_features=None, nb_unet_levels=None, unet_feat_mult=1, nb_unet_conv_per_level=1,
                   int_steps=7, int_downsize=2, bidir=False, use_probs=False, src_feats=1, trg_feats=1, unet_half_res=False)
        sd = {k: v.requires_grad_(True) for k, v in ref_torch.init_state_dict(cfg, seed=1234, flow_std=1e-2).items()}
        opt = torch.optim.Adam(list(sd.values()), lr=1e-4)
        g = torch.Generator().manual_seed(1234)
        s = torch.rand((1, 1) + tuple(shp), generator=g)
        t = torch.rand((1, 1) + tuple(shp), generator=g)
        return cfg, sd, opt, s, t

    def run(shp, n):
        cfg, sd, opt, s, t = make(shp)
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            ref_torch.train_step(sd, cfg, opt, s, t, image_loss="ncc", lam=0.01)
            ts.append(time.perf_counter() - t0)
        return ts

    sub = tuple(max(16, (d // 2 // 16) * 16) for d in shape)
    frac = float(np.prod(sub)) / float(np.prod(shape))
    # give the CPU path its best thread count (oneDNN / ATen do not always scale to every core of a big host)
    best = None
    for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16)}, reverse=True):
        torch.set_num_threads(nt)
        tt = run(sub, 2)[-1]
        if best is None or tt < best[0]:
            best = (tt, nt)
    t_sub, cores_used = best
    torch.set_num_threads(cores_used)
    cores = cores_used
    est_full = t_sub / frac
    # Full-size steps first: as many of the requested steps as fit the time budget (at least `min_full` — one is already the
    # whole workload of the metric), after one untimed full-size warm-up when it fits too.  Only when not even that fits does
    # the sample fall back to a sub-volume with the time scaled by the voxel ratio (never on the boxes seen so far).
    n_fit = int(budget_s / max(est_full, 1e-3))
    if n_fit >= min_full:
        w = 1 if n_fit >= min_full + 1 else 0
        n = max(min_full, min(steps, n_fit - w))
        ts = run(shape, n + w)[w:]
        return sum(ts) / len(ts), cores, "%d full-size %s steps after %d warm-up (of %d requested), torch %s CPU fp32, %d threads" % (
            len(ts), "x".join(map(str, shape)), w, steps, torch.__version__, cores), True
    n = max(1, min(steps, int(budget_s / max(t_sub, 1e-3)) - 1))
    ts = run(sub, n + 1)[1:]
    per_full = (sum(ts) / len(ts)) / frac
    return per_full, cores, ("%d steps on a %s sub-volume (%.3f of the voxels; time scaled by 1/%.3f), torch %s CPU fp32, "
                             "%d threads" % (len(ts), "x".join(map(str, sub)), frac, frac, torch.__version__, cores)), False


def reference_arm(args):
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sec, cores, sample, full = cpu_step_time(tuple(args.shape), args.steps, args.warmup, budget_s=150.0, min_full=3)
    v = 1.0 / sec
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload="3D %s VxmDense diffeomorphic (int_steps=7, int_downsize=2), NCC+0.01*Grad, Adam, batch 1"
                            % "x".join(map(str, args.shape)), note="reference torch CPU path (oracle port) on host cores",
                            same_config=bool(full), sample_steps_are_full_size=bool(full)),
                cpu_baseline=dict(value=v, unit=UNIT, cores=cores, kind="port", sample=sample),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)



# ------------------------------------------------------------------------------------------------
# helper legs of the B200 arm
# ------------------------------------------------------------------------------------------------
CONV_SOURCES = ("conv3d_tc_s.cu", "conv3d_tc_s2.cu", "conv3d_tc_wgrad2.cu", "tc_common.cuh")


def _strip_comments(text):
    """C / CUDA source without comments and blank lines (string literals respected): the hash below identifies the CODE the
    committed ncu pass measured — rewording a comment must not invalidate it, changing a statement must."""
    out, i, n, in_str = [], 0, len(text), False
    while i < n:
        c = text[i]
        if in_str:
            out.append(c)
            if c == "\\" and i + 1 < n:
                out.append(text[i + 1]); i += 1
            elif c == '"':
                in_str = False
        elif c == '"':
            in_str = True; out.append(c)
        elif text.startswith("//", i):
            while i < n and text[i] != "\n":
                i += 1
            continue
        elif text.startswith("/*", i):
            j = text.find("*/", i + 2)
            i = n if j < 0 else j + 2
            continue
        else:
            out.append(c)
        i += 1
    return "\n".join(l.strip() for l in "".join(out).splitlines() if l.strip())


def conv_source_hash():
    import hashlib
    h = hashlib.sha256()
    for f in CONV_SOURCES:
        with open(os.path.join(ROOT, "voxelmorph_b200", "csrc", f), "r") as fh:
            h.update(_strip_comments(fh.read()).encode())
    return h.hexdigest()[:16]


def default_cfg(shape):
    return dict(inshape=tuple(shape), nb_unet_features=None, nb_unet_levels=None, unet_feat_mult=1, nb_unet_conv_per_level=1,
                int_steps=7, int_downsize=2, bidir=False, use_probs=False, src_feats=1, trg_feats=1, unet_half_res=False)


def oracle_first_step_loss(model, shape, S_host, T_host):
    """Loss of the reference's step (fp32, CPU: oracle/ref_torch) on the benchmark's own initial weights and first pair."""
    import torch
    from oracle import ref_torch
    sd = {k: v.detach().float().cpu().clone() for k, v in model.state_dict().items()}
    cfg = default_cfg(shape)
    torch.set_num_threads(max(1, min(64, os.cpu_count() or 1)))
    with torch.no_grad():
        y, pre = ref_torch.vxm_forward(sd, cfg, S_host, T_host)
        return float(ref_torch.ncc_loss(T_host, y) + 0.01 * ref_torch.grad_loss(pre, "l2", 2))


def gpu_eager_baseline(dev, shape, pairs_dev, steps=5, warmup=2):
    """The reference's own torch path on this GPU (SURVEY 2 / BASELINE.md 4 step 5): oracle/ref_torch.train_step — the
    same ATen / cuDNN operators voxelmorph/torch calls (nn.Conv3d, F.grid_sample, 5 x F.conv3d NCC) — eager, fp32 tensors
    with cuDNN's default TF32 convolutions, and again with bf16 autocast around the U-Net."""
    import torch
    from oracle import ref_torch
    out = {}
    cfg = default_cfg(shape)
    for name, ac in (("tf32_default", None), ("bf16_autocast_unet", torch.bfloat16)):
        try:
            sd = {k: v.to(dev).requires_grad_(True) for k, v in ref_torch.init_state_dict(cfg, seed=1234, flow_std=1e-2).items()}
            opt = torch.optim.Adam(list(sd.values()), lr=1e-4)
            for i in range(warmup):
                ref_torch.train_step(sd, cfg, opt, *pairs_dev[i % len(pairs_dev)], image_loss="ncc", lam=0.01, unet_autocast=ac, sync=False)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                ref_torch.train_step(sd, cfg, opt, *pairs_dev[i % len(pairs_dev)], image_loss="ncc", lam=0.01, unet_autocast=ac, sync=False)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = dict(value=1e3 / ms, unit=UNIT, ms_per_step=ms, steps=steps, warmup=warmup,
                             peak_mem_gb=torch.cuda.max_memory_allocated(dev) / 1e9)
            del sd, opt
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001 - a baseline leg must not kill the bench
            out[name] = dict(error=str(e)[:200])
    out["what"] = ("reference torch path (oracle/ref_torch restatement of voxelmorph/torch) on the same GPU: eager ATen/cuDNN, "
                   "torch %s, cudnn.allow_tf32=%s, device-resident pairs, CUDA events" % (torch.__version__, torch.backends.cudnn.allow_tf32))
    return out


def engine_leg(vxm, dev, shape, pairs_dev, engine, steps=10, warmup=3):
    """One more timed training-step loop on a FRESH model with another convolution engine (graph-captured like the headline)."""
    import torch
    from voxelmorph_b200.trainer import GraphedTrainStep
    prev = os.environ.get("VXM_B200_CONV_ENGINE")
    os.environ["VXM_B200_CONV_ENGINE"] = engine
    try:
        torch.manual_seed(1234)
        model = vxm.networks.VxmDense(inshape=shape, int_steps=7, int_downsize=2)
        with torch.no_grad():
            model.flow.weight.normal_(0, 1e-2)
        model.to(dev).train()
        opt = vxm.optim.FusedAdam(model.parameters(), lr=1e-4)
        step = GraphedTrainStep(model, opt, image_loss="ncc", lam=0.01, int_downsize=2).capture(*pairs_dev[0])
        for i in range(warmup):
            step(*pairs_dev[i % len(pairs_dev)])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(*pairs_dev[i % len(pairs_dev)])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return dict(engine=engine, value=1e3 / ms, unit=UNIT, ms_per_step=ms, steps=steps, warmup=warmup, cuda_graph=True)
    finally:
        if prev is None:
            os.environ.pop("VXM_B200_CONV_ENGINE", None)
        else:
            os.environ["VXM_B200_CONV_ENGINE"] = prev


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def b200_arm(args):
    import numpy as np
    import torch
    import voxelmorph_b200 as vxm
    from voxelmorph_b200 import dist as vdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)")
    os.environ["VXM_B200_TRANSPARENT_DP"] = "0"     # bench drives its one allreduce per step itself (inside the CUDA graph)
    world, rank, local = vdist.init_from_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py: --gpus %d needs torchrun (one process per GPU)" % args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    vxm._lib.load()
    os.environ["VXM_B200_CONV_ENGINE"] = args.engine or os.environ.get("VXM_B200_CONV_ENGINE", "bf16")
    peaks = load_peaks()
    shape = tuple(args.shape)
    V = int(np.prod(shape))

    # ---- model, optimizer, data ----------------------------------------------------------------
    torch.manual_seed(1234)
    semi = args.config == 5
    NLAB = 30
    if semi:
        model = vxm.networks.VxmDenseSemiSupervisedSeg(shape, NLAB, int_steps=7, int_downsize=2)
        flow_head = model.vxm_model.flow
    else:
        model = vxm.networks.VxmDense(inshape=shape, int_steps=7, int_downsize=2)
        flow_head = model.flow
    with torch.no_grad():
        flow_head.weight.normal_(0, 1e-2)   # trained-like flow scale so that warps / VecInt do real work
    model.to(dev).train()
    opt = vxm.optim.FusedAdam(model.parameters(), lr=1e-4, world_size=world)
    vdist.broadcast_params(opt.fp.flat)
    ncc = vxm.losses.NCC().loss
    grad = vxm.losses.Grad("l2", loss_mult=2).loss

    # synthetic pairs (generated on the device by torch, seeds differ per rank): smooth volume + warped copy
    NPAIR = 4
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    pairs_host = []
    st = vxm.layers.SpatialTransformer(shape)
    for i in range(NPAIR):
        coarse = torch.rand((1, 1, shape[0] // 8, shape[1] // 8, shape[2] // 8), generator=g, device=dev)
        src = torch.nn.functional.interpolate(coarse, size=shape, mode="trilinear", align_corners=True)
        src = (src + 0.05 * torch.rand(src.shape, generator=g, device=dev)).clamp_(0, 1).contiguous()
        fl = torch.nn.functional.interpolate(torch.randn((1, 3, shape[0] // 16, shape[1] // 16, shape[2] // 16), generator=g,
                                                         device=dev) * 3.0, size=shape, mode="trilinear", align_corners=True)
        trg = st(src, fl.contiguous())
        sample = [src, trg]
        if semi:
            # synthetic anatomy: NLAB smooth blobs -> label map at half resolution -> one-hot (1, 30, 80, 96, 112) for both images
            # (generators.semisupervised: [::2] sub-sampled one-hot of the label map); the target's labels are the source's
            # moved by the same flow (nearest), so the Dice term has something to align
            half = tuple(d // 2 for d in shape)
            blobs = torch.nn.functional.interpolate(torch.randn((1, NLAB, shape[0] // 16, shape[1] // 16, shape[2] // 16), generator=g, device=dev),
                                                    size=shape, mode="trilinear", align_corners=True)
            lab_s = blobs.argmax(1, keepdim=True).float()
            lab_t = vxm.layers.SpatialTransformer(shape, mode="nearest")(lab_s, fl.contiguous())
            oh = lambda lab: (lab[:, :, ::2, ::2, ::2] == torch.arange(NLAB, device=dev).view(1, NLAB, 1, 1, 1)).float().contiguous()  # noqa: E731
            sample += [oh(lab_s), oh(lab_t)]
            del blobs, lab_s, lab_t
        pairs_host.append(tuple(x.cpu().pin_memory() for x in sample))
    pairs_dev = [tuple(x.to(dev) for x in smp) for smp in pairs_host]
    dice = vxm.losses.Dice().loss

    def forward_loss(*inp):
        if semi:
            y, pre, yseg = model(inp[0], inp[1], inp[2])
            return ncc(inp[1], y) + 0.01 * grad(None, pre) + 0.01 * dice(inp[3], yseg)
        y, flow = model(inp[0], inp[1])
        return ncc(inp[1], y) + 0.01 * grad(None, flow)
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    # ---- parity of the timed configuration at its own size: first-step loss vs the CPU oracle -------------------------
    parity = None
    if rank == 0 and not args.no_parity and not semi:
        with torch.no_grad():
            y0, f0 = model(*pairs_dev[0])
            loss_gpu = float(ncc(pairs_dev[0][1], y0) + 0.01 * grad(None, f0))
        del y0, f0
        loss_ref = oracle_first_step_loss(model, shape, pairs_host[0][0], pairs_host[0][1])
        tol = PARITY_TOL.get(os.environ["VXM_B200_CONV_ENGINE"], 1e-4)
        err = abs(loss_gpu - loss_ref) / abs(loss_ref)
        parity = dict(loss_gpu=loss_gpu, loss_oracle=loss_ref, rel_err=err, tol=tol, ok=bool(err <= tol),
                      what="NCC + 0.01 Grad of the first pair on the initial weights: timed engine vs oracle/ref_torch (fp32 CPU "
                           "restatement of the reference); the full forward / gradient comparison at this size is "
                           "tests/test_gpu_bf16_engine.py::test_full_size_step_vs_oracle")
        if not parity["ok"]:
            raise SystemExit("bench.py: first-step loss %.6f deviates from the oracle's %.6f by %.2e (> %.1e): the timed path is "
                             "not computing the reference's step" % (loss_gpu, loss_ref, err, tol))

    def eager_step(*inp):
        opt.zero_grad()
        loss = forward_loss(*inp)
        loss.backward()
        vdist.allreduce_grads(opt.fp.grad)
        opt.step()
        return loss

    # the whole step (zero-grad, fwd, losses, bwd, allreduce, Adam) captured once in a CUDA graph and replayed
    step, graphed = eager_step, False
    launches_per_step = None
    trainer_ref = []
    if not args.no_graph:
        from voxelmorph_b200.trainer import GraphedTrainStep
        try:
            n0 = vxm._lib.launch_count()
            eager_step(*pairs_dev[0])
            launches_per_step = vxm._lib.launch_count() - n0
            trainer = GraphedTrainStep(model, opt, loss_fn=lambda m, *inp: forward_loss(*inp)).capture(*pairs_dev[0])
            step, graphed = trainer, True
            trainer_ref.append(trainer)
        except Exception as e:  # noqa: BLE001 - report and fall back to eager launches
            print("bench.py: CUDA graph capture failed (%s); timing eager launches" % e, file=sys.stderr)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ---------------------------------------------------------------------------------
    W, K = max(3, args.warmup), args.steps
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    for i in range(W):
        step(*pairs_dev[i % NPAIR])
    barrier()

    # ---- device-resident timed region ------------------------------------------------------------
    n0 = vxm._lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_host0 = time.time()
    e0.record()
    for i in range(K):
        loss_last = step(*pairs_dev[i % NPAIR])
    e1.record()
    barrier()
    t_host1 = time.time()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss_last, model)
    ms = e0.elapsed_time(e1)
    launches = (launches_per_step * K) if graphed else (vxm._lib.launch_count() - n0)
    ms = vdist.max_over_ranks(ms, dev)
    clk = clocks.stop(t_host0, t_host1) if rank == 0 else None
    value = world * K / (ms * 1e-3)

    # ---- end-to-end: host buffers, H2D of the pair + D2H of the loss inside the timed region --------
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [tuple(torch.empty_like(x) for x in pairs_dev[0]) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[b])
            for dst, srcbuf in zip(bufs[b], pairs_host[i % NPAIR]):
                dst.copy_(srcbuf, non_blocking=True)
            ready[b].record(copy_stream)

    for b in range(2):
        freed[b].record()
    barrier()
    e0.record()
    prefetch(0)
    for i in range(K):
        if i + 1 < K:
            prefetch(i + 1)
        b = i % 2
        torch.cuda.current_stream().wait_event(ready[b])
        loss = step(*bufs[b])
        freed[b].record()
        loss_host.copy_(loss.detach(), non_blocking=True)
    e1.record()
    barrier()
    ms_e2e = vdist.max_over_ranks(e0.elapsed_time(e1), dev)
    e2e = dict(value=world * K / (ms_e2e * 1e-3), unit=UNIT, h2d_bytes_per_step=int(sum(x.numel() * 4 for x in pairs_host[0])), d2h_bytes_per_step=4,
               ms_per_step=ms_e2e / K, api="voxelmorph_b200.networks.VxmDense + losses.NCC/Grad + optim.FusedAdam, pinned host "
               "buffers, H2D double-buffered on a copy stream")

    # ---- roofline of the dominant kernel family (Conv3d) measured live with CUDA events -------------
    # One eager step records every convolution launch (function + arguments); the recorded launches are then
    # re-issued back to back between two CUDA events on the launching stream, behind a device-side sleep so that the
    # host runs ahead and the events bracket kernel time only (no launch gaps).
    from voxelmorph_b200 import ops
    from voxelmorph_b200 import tc as tcmod
    calls = []

    def recording(fn):
        def inner(*a, **k):
            calls.append((fn, a, k))
            return fn(*a, **k)
        return inner

    o_cf, o_cw, o_ct = tcmod.conv_fwd, tcmod.conv_wgrad, tcmod.conv_fwd_t
    orig_fwd, orig_bwd = ops._ConvK3Fn.forward, ops._ConvK3Fn.backward
    conv_total_ms = None
    if ops.conv_engine() == "bf16":
        tcmod.conv_fwd, tcmod.conv_wgrad, tcmod.conv_fwd_t = recording(o_cf), recording(o_cw), recording(o_ct)
        eager_step(*pairs_dev[0])
        tcmod.conv_fwd, tcmod.conv_wgrad, tcmod.conv_fwd_t = o_cf, o_cw, o_ct
        torch.cuda.synchronize()
        reps = []
        for _ in range(3):
            torch.cuda._sleep(12000000)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for fn, a, k in calls:
                fn(*a, **k)
            c1.record()
            torch.cuda.synchronize()
            reps.append(c0.elapsed_time(c1))
        conv_total_ms = statistics.median(reps)
        n_conv_launches = len(calls)
        if os.environ.get("VXM_BENCH_VERBOSE") and rank == 0:
            for fn, a, k in calls:      # per-launch breakdown (stderr)
                torch.cuda._sleep(2000000)
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(); fn(*a, **k); c1.record(); torch.cuda.synchronize()
                shp = [tuple(x.shape) for x in a[:3] if hasattr(x, "shape")]
                print("  %-12s %8.1f us  %s" % (fn.__name__, c0.elapsed_time(c1) * 1e3, shp), file=sys.stderr)
        del calls
    else:
        conv_ms = []

        def timed(fn):
            def inner(*a, **k):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                r = fn(*a, **k)
                a1.record()
                conv_ms.append((a0, a1))
                return r
            return inner

        ops._ConvK3Fn.forward = staticmethod(timed(orig_fwd))
        ops._ConvK3Fn.backward = staticmethod(timed(orig_bwd))
        eager_step(*pairs_dev[0])
        torch.cuda.synchronize()
        ops._ConvK3Fn.forward, ops._ConvK3Fn.backward = staticmethod(orig_fwd), staticmethod(orig_bwd)
        conv_total_ms = sum(x.elapsed_time(y) for x, y in conv_ms)
        n_conv_launches = len(conv_ms)
    if rank != 0:
        _leave(world, rank)
        return
    _, flops_step = conv_flops_per_step(shape)
    ach = flops_step / (conv_total_ms * 1e-3) / 1e12
    engine = ops.conv_engine()
    # DRAM traffic of the conv family per step: taken from the committed ncu pass over this same command
    # (profiles/r1_traffic.json; ncu cannot run inside a timed bench), valid for the full-size bf16 workload only.
    traffic, traffic_src = None, None
    tj = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if engine == "bf16" and tuple(shape) == (160, 192, 224) and os.path.exists(tj):
        with open(tj) as f:
            tinfo = json.load(f)
        if tinfo.get("conv_source_sha") == conv_source_hash():
            traffic, traffic_src = tinfo["conv_dram_mbytes_per_step"] * 1e6, tinfo["source"]
        else:
            traffic_src = ("stale: profiles/r2_traffic.json was captured for conv sources %s, the library was built from %s"
                           % (tinfo.get("conv_source_sha"), conv_source_hash()))
    roofline = dict(bound="tensor", kernel="conv3d k3 fwd+dgrad+wgrad, all 12 layers (%s)" % ("tcgen05 bf16 implicit GEMM" if engine == "bf16" else "fp32 FFMA engine"),
                    achieved=ach, peak=peaks["tf_burst"], unit="TFLOP/s", frac=ach / peaks["tf_burst"], traffic=traffic, traffic_unit="bytes per step (all conv launches)", traffic_source=traffic_src,
                    peak_source=peaks["source"] + ", burst bf16 (the conv launches are replayed in isolation behind a sleep, not inside the long step)",
                    frac_of_sustained=ach / peaks["tf_sus"], ms_per_step=conv_total_ms, conv_launches=n_conv_launches,
                    share_of_step=conv_total_ms / (ms / K), flops_per_step=flops_step)

    kernels = {} if (args.no_kernels or semi) else kernel_rooflines(vxm, dev, shape, peaks)
    parity_mode = None
    if not args.no_parity and engine == "bf16" and world == 1 and not semi:
        try:
            parity_mode = engine_leg(vxm, dev, shape, pairs_dev, "bf16x3")
            parity_mode["note"] = ("same step with the split-precision tensor-core forward (3 tcgen05 passes per layer, flow / moved image "
                                   "within 1e-4 of the fp32 reference: tests/test_gpu_bf16_engine.py); backward on bf16 operands")
        except Exception as e:  # noqa: BLE001
            parity_mode = dict(error=str(e)[:300])
    c4 = None
    if not args.no_c4 and world == 1 and not semi:
        try:
            c4 = c4_sweep(vxm, dev, peaks)
        except Exception as e:  # noqa: BLE001
            c4 = dict(error=str(e)[:300])
    gpu_eager = None
    if not args.no_gpu_eager and world == 1 and not semi:
        del trainer_ref[:]
        torch.cuda.empty_cache()
        gpu_eager = gpu_eager_baseline(dev, shape, pairs_dev)

    # ---- CPU baseline (oracle port of the reference's torch CPU path) -------------------------------
    cpu = None
    if not args.no_cpu_baseline:
        sec, cores, sample, _ = cpu_step_time(shape, 1, 0, budget_s=30.0)
        cpu = dict(value=1.0 / sec, unit=UNIT, cores=cores, kind="port", sample=sample)

    act_gb = 4.0 * V * (2 + 16 + 48 + 32 + 16 + 16 + 3) / 1e9
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms / K,
                higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32" if engine == "f32" else "bf16 (conv operands) / f32 (accumulate, warp, VecInt, losses)",
                data="synthetic", impl="b200",
                config=dict(workload=("3D %s VxmDense diffeomorphic (int_steps=7, int_downsize=2), default U-Net features, "
                                      "NCC(9^3)+0.01*Grad(l2), Adam lr 1e-4, 1 pair per GPU" % "x".join(map(str, shape)))
                            + (" + semi-supervised branch (BASELINE config 5): 30-label one-hot segmentations at half resolution warped "
                               "linearly, + 0.01*Dice" if semi else ""), baseline_config=args.config,
                            global_batch=world, parallelism="dp%d (one flat-gradient allreduce per step)" % world,
                            conv_engine=engine, cuda_graph=graphed,
                            l2="inputs rotate over %d resident pairs; per-step working set ~%.1f GB of full-resolution "
                               "activations >> 126 MB L2, so no explicit flush" % (NPAIR, act_gb)),
                clocks=clk, e2e=e2e, gpu_launches=int(launches), launches_per_step=launches / K,
                roofline=roofline, kernels=kernels, cpu_baseline=cpu, parity_check=parity, parity_mode=parity_mode,
                gpu_eager_baseline=gpu_eager, c4_sweep=c4)
    print(json.dumps(line), flush=True)
    _leave(world, rank)


def dump_outputs(out_dir, loss, model):
    """The arrays a caller of the training step has after its last timed step: the loss it returned and the model's
    parameters after the Adam update, one float32 .npy each (about 1.3 MB for the default U-Net, whatever the shape).
    The inputs, the initial weights and the number of steps depend only on the arguments, so two builds run with the same
    arguments can be compared file by file.  Gradient sums accumulated with atomics make even two runs of one build differ
    in the last bits, and Adam magnifies that where a gradient is near zero: compare the weights with a tolerance."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = dict(loss=loss.detach().float().reshape(1))
    arrays.update(("param." + k, p.detach().float()) for k, p in model.named_parameters())
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def _leave(world, rank=None):
    """End of a rank's work.  Under torchrun every rank leaves with os._exit(0), rank 0 last: the captured CUDA graph
    still holds NCCL kernels, and tearing the process group down with it alive (destroy_process_group / interpreter
    shutdown) blocked both ranks after the JSON line had been printed (2 x B200, round 1).  The ranks meet on the
    rendezvous store (no collective): rank 0 posts `bench_done`, the others acknowledge, then everybody exits."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world <= 1:
        return
    import datetime
    import torch
    import torch.distributed as dist
    try:
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        store = dist.distributed_c10d._get_default_store()
        store.set_timeout(datetime.timedelta(seconds=1800))
        if rank is None:
            rank = dist.get_rank()
        if rank == 0:
            store.set("bench_done", "1")
            t0 = time.time()
            while store.add("bench_ack", 0) < world - 1 and time.time() - t0 < 60.0:
                time.sleep(0.05)
        else:
            store.wait(["bench_done"])      # rank 0 may still be timing its CPU baseline
            store.add("bench_ack", 1)
            time.sleep(0.2)
    except Exception as e:  # noqa: BLE001 - leaving must not fail
        print("bench.py: exit rendezvous skipped (%s)" % e, file=sys.stderr)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def kernel_rooflines(vxm, dev, shape, peaks):
    """Each memory-bound kernel timed alone (CUDA events, 3 warm-up + 10 timed launches, 256 MB L2 flush between
    launches); algorithmic bytes per SURVEY.md section 8(d)."""
    import numpy as np
    import torch
    V = int(np.prod(shape))
    half = tuple(s // 2 for s in shape)
    Vh = int(np.prod(half))
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    out = {}

    def timeit(fn, nbytes, name, note=""):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(10):
            flush.zero_()
            torch.cuda._sleep(400000)   # keep the GPU busy while the host enqueues, so the events bracket the kernel only
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        t = statistics.median(ts)
        gbs = nbytes / (t * 1e-3) / 1e9
        out[name] = dict(bound="hbm", achieved=gbs, peak=peaks["hbm"], unit="GB/s", frac=gbs / peaks["hbm"], us=t * 1e3,
                         algorithmic_bytes=nbytes, note=note)

    src = torch.rand((1, 1) + shape, device=dev)
    smooth = lambda shp, sig: (torch.nn.functional.interpolate(  # noqa: E731  registration-like smooth displacement field
        torch.randn((1, 3) + tuple(max(2, s // 16) for s in shp), device=dev) * sig, size=shp, mode="trilinear",
        align_corners=True).contiguous())
    flow = smooth(shape, 3.0)
    rough = torch.randn((1, 3) + shape, device=dev) * 3.0
    st = vxm.layers.SpatialTransformer(shape)
    stn = vxm.layers.SpatialTransformer(shape, mode="nearest")
    vel = smooth(half, 2.0)
    vi = vxm.layers.VecInt(half, 7)
    down, up = vxm.layers.ResizeTransform(2, 3), vxm.layers.ResizeTransform(0.5, 3)
    I, J = torch.rand((1, 1) + shape, device=dev), torch.rand((1, 1) + shape, device=dev)
    ncc = vxm.losses.NCC().loss
    with torch.no_grad():
        timeit(lambda: st(src, flow), V * 20, "warp_fwd_linear", "C=1, smooth flow sigma=3 voxels (registration-like)")
        timeit(lambda: stn(src, flow), V * 20, "warp_fwd_nearest", "C=1, smooth flow; exact replay of the reference's coordinate arithmetic (bit-exact labels)")
        timeit(lambda: st(src, rough), V * 20, "warp_fwd_linear_white_noise_flow", "C=1, i.i.d. N(0,3^2) flow per voxel (worst-case gather locality)")
        timeit(lambda: vi(vel), Vh * 24 * 7, "vecint_fwd_7steps", "single cooperative launch; field is L2 resident, so frac can "
               "exceed 1 against the HBM peak")
        timeit(lambda: down(flow), (V + Vh) * 12, "resize_down")
        timeit(lambda: up(vel), (V + Vh) * 12, "resize_up")
        timeit(lambda: ncc(I, J), V * 8, "ncc_fwd", "no saved fields (inference / validation)")

    # backward legs: the autograd node's backward is timed alone (forward outside the events); bytes per SURVEY 8(d)
    def timeit_bwd(make, nbytes, name, note=""):
        def run():
            y, g = make()
            return lambda: y.backward(g, retain_graph=True)
        fn = run()
        timeit(fn, nbytes, name, note)

    fl = flow.clone().requires_grad_(True)
    timeit_bwd(lambda: (st(src, fl), torch.ones((1, 1) + shape, device=dev)), V * 36, "warp_bwd_linear",
               "d/d flow only (the moving image needs no gradient in training): reads grad, flow, src; writes 3 planes")
    vl = vel.clone().requires_grad_(True)
    timeit_bwd(lambda: (vi(vl), torch.ones_like(vel)), Vh * 36 * 7, "vecint_bwd_7steps", "single cooperative launch, red.global.add.v4 scatter")
    timeit_bwd(lambda: (up(vl), torch.ones((1, 3) + shape, device=dev)), (V + Vh) * 12, "resize_up_bwd", "adjoint of the x2 upsampling (reads the full-resolution gradient)")
    timeit_bwd(lambda: (down(fl), torch.ones((1, 3) + half, device=dev)), (V + Vh) * 12, "resize_down_bwd")
    Jg = J.clone().requires_grad_(True)
    timeit(lambda: ncc(I, Jg), V * 8 + V * 12, "ncc_fwd_training", "forward that also stores the 3 fields the backward box-filters")
    timeit_bwd(lambda: (ncc(I, Jg), torch.ones((), device=dev)), V * 12 + V * 12, "ncc_bwd", "reads I, J + 3 saved fields, writes dJ")
    return out


def c4_sweep(vxm, dev, peaks):
    """BASELINE config 4 (SURVEY 8(d) C4): inference-only SpatialTransformer + VecInt throughput sweep at 256^3 / 128^3,
    fp32, white-noise flows of std sigma voxels.  GB/s are algorithmic bytes (SURVEY 8(d)) / CUDA-event time."""
    import torch
    full, half = (256,) * 3, (128,) * 3
    V, Vh = 256 ** 3, 128 ** 3
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    out = dict(warp={}, vecint={}, note="256^3 warp: src rand (1,C,256^3), flow randn*sigma; VecInt on randn*2 fields (1..B,3,S^3); "
               "3 warm-up + 5 timed launches, 256 MB L2 flush between launches; frac = GB/s / measured copy peak")

    def timeit(fn, nbytes):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(5):
            flush.zero_()
            torch.cuda._sleep(300000)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        t = statistics.median(ts)
        gbs = nbytes / (t * 1e-3) / 1e9
        return dict(us=round(t * 1e3, 1), gbs=round(gbs, 1), frac=round(gbs / peaks["hbm"], 3))

    with torch.no_grad():
        noise = torch.randn((1, 3) + full, device=dev)
        for C in (1, 3, 30):
            src = torch.rand((1, C) + full, device=dev)
            for mode in ("bilinear", "nearest"):
                st = vxm.layers.SpatialTransformer(full, mode=mode)
                for sigma in (0, 1, 4, 16):
                    flow = noise * float(sigma)
                    out["warp"]["C%d_%s_sigma%d" % (C, mode, sigma)] = timeit(lambda: st(src, flow), V * (8 * C + 12))
                    del flow
            del src
        del noise
        for S, Vs in ((128, Vh), (256, V)):
            for B in (1, 2, 4):
                vel = torch.randn((B, 3) + (S,) * 3, device=dev) * 2.0
                for n in range(1, 8):
                    vi = vxm.layers.VecInt((S,) * 3, n)
                    out["vecint"]["S%d_B%d_n%d" % (S, B, n)] = timeit(lambda: vi(vel), B * Vs * 24 * n)
                del vel
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    else:
        b200_arm(a)
