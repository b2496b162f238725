"""Drop-in boundary (SURVEY.md section 8(b1), 8(e)): `import voxelmorph as vxm` resolves to this repo, the training loop
of the reference's scripts/torch/train.py (restated in tests/train_loop_body.py) runs against it, and a training script
started once per GPU becomes data parallel without a wrapper.

CPU part: import surface, TransparentDP under gloo (world 2), the launcher.  GPU part (`-m gpu`): the train.py loop body
for three steps on one GPU, and on two GPUs under the launcher (skipped with fewer than two devices)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

HERE = os.path.dirname(os.path.abspath(__file__))


def run_py(args, env=None, cwd=None, timeout=600):
    e = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    e.pop("VXM_BACKEND", None)
    e.update(env or {})
    return subprocess.run([sys.executable] + list(args), env=e, cwd=cwd, capture_output=True, text=True, timeout=timeout)


def make_volumes(tmp_path, n=3, shape=(32, 32, 32), seed=0):
    from oracle import cases
    names = []
    for i in range(n):
        p = tmp_path / ("vol%d.npz" % i)
        np.savez_compressed(p, vol=cases.smooth_volume(seed + i, shape)[0, 0])
        names.append(str(p))
    lst = tmp_path / "list.txt"
    lst.write_text("\n".join(names) + "\n")
    return str(lst), names


def test_import_surface_matches_reference_package():
    code = (
        "import os; os.environ['VXM_BACKEND']='pytorch'\n"
        "import voxelmorph as vxm, inspect\n"
        "assert vxm.__file__.startswith(%r), vxm.__file__\n"
        "for n in ('SpatialTransformer','VecInt','ResizeTransform'): assert hasattr(vxm.layers, n) and hasattr(vxm.torch.layers, n)\n"
        "for n in ('VxmDense','Unet','ConvBlock'): assert hasattr(vxm.networks, n) and hasattr(vxm.torch.networks, n)\n"
        "for n in ('NCC','MSE','Dice','Grad'): assert hasattr(vxm.losses, n)\n"
        "for n in ('volgen','scan_to_scan','scan_to_atlas','semisupervised'): assert hasattr(vxm.generators, n)\n"
        "for n in ('read_file_list','read_pair_list','load_volfile','save_volfile','load_labels','pad','resize','dice',"
        "'jacobian_determinant','filter_labels','affine_shift_to_matrix','default_unet_features','get_backend'): assert hasattr(vxm.py.utils, n), n\n"
        "assert vxm.default_unet_features() == [[16,32,32,32],[32,32,32,32,32,16,16]]\n"
        "assert vxm.torch.modelio.LoadableModel in vxm.networks.VxmDense.__mro__\n"
        "sig = inspect.signature(vxm.networks.VxmDense.__init__)\n"
        "assert list(sig.parameters)[1:] == ['inshape','nb_unet_features','nb_unet_levels','unet_feat_mult','nb_unet_conv_per_level',"
        "'int_steps','int_downsize','bidir','use_probs','src_feats','trg_feats','unet_half_res']\n"
        "m = vxm.networks.VxmDense((32,32,32))\n"
        "assert vxm.networks.ops.resolve_engine(m) == 'bf16x3'      # tensor cores by default through the drop-in package\n"
        "m2 = vxm.networks.VxmDense((32,32,32), nb_unet_features=[[4,8,8,8],[8,8,8,8,8,4,4]])\n"
        "assert vxm.networks.ops.resolve_engine(m2) == 'f32'        # shapes the tensor-core engine lacks fall back to the fp32 CUDA engine\n"
        "print('surface ok')\n" % ROOT)
    r = run_py(["-c", code])
    assert r.returncode == 0 and "surface ok" in r.stdout, r.stdout + r.stderr


def test_other_backends_are_refused():
    r = run_py(["-c", "import voxelmorph"])
    assert r.returncode != 0 and "pytorch backend only" in r.stderr


DP_WORKER = r'''
import os, sys, json
sys.path.insert(0, os.environ["VXM_ROOT"])
import torch
from voxelmorph_b200 import dist as vdist
rank = int(os.environ["RANK"])
torch.manual_seed(100 + rank)                      # every rank draws DIFFERENT initial weights ...
net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Tanh(), torch.nn.Linear(5, 1))
dp = vdist.attach_if_distributed(net)
assert dp is not None and dp.world == 2
w0 = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).clone()
opt = torch.optim.Adam(net.parameters(), lr=1e-2)
g = torch.Generator().manual_seed(7)
X = torch.randn(8, 6, generator=g); Y = torch.randn(8, 1, generator=g)
xs, ys = X[rank::2], Y[rank::2]                      # ... and sees its own shard of the batch
for step in range(3):
    loss = ((net(xs) - ys) ** 2).mean()
    opt.zero_grad()
    loss.backward()
    opt.step()
w = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
json.dump(dict(w0=w0.tolist(), w=w.tolist(), n=dp.allreduces, writer=dp.is_writer()), open(os.path.join(os.environ["VXM_OUT"], "dp_%d.json" % rank), "w"))
'''


def test_transparent_dp_gloo_world2(tmp_path):
    """Two CPU processes (gloo): initial weights are rank 0's after the broadcast, every step issues exactly one
    allreduce, and three Adam steps on per-rank shards equal three single-process steps on the full batch."""
    import socket
    import torch
    script = tmp_path / "dp_worker.py"
    script.write_text(DP_WORKER)
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    env = dict(os.environ, VXM_ROOT=ROOT, VXM_OUT=str(tmp_path))
    r = subprocess.run([sys.executable, "-m", "voxelmorph_b200.launch", "--nproc", "2", "--gpu-flag", "", "--master-port", str(port), str(script)],
                       env=dict(env, PYTHONPATH=ROOT), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    a, b = (json.load(open(tmp_path / ("dp_%d.json" % k))) for k in (0, 1))
    assert a["w0"] == b["w0"] and a["w"] == b["w"]            # replicas identical before and after
    assert a["n"] == b["n"] == 3 and a["writer"] and not b["writer"]
    # single-process reference on the full batch from rank 0's initial weights
    torch.manual_seed(100)
    net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Tanh(), torch.nn.Linear(5, 1))
    opt = torch.optim.Adam(net.parameters(), lr=1e-2)
    g = torch.Generator().manual_seed(7)
    X = torch.randn(8, 6, generator=g)
    Y = torch.randn(8, 1, generator=g)
    for _ in range(3):
        loss = ((net(X) - Y) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
    w = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
    assert np.allclose(np.array(a["w"]), w.numpy(), rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_train_loop_body_three_steps_single_gpu(cuda, tmp_path):
    lst, _ = make_volumes(tmp_path, n=3)
    rep = str(tmp_path / "rep.json")
    r = run_py([os.path.join(HERE, "train_loop_body.py"), "--img-list", lst, "--model-dir", str(tmp_path / "m"), "--image-loss", "ncc",
                "--steps-per-epoch", "3", "--report", rep], cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.load(open(rep + ".0"))
    assert len(d["losses"]) == 3 and all(np.isfinite(d["losses"])) and d["engine"] == "bf16x3" and d["allreduces"] is None
    assert (tmp_path / "m" / "0000.pt").exists() and (tmp_path / "m" / "0001.pt").exists()
    import voxelmorph_b200 as vxm
    m = vxm.networks.VxmDense.load(str(tmp_path / "m" / "0001.pt"), "cuda")
    assert m.config["inshape"] == (32, 32, 32)


@pytest.mark.gpu
def test_train_loop_body_two_gpus_transparent_dp(cuda, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    lst, _ = make_volumes(tmp_path, n=4)
    rep = str(tmp_path / "rep.json")
    e = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "voxelmorph_b200.launch", "--nproc", "2", os.path.join(HERE, "train_loop_body.py"),
                        "--img-list", lst, "--model-dir", str(tmp_path / "m"), "--image-loss", "ncc", "--steps-per-epoch", "3",
                        "--report", rep], env=e, cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout + r.stderr)[-4000:]
    a, b = json.load(open(rep + ".0")), json.load(open(rep + ".1"))
    assert a["allreduces"] == b["allreduces"] == 3                   # one gradient exchange per step
    assert abs(a["param_sum"] - b["param_sum"]) <= 1e-9 * a["param_abs"]   # replicas stay identical
    assert sorted(os.listdir(tmp_path / "m")) == ["0000.pt", "0001.pt"]     # written once (rank 0), not twice


@pytest.mark.gpu
def test_data_feed_never_creates_the_cuda_context(cuda, tmp_path):
    """scripts/torch/train.py draws its first batch (:113) before it sets CUDA_VISIBLE_DEVICES (:125): importing the package and
    drawing batches must leave CUDA uninitialised, or `--gpu N` / one process per GPU silently land on device 0."""
    lst, _ = make_volumes(tmp_path, n=2)
    code = ("import os, torch\n"
            "os.environ['VXM_BACKEND'] = 'pytorch'\n"
            "import voxelmorph as vxm\n"
            "g = vxm.generators.scan_to_scan(vxm.py.utils.read_file_list(%r), batch_size=1, bidir=False, add_feat_axis=True)\n"
            "a = next(g); b = next(g)\n"
            "assert not torch.cuda.is_initialized(), 'the data feed initialised CUDA'\n"
            "os.environ['CUDA_VISIBLE_DEVICES'] = '0'\n"
            "x = torch.from_numpy(a[0][0]).to('cuda').float()\n"
            "c = next(g)\n"                              # later draws may page-lock: the process has its context now
            "print('ok', torch.cuda.device_count(), float(x.sum()))\n" % lst)
    r = run_py(["-c", code], cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout.startswith("ok 1 "), (r.stdout + r.stderr)[-2000:]
