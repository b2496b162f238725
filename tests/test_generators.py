"""CPU tests of the host-side data feed (voxelmorph_b200/generators.py, "next" row N1) against the reference generators:
same yield structure, shapes, values and the same sequence of np.random draws, as frozen from the unmodified reference:
shapes and sums in tests/golden/generators.json (oracle/make_golden_generators.py), every yielded array by digest in
tests/golden/reference_outputs.json (oracle/make_golden_outputs.py)."""
import json
import os

import numpy as np
import pytest

from conftest import ROOT
from oracle import cases

GOLDEN = os.path.join(ROOT, "tests", "golden", "generators.json")
REFERENCE_OUTPUTS = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")


def make_dataset(tmp_path, n=5, shape=(6, 8, 10), with_seg=True):
    """n small npz volumes; volume i is filled with a smooth pattern offset by i so that every draw is identifiable."""
    rng = np.random.RandomState(1234)
    files = []
    for i in range(n):
        vol = (rng.rand(*shape) * 0.5 + i).astype(np.float32 if i % 2 else np.float64)
        seg = rng.randint(0, 4, size=shape).astype(np.int32)
        f = os.path.join(str(tmp_path), "vol%02d.npz" % i)
        if with_seg:
            np.savez_compressed(f, vol=vol, seg=seg)
        else:
            np.savez_compressed(f, vol=vol)
        files.append(f)
    return files


def summarize(item):
    """Nested lists/tuples of arrays -> nested lists of [shape, float64 sum, first volume id]."""
    if isinstance(item, (list, tuple)):
        return [summarize(x) for x in item]
    a = np.asarray(item)
    return [list(a.shape), round(float(a.astype(np.float64).sum()), 4)]


CASES = {
    "volgen_b1": dict(kind="volgen", kw=dict(batch_size=1)),
    "volgen_b3_seg": dict(kind="volgen", kw=dict(batch_size=3, segs=True)),
    "volgen_pad": dict(kind="volgen", kw=dict(batch_size=2, pad_shape=(8, 8, 12))),
    "s2s": dict(kind="scan_to_scan", kw=dict(batch_size=1)),
    "s2s_bidir_same": dict(kind="scan_to_scan", kw=dict(batch_size=2, bidir=True, prob_same=0.5)),
    "s2s_nowarp": dict(kind="scan_to_scan", kw=dict(batch_size=1, no_warp=True)),
    "s2a": dict(kind="scan_to_atlas", kw=dict(batch_size=2)),
    "s2a_bidir_seg": dict(kind="scan_to_atlas", kw=dict(batch_size=1, bidir=True, segs=True)),
    "semi": dict(kind="semisupervised", kw=dict(labels=[1, 2, 3], downsize=2)),
    "semi_atlas": dict(kind="semisupervised", kw=dict(labels=[0, 2], downsize=2, atlas=True)),
}


def run_case(mod, files, case, steps=6, seed=7):
    np.random.seed(seed)
    kw = dict(case["kw"])
    if case["kind"] == "volgen":
        gen = mod.volgen(files, **kw)
    elif case["kind"] == "scan_to_scan":
        gen = mod.scan_to_scan(files, **kw)
    elif case["kind"] == "semisupervised":   # the npz files carry 'vol' and 'seg' (seg_names=True, generators.py:158)
        atlas = files[0] if kw.pop("atlas", False) else None
        gen = mod.semisupervised(files, True, kw.pop("labels"), atlas_file=atlas, **kw)
    else:
        atlas = np.load(files[0])["vol"][np.newaxis, ..., np.newaxis]
        gen = mod.scan_to_atlas(files, atlas, **kw)
    return [next(gen) for _ in range(steps)]


def fingerprint(item):
    """Nested lists/tuples of arrays -> nested lists of cases.digest of each array's float32 values."""
    if isinstance(item, (list, tuple)):
        return [fingerprint(x) for x in item]
    return cases.digest(np.asarray(item).astype(np.float32))


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_frozen_reference_behaviour(tmp_path, name):
    from voxelmorph_b200 import generators
    gold = json.load(open(GOLDEN))
    files = make_dataset(tmp_path)
    got = [summarize(x) for x in run_case(generators, files, CASES[name])]
    assert got == gold[name]


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_live_reference(tmp_path, name):
    """Every array of six yields equals the reference generator's, value for value (as float32)."""
    from voxelmorph_b200 import generators
    gold = json.load(open(REFERENCE_OUTPUTS))["generators"]
    files = make_dataset(tmp_path)
    assert fingerprint(run_case(generators, files, CASES[name])) == gold[name]


def test_decode_once_float32_and_views(tmp_path):
    from voxelmorph_b200 import generators
    files = make_dataset(tmp_path, n=3)
    cache = generators.VolumeCache(pin=False)
    np.random.seed(0)
    gen = generators.volgen(files, batch_size=1, cache=cache)
    batches = [next(gen)[0] for _ in range(12)]
    assert cache.misses <= 3 and cache.hits >= 9                    # every file inflated at most once
    assert all(b.dtype == np.float32 and b.shape == (1, 6, 8, 10, 1) for b in batches)
    assert all(not b.flags.owndata for b in batches)                # batch of one is a view of the cached volume
    with pytest.raises(ValueError):
        batches[0][0, 0, 0, 0, 0] = 1.0                             # cached volumes are read-only
    inv, outv = next(generators.scan_to_scan(files, batch_size=2, cache=cache))
    assert outv[-1].dtype == np.float32 and outv[-1].shape == (2, 6, 8, 10, 3) and not outv[-1].any()
    seg = next(generators.volgen(files, segs=True, cache=cache))[1]
    assert seg.dtype == np.int32                                    # label maps keep their integer type


def test_cache_eviction_and_errors(tmp_path):
    from voxelmorph_b200 import generators
    files = make_dataset(tmp_path, n=4, with_seg=False)
    one = 6 * 8 * 10 * 4
    cache = generators.VolumeCache(max_bytes=2 * one, pin=False)
    for f in files:
        cache.get(f)
    assert len(cache) == 2
    with pytest.raises(ValueError, match="is not a file"):
        generators.load_volfile(os.path.join(str(tmp_path), "missing.npz"))
    with pytest.raises(ValueError, match="must match"):
        next(generators.volgen(files, segs=files[:2]))
    with pytest.raises(ValueError, match="cannot hold"):
        next(generators.volgen(files, pad_shape=(4, 4, 4), cache=generators.VolumeCache(pin=False)))


def test_prefetcher_preserves_order_and_propagates_errors(tmp_path):
    from voxelmorph_b200 import generators
    files = make_dataset(tmp_path, n=4)
    np.random.seed(3)
    direct = [summarize(x) for x in run_case(generators, files, CASES["s2s"], steps=8, seed=3)]
    np.random.seed(3)
    pf = generators.Prefetcher(generators.scan_to_scan(files, batch_size=1), depth=3)
    assert [summarize(next(pf)) for _ in range(8)] == direct
    pf.close()

    def boom():
        yield 1
        raise RuntimeError("decode failed")

    pf = generators.Prefetcher(boom())
    assert next(pf) == 1
    with pytest.raises(RuntimeError, match="decode failed"):
        next(pf)


def test_data_feed_never_asks_for_cuda(tmp_path, monkeypatch):
    """The reference's train.py sets CUDA_VISIBLE_DEVICES (scripts/torch/train.py:125) AFTER drawing its first batch (:113); the CUDA
    runtime reads that variable when it initialises, so the feed must not touch it: neither torch.cuda.is_available() (which
    initialises the driver) nor page-locked allocations before the process has a context of its own."""
    import numpy as np
    import torch
    from voxelmorph_b200 import generators as G

    def boom(*a, **k):
        raise AssertionError("the data feed queried / initialised CUDA")
    monkeypatch.setattr(torch.cuda, "is_available", boom)
    monkeypatch.setattr(torch.cuda, "init", boom)
    monkeypatch.setattr(torch.cuda, "is_initialized", lambda: False)
    names = []
    for i in range(2):
        p = tmp_path / ("v%d.npz" % i)
        np.savez_compressed(p, vol=np.random.default_rng(i).random((8, 10, 12)))
        names.append(str(p))
    g = G.scan_to_scan(names, batch_size=2, bidir=False, add_feat_axis=True)
    (a, b), _ = next(g)
    assert a.dtype == np.float32 and a.shape == (2, 8, 10, 12, 1) and b.shape == a.shape
    next(g)
