"""CPU tests of the host-side evaluation helpers (voxelmorph_b200/utils.py, next rows N2 / N3) against the oracle
restatements (oracle/spec_np.py) and the reference's outputs (py/utils.py:265-287, :473-516) frozen into
tests/golden/reference_outputs.json by oracle/make_golden_outputs.py."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import cases, spec_np


def fields():
    for shape in ((7, 9), (6, 7, 8), (2, 3, 2)):
        d = cases.smooth_field(21, len(shape), shape, scale=4.0)[0]
        yield np.moveaxis(d, 0, -1).astype(np.float64)


def test_dice_matches_oracle():
    from voxelmorph_b200 import utils
    rng = np.random.RandomState(9)
    a, b = rng.randint(0, 6, size=(8, 9, 10)), rng.randint(0, 7, size=(8, 9, 10))
    for kw in (dict(), dict(include_zero=True), dict(labels=[2, 5, 11]), dict(labels=[0, 3], include_zero=True)):
        assert np.allclose(utils.dice(a, b, **kw), spec_np.dice_overlap(a, b, **kw), rtol=0, atol=1e-15), kw
    assert np.array_equal(utils.dice(a, a), np.ones(5))
    with pytest.raises(ValueError):
        utils.dice(a, b[:4])


def test_jacobian_determinant_matches_oracle_and_counts_folds():
    from voxelmorph_b200 import utils
    for d in fields():
        np.testing.assert_allclose(utils.jacobian_determinant(d), spec_np.jacobian_determinant(d), rtol=0, atol=1e-12)
    shape = (5, 6, 7)
    grid = np.stack(np.meshgrid(*[np.arange(s, dtype=np.float64) for s in shape], indexing="ij"), 0)
    assert utils.count_folds(np.zeros((3,) + shape)) == 0
    assert utils.count_folds((-2.0 * grid)[np.newaxis]) == int(np.prod(shape))      # x -> -x folds everywhere in 3-D
    with pytest.raises(AssertionError):
        utils.jacobian_determinant(np.zeros((4, 4, 4, 2)))


def test_against_live_reference():
    from voxelmorph_b200 import utils
    ref = json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))["eval_helpers"]
    rng = np.random.RandomState(2)
    a, b = rng.randint(0, 5, size=(9, 10, 11)), rng.randint(0, 5, size=(9, 10, 11))
    assert np.allclose(utils.dice(a, b), np.array(ref["utils_dice"]), rtol=0, atol=1e-15)
    for d, r in zip(list(fields())[:2], ref["utils_jacdet"], strict=True):
        np.testing.assert_allclose(utils.jacobian_determinant(d), np.array(r), rtol=0, atol=1e-12)
