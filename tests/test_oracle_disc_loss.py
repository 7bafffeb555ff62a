"""CPU: the numpy oracle of the discriminative loss against golden vectors produced by the
reference itself (tests/golden/make_golden.py)."""
import os
import sys

import numpy as np
import pytest

from isa_b200 import synth
from oracle import disc_loss as O

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import DISC_CASES  # noqa: E402


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "disc_loss.npz"))


@pytest.mark.parametrize("case", DISC_CASES, ids=[c[0] for c in DISC_CASES])
@pytest.mark.parametrize("dense", [False, True])
def test_oracle_matches_reference_golden(golden, case, dense):
    name, seed, bs, C, H, W, K, norm, kw = case
    d = synth.batch(seed, bs, C, H, W, K, **kw)
    tgt = synth.onehot(d["labels"], K) if dense else d["labels"]
    o = O.discriminative_loss(d["emb"], tgt, d["n_objects"], K, 0.5, 1.5, norm, want_grad=True,
                              grad_means=golden[name + "_gm"])
    assert abs(float(o["loss"]) - float(golden[name + "_loss"])) <= 1e-5 * abs(float(golden[name + "_loss"]))
    np.testing.assert_allclose(o["means"], golden[name + "_means"], atol=2e-6)
    gref = golden[name + "_grad"]
    assert np.abs(o["grad"] - gref).max() <= 1e-5 * np.abs(gref).max()
    o4 = O.discriminative_loss(d["emb"], tgt, d["n_objects"], K, 0.5, 1.5, norm, terms=(1, 1, 1, 1))
    np.testing.assert_allclose(o4["terms"], golden[name + "_terms"], rtol=1e-5, atol=1e-6)


def test_oracle_nan_on_empty_instance():
    # the reference's mean of an instance id < n_objects with no pixels is 0/0 -> NaN loss
    d = synth.batch(5, 1, 8, 16, 16, 4, n_min=2, n_max=2)
    n = np.array([3], dtype=np.int32)
    o = O.discriminative_loss(d["emb"], d["labels"], n, 4, 0.5, 1.5, 2)
    assert np.isnan(o["loss"])
