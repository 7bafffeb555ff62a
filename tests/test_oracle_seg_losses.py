"""CPU: the semantic-loss restatement (oracle/seg_losses_ref.py) against golden vectors produced by the reference's own
dice_loss (tests/golden/make_golden_seg.py)."""
import os

import numpy as np
import pytest

from oracle import seg_losses_ref as O
from tests.golden.make_golden_seg import SEG_CASES, seg_case


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "seg_losses.npz"))


@pytest.mark.parametrize("case", SEG_CASES, ids=[c[0] for c in SEG_CASES])
def test_restatement_matches_reference_golden(golden, case):
    name, seed, bs, nc, H, W, w, obg, time = case
    logits, cls, onehot = seg_case(case)
    o = O.seg_losses(logits, onehot, w, obg, 1.0, time, g_ce=0.7, g_dice=1.3)
    assert abs(o["ce"] - float(golden[name + "_ce"])) < 2e-6 * abs(o["ce"])
    assert abs(o["dice"] - float(golden[name + "_dice"])) < 2e-6
    g = golden[name + "_grad"]
    assert np.abs(o["grad"] - g).max() < 2e-6 * np.abs(g).max() + 1e-10
