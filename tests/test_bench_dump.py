"""CPU: bench.py --dump-outputs writes float32 / float64 .npy files within its byte budget, whole where they fit and as
the same seeded sample from run to run where they do not."""
import os

import numpy as np
import torch

import bench


def _dump(out_dir, arrays):
    bench.dump_outputs(str(out_dir), arrays)
    return {f[:-4]: np.load(os.path.join(str(out_dir), f)) for f in os.listdir(str(out_dir))}


def test_dump_outputs_budget_dtypes_and_repeatable_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 1 << 20)
    g = torch.Generator().manual_seed(0)
    arrays = {"cost": torch.tensor(1.5), "inertia": torch.arange(35, dtype=torch.float64),
              "mask": torch.randint(0, 16, (64, 64), dtype=torch.uint8, generator=g),
              "emb": torch.randn(8, 256, 256, generator=g)}
    a = _dump(tmp_path / "a", arrays)
    b = _dump(tmp_path / "b", arrays)
    assert sorted(a) == sorted(arrays)
    assert sum(os.path.getsize(os.path.join(str(tmp_path / "a"), f)) for f in os.listdir(str(tmp_path / "a"))) <= 1 << 20
    assert a["inertia"].dtype == np.float64 and all(a[n].dtype == np.float32 for n in ("cost", "mask", "emb"))
    for n in ("cost", "inertia", "mask"):             # small enough: written whole, shape kept
        np.testing.assert_array_equal(a[n], arrays[n].numpy().astype(a[n].dtype))
    emb = arrays["emb"].numpy().reshape(-1)
    assert a["emb"].ndim == 1 and 0 < a["emb"].size < emb.size
    assert np.isin(a["emb"], emb).all()
    for n in arrays:
        np.testing.assert_array_equal(a[n], b[n])
