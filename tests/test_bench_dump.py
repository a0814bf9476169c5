"""bench.py --dump-outputs: float32 .npy files, kept under the size cap by one seeded subset of rows shared by same-length arrays."""
import os

import numpy as np
import torch

import bench


def _outputs(pairs, h=24, w=48, num=50):
    g = torch.Generator().manual_seed(0)
    return {"warp": torch.rand(pairs, h, w, 4, generator=g, dtype=torch.float64), "certainty": torch.rand(pairs, h, w, generator=g),
            "sample_matches": torch.rand(pairs * num, 4, generator=g), "sample_certainty": torch.rand(pairs * num, generator=g)}


def test_dump_outputs_whole(tmp_path):
    out = _outputs(2)
    bench.dump_outputs(str(tmp_path), out)
    for k, v in out.items():
        a = np.load(tmp_path / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.float().numpy())


def test_dump_outputs_seeded_subset_under_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT", 64 << 10)
    out = _outputs(4)
    runs = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= bench.DUMP_LIMIT
        runs.append({k: np.load(tmp_path / d / f"{k}.npy") for k in out})
    assert all(np.array_equal(runs[0][k], runs[1][k]) for k in out)
    w, c = runs[0]["warp"], runs[0]["certainty"]
    assert w.ndim == 2 and w.shape[1] == 4 and 0 < len(w) < 4 * 24 * 48 and len(c) == len(w)
    # warp and certainty keep the same pixels, in pixel order
    flat_w, flat_c = out["warp"].float().reshape(-1, 4).numpy(), out["certainty"].reshape(-1).numpy()
    idx = np.flatnonzero(np.isin(flat_c, c))
    assert np.array_equal(flat_c[idx], c) and np.array_equal(flat_w[idx], w)
