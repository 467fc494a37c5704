"""bench.py --dump-outputs: the arrays it writes (float32 / float64 .npy, whole when they fit the budget, otherwise the same
seeded rows of every array of the same length, under the budget in all)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def outputs(n, e):
    g = torch.Generator().manual_seed(n)
    return {"loss": torch.tensor(1.25), "recon_loss": torch.tensor(0.5), "hs": torch.randn(n, 64, generator=g),
            "hf": torch.randn(n, 64, generator=g), "pred_bin": torch.randint(0, 2, (2 * e,), generator=g, dtype=torch.int32)}


def load_dir(d):
    out = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    return out


def test_outputs_that_fit_are_written_whole(tmp_path):
    arrays = outputs(300, 500)
    bench.write_outputs(str(tmp_path), arrays)
    got = load_dir(str(tmp_path))
    assert set(got) == set(arrays)
    for k, a in arrays.items():
        assert got[k].shape == tuple(a.shape) and np.array_equal(got[k], a.float().numpy()), k


def test_large_outputs_keep_the_same_seeded_rows_under_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 400_000)
    arrays = outputs(4000, 3000)
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays)
    a, b = load_dir(str(tmp_path / "a")), load_dir(str(tmp_path / "b"))
    assert set(a) == set(arrays) | {"hs_rows", "hf_rows", "pred_bin_rows"}
    assert all(np.array_equal(a[k], b[k]) for k in a)                       # fixed seed: the same sample every time
    assert sum(x.nbytes for x in a.values()) <= 400_000
    rows = a["hs_rows"].astype(np.int64)
    assert 0 < len(rows) < 4000 and np.all(np.diff(rows) > 0) and np.array_equal(rows, a["hf_rows"])
    assert np.array_equal(a["hs"], arrays["hs"].numpy()[rows]) and np.array_equal(a["hf"], arrays["hf"].numpy()[rows])
    prow = a["pred_bin_rows"].astype(np.int64)
    assert np.array_equal(a["pred_bin"], arrays["pred_bin"].float().numpy()[prow])
    assert float(a["loss"]) == 1.25                                          # scalars stay whole


@pytest.mark.parametrize("extra", [["--impl", "reference", "--dump-outputs", "out"], ["--steps", "0"]])
def test_bench_rejects_arguments_it_cannot_honour(extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True)
    assert r.returncode == 2 and "error" in r.stderr
