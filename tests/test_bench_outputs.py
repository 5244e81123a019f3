"""bench.py --dump-outputs: the files written for one step's results (CPU tensors stand in for the device ones)."""
import os

import numpy as np
import pytest
import torch

import bench
from manuscript_b200.batch import PageBatchResult


def _result(n_pages=4, per_page=30, n_crops=100, cap=120):
    g = torch.Generator().manual_seed(0)
    return PageBatchResult(boxes=torch.rand((n_pages, 2 * per_page, 9), generator=g),
                           box_counts=torch.full((n_pages,), per_page, dtype=torch.int32),
                           crops=torch.randint(0, 2048, (cap, 5), dtype=torch.int32, generator=g),
                           n_crops=torch.tensor([n_crops], dtype=torch.int32),
                           batch=torch.rand((cap, 3, 32, 128), generator=g),
                           flags=torch.zeros((n_pages,), dtype=torch.int32))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_the_step_results(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_CROPS", 10)
    res = _result()
    info = bench.dump_outputs(str(tmp_path / "a"), res)
    out = _load(tmp_path / "a")
    assert sorted(out) == info["files"] and info["bytes"] == sum(a.nbytes for a in out.values())
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    np.testing.assert_array_equal(out["boxes"], res.boxes[:, :30].reshape(-1, 9).numpy())
    np.testing.assert_array_equal(out["box_counts"], [30] * 4)
    np.testing.assert_array_equal(out["flags"], [0] * 4)
    np.testing.assert_array_equal(out["crops"], res.crops[:100].numpy())
    np.testing.assert_array_equal(out["batch_crop_sums"],
                                  torch.sum(res.batch[:100], dim=(1, 2, 3), dtype=torch.float64).numpy())
    idx = out["batch_sample_index"].astype(np.int64)
    assert len(idx) == 10 and len(set(idx)) == 10 and (np.diff(idx) > 0).all() and idx[-1] < 100
    np.testing.assert_array_equal(out["batch_sample"], res.batch[idx].numpy())
    # the sample is fixed: a second dump of the same results is identical file for file
    bench.dump_outputs(str(tmp_path / "b"), res)
    again = _load(tmp_path / "b")
    assert all(np.array_equal(out[k], again[k]) for k in out)


def test_dump_outputs_stays_within_its_budget(tmp_path, monkeypatch):
    res = _result()
    bench.dump_outputs(str(tmp_path / "full"), res)
    fixed = sum(a.nbytes for k, a in _load(tmp_path / "full").items() if not k.startswith("batch_sample"))
    crop = 3 * 32 * 128 * 4  # one float32 crop of the batch; its index takes 8 more bytes
    monkeypatch.setattr(bench, "DUMP_BYTES", fixed + 3 * (crop + 8) + 5)
    bench.dump_outputs(str(tmp_path / "small"), res)
    assert len(np.load(tmp_path / "small" / "batch_sample_index.npy")) == 3
    monkeypatch.setattr(bench, "DUMP_BYTES", fixed - 1)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "over"), res)
