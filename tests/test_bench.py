"""bench.py --dump-outputs: what the timed path computed, written as .npy files that two builds can be compared by."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _positions(full, sample):
    where = {v: i for i, v in enumerate(full.reshape(-1).tolist())}
    return np.array([where[v] for v in sample.tolist()])


def test_dump_outputs_writes_float32_and_a_fixed_sample_of_large_arrays(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 1000)
    g = torch.Generator().manual_seed(3)
    big64 = torch.rand((4, 3, 20, 30), generator=g, dtype=torch.float64)
    big32 = torch.rand((4, 3, 20, 30), generator=g)
    small = torch.rand((2, 5), generator=g).to(torch.bfloat16)
    arrays = {"big64": big64, "big32": big32, "small": small, "scalar": torch.tensor(1.5), "flag": False, "none": None,
              "ints": torch.arange(3)}
    bench.dump_outputs(arrays, str(tmp_path / "a"))
    bench.dump_outputs(arrays, str(tmp_path / "b"))
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["big32.npy", "big64.npy", "scalar.npy", "small.npy"]
    a = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        assert np.array_equal(a[n[:-4]], np.load(tmp_path / "b" / n)), n             # the same sample from call to call
    assert a["big64"].dtype == np.float64 and a["big32"].dtype == np.float32 and a["small"].dtype == np.float32
    assert a["big64"].shape == a["big32"].shape == (1000,) and a["small"].shape == (2, 5) and a["scalar"].shape == ()
    np.testing.assert_array_equal(a["small"], small.float().numpy())
    # distinct elements in ascending flat order, and one index set for arrays of the same size
    pos = _positions(big64.numpy(), a["big64"])
    assert np.all(np.diff(pos) > 0)
    np.testing.assert_array_equal(pos, _positions(big32.numpy(), a["big32"]))


def test_dump_outputs_keeps_to_its_size_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1000)
    with pytest.raises(ValueError):
        bench.dump_outputs({"x": torch.zeros(300)}, str(tmp_path / "d"))
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_bench_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    """With --steps 1 the one timed step runs on the batch whose rd terms the JSON line reports, so the dumped terms must match it."""
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--batch", "2", "--dump-outputs", str(out),
           "--no-cpu-baseline", "--no-residual", "--no-strong", "--no-config3", "--no-other-arms", "--no-scalable", "--no-train-step"]
    r = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 1
    a = {p.name[:-4]: np.load(p) for p in out.glob("*.npy")}
    assert {"x_hat", "y", "y_in", "z_in", "p_y", "logp_y", "p_z", "weights", "mus", "sigmas", "bpp_total", "psnr",
            "mse_per_image"} <= set(a)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["x_hat"].shape == (bench.DUMP_MAX_ELEMS,) and a["y_in"].shape == (2, 128, 32, 48) and a["mse_per_image"].shape == (2,)
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
    assert np.array_equal(a["y_in"], np.round(a["y_in"]))
    assert abs(float(a["bpp_total"]) - line["rd"]["bpp_total"]) <= 1e-6 * abs(line["rd"]["bpp_total"])
    assert abs(float(a["psnr"]) - line["rd"]["psnr"]) <= 1e-6 * abs(line["rd"]["psnr"])
