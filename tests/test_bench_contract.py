"""bench.py's reference arm prints one JSON line with the contract's keys (runs the CPU oracle port on one keyframe)."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line(tmp_path):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    lines = [l for l in r.stdout.strip().splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-500:] + r.stderr[-500:]
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]
    assert d["steps"] == 1
    import numpy as np
    cv, sf = np.load(tmp_path / "dump" / "cost_volume.npy"), np.load(tmp_path / "dump" / "single_frame_cvs.npy")
    assert cv.dtype == np.float32 and sf.dtype == np.float32 and cv.shape[1] == 32 and sf.shape[1:] == (4, 32)
    assert cv.shape[0] == sf.shape[0] > 0 and np.isfinite(cv).all() and np.isfinite(sf).all()


def test_steps_below_one_is_rejected():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=300, cwd=str(ROOT))
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_is_a_fixed_pixel_sample(tmp_path, monkeypatch):
    """--dump-outputs: float32 depth-plane profiles of the same pixels on every call, each row read from the volumes at one
    (b, y, x), pixels in ascending order, the sample bounded by DUMP_BYTES."""
    import numpy as np
    import torch
    sys.path.insert(0, str(ROOT))
    import bench
    g = torch.Generator().manual_seed(1)
    cv, sfcv = torch.randn(2, 8, 6, 10, generator=g), torch.randn(3, 2, 8, 6, 10, generator=g)
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 8 * (1 + 3) * 50)         # room for 50 of the 120 pixels
    bench.dump_outputs(tmp_path / "a", cv, sfcv)
    bench.dump_outputs(tmp_path / "b", cv, sfcv)
    a_cv, a_sf = np.load(tmp_path / "a" / "cost_volume.npy"), np.load(tmp_path / "a" / "single_frame_cvs.npy")
    assert a_cv.dtype == np.float32 and a_cv.shape == (50, 8) and a_sf.dtype == np.float32 and a_sf.shape == (50, 3, 8)
    assert np.array_equal(a_cv, np.load(tmp_path / "b" / "cost_volume.npy"))
    assert np.array_equal(a_sf, np.load(tmp_path / "b" / "single_frame_cvs.npy"))
    profiles = cv.permute(0, 2, 3, 1).reshape(-1, 8).numpy()               # [b, y, x] -> D planes
    pix = [int(np.flatnonzero((profiles == row).all(1))[0]) for row in a_cv]
    assert pix == sorted(set(pix))
    assert np.array_equal(a_sf, sfcv.permute(1, 3, 4, 0, 2).reshape(-1, 3, 8).numpy()[pix])
    assert bench.DUMP_BYTES <= 64 * 10 ** 6
