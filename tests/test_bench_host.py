"""bench.py host logic that needs no GPU: the reference arm's JSON line (the contract the driver parses), the shared config object of
the two arms, and the rank-independence of the synthetic snapshot block (what makes the N-GPU runs strong-scaled)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _bench():
    import importlib
    return importlib.import_module("bench")


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "small", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["r"] == 16 and d["config"]["freq_points_total"] == 512 and "small" in d["config"]["workload"]


def test_both_arms_share_one_config_object():
    b = _bench()
    wl = b.WORKLOADS["cfg3"]
    n = 1_000_000
    cfg = b.workload_config("cfg3", wl, n)
    assert cfg["N_dof_total"] == n and cfg["r"] == 256 and cfg["ports"] == 4 and cfg["freq_points_total"] == 100000
    assert cfg["workload"].startswith("cfg3: BASELINE configs[2]") and cfg["scaling"].startswith("strong")
    assert not any(k in cfg for k in ("model", "global_batch", "seq_len"))           # a workload, not a model
    # the default workload is the configuration the metric is quoted on
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'ap.add_argument("--workload", default="cfg3"' in src


def test_snapshot_block_does_not_depend_on_the_rank_count():
    b = _bench()
    n, r = 4003, 12
    whole = b.snapshot_rows(n, r, 0, n)
    assert whole.shape == (n, r) and np.isfinite(whole).all()
    for world in (2, 3, 8):
        parts = []
        for rank in range(world):
            lo, hi = rank * n // world, (rank + 1) * n // world
            parts.append(b.snapshot_rows(n, r, lo, hi))
        assert np.array_equal(np.concatenate(parts, axis=0), whole)                  # bit-identical global problem at every N
    assert np.linalg.matrix_rank(whole) == r


def test_dump_outputs_float64_capped_and_seeded(tmp_path, monkeypatch):
    """--dump-outputs: float64 files, complex arrays with a trailing (real, imag) axis, no file for an all-zero (None) operator, an
    array over its cap cut to a sorted seeded sample of its rows (the same rows on every run), 64 MB in all at the default caps."""
    import torch
    b = _bench()
    assert sum(b.DUMP_CAP.values()) + 4 * b.DUMP_CAP_OTHER <= 64e6          # gsm, q, info and the four reduced operators
    monkeypatch.setitem(b.DUMP_CAP, "gsm", 1 << 16)
    gsm = torch.randn(10000, 2, 2, dtype=torch.complex128)
    q = torch.randn(300, 8, dtype=torch.float64)
    info = torch.arange(10000, dtype=torch.int32)
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), {"gsm": gsm, "q": q, "a1_r": None, "info": info})
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["gsm.npy", "gsm_rows.npy", "info.npy", "q.npy"]
    for name in names:
        x = np.load(tmp_path / "a" / name)
        assert x.dtype == np.float64 and np.array_equal(x, np.load(tmp_path / "b" / name))
    rows = np.load(tmp_path / "a" / "gsm_rows.npy").astype(np.int64)
    g = np.load(tmp_path / "a" / "gsm.npy")
    assert g.shape == (rows.size, 2, 2, 2) and g.nbytes + rows.nbytes <= 1 << 16 and np.all(np.diff(rows) > 0)
    assert np.array_equal(g[..., 0] + 1j * g[..., 1], gsm.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "q.npy"), q.numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "info.npy"), np.arange(10000.0))
