"""bench.py contract (task statement, section 4): the committed bench line of the measured arm carries every required key with a
sane value, and the reference arm (CPU) prints one JSON line with the same metric / unit and the e2e / cpu_baseline objects."""
import json
import os
import subprocess
import sys

import glob

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _latest_bench_line():
    """the newest committed 1-GPU bench line (profiles/rNN_bench_fast_mode.json)"""
    return json.load(open(sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_bench_fast_mode.json")))[-1]))


def _check_common(d):
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and d["e2e"]["unit"] == d["unit"]
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and d["cpu_baseline"]["kind"] in ("port", "reference")


def test_committed_bench_line_has_the_contract_keys():
    d = _latest_bench_line()
    _check_common(d)
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["dtype"] == "bf16" and d["gpu_launches"] > 0
    assert abs(d["value"] - 1024 * 1024 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 2 * 1024 * 256 * 3 * 4 and d["e2e"]["d2h_bytes_per_step"] == 1024 * 1024 * 4
    r = d["roofline"]
    assert set(r) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and r["bound"] in ("hbm", "tensor")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
    c = d["clocks"]
    assert set(c) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"])
    assert "l2" in d["config"]                      # says how L2 reuse between timed iterations is ruled out


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    _check_common(d)
    assert d["impl"] == "reference" and d["dtype"] == "f32"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    ours = _latest_bench_line()
    assert d["metric"] == ours["metric"] and d["unit"] == ours["unit"]


def test_dump_outputs_samples_rows_beyond_the_budget(tmp_path, monkeypatch):
    """score rows over a rank's share of the byte budget are cut to the same seeded row sample on every run"""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    budget = 2 * (10 * (4 * 32 + 8) + 2 * 128)          # two ranks, room for ten rows and two .npy headers each
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    rows = torch.arange(100 * 32, dtype=torch.float32).reshape(100, 32)
    for run in ("a", "b"):
        bench.dump_scores(str(tmp_path / run), rows, 1, 2)
    idx = np.load(tmp_path / "a" / "scores_rank1_rows.npy")
    s = np.load(tmp_path / "a" / "scores_rank1.npy")
    assert idx.dtype == np.float64 and idx.shape == (10,) and (np.diff(idx) > 0).all()
    assert s.dtype == np.float32 and np.array_equal(s, rows.numpy()[idx.astype(np.int64)])
    assert np.array_equal(idx, np.load(tmp_path / "b" / "scores_rank1_rows.npy"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget // 2


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_steps_scores(tmp_path):
    """--dump-outputs writes the score rows the timed path returned, and they are what the public API computes on the same seeded
    inputs in another process; --steps sets the number of timed steps"""
    import numpy as np
    from pcreid_b200.parallel import match_all_pairs_sharded
    sys.path.insert(0, ROOT)
    import bench
    T, D = 64, 48
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--tracks", str(T),
                          "--dets", str(D), "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3 and len(line["per_step_ms"]) == 3
    assert sorted(os.listdir(tmp_path)) == ["scores_rank0.npy"]
    got = np.load(tmp_path / "scores_rank0.npy")
    assert got.dtype == np.float32 and got.shape == (T, D) and np.isfinite(got).all()
    cfg = bench.CONFIGS["c2"]                  # bench.py's defaults: the headline configuration and mode
    model = bench.bench_model(cfg, "parity_tc", "cuda")
    t, d = bench.bench_inputs(cfg["npts"], T, D)
    rows = match_all_pairs_sharded(model, t.cuda(), d.cuda(), [D])
    assert np.array_equal(got, rows.cpu().numpy())
