"""bench.py's reference arm runs on the CPU alone (the oracle's OpenMP port of SUBSEG_MATCH), so its
side of the driver contract can be held here: one JSON line with the contract's keys, hermetic (the
product library is not loaded), and a `config` object that is the one the product arm prints."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_reference(*extra, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", *extra], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines          # ONE JSON line
    return json.loads(lines[0])


@pytest.mark.parametrize("workload", ["config1", "dictionary"])
def test_reference_arm_line(workload):
    import bench
    line = run_reference("--workload", workload)
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "input GB/s matched" and line["unit"] == "GB/s"
    assert line["steps"] == 2 and line["warmup"] == 1 and line["higher_is_better"] is True
    assert line["vs_baseline"] is None and line["dtype"] == "u8" and line["gpu_launches"] == 0
    assert line["value"] > 0 and abs(line["ms_per_step"] * 1e-3 * line["value"] * 1e9 - 1048575) < 1048575 * 1e-6
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "1048575 bytes" in cb["sample"]
    # the config object is shared_config's: what the product arm prints for the same command line
    args = SimpleNamespace(scaling="weak", bytes=0, streams=4)
    _, desc, nbytes, fixture, _ = bench.workload_patterns(workload)
    assert line["config"] == bench.shared_config(args, desc, nbytes, fixture, 1)
    assert line["config"]["bytes_per_gpu"] == 1048575 and "written between" in line["config"]["l2"]


def test_reference_arm_other_ranks_print_nothing():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "config1",
                        "--gpus", "2", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs(tmp_path, monkeypatch):
    """--dump-outputs: float64 arrays, every record up to DUMP_MAX_RECORDS, a fixed sample beyond (the same on every
    run), under 64 MB at the largest sample."""
    import numpy as np
    import bench
    rec = np.array([[5, 3], [-1, 7], [1 << 30, 10000]], dtype=np.int32)
    bench.dump_outputs(tmp_path / "small", rec)
    got = {n: np.load(tmp_path / "small" / f"{n}.npy") for n in ("count", "rows", "pos", "id")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["count"].tolist() == [3] and got["rows"].tolist() == [0, 1, 2]
    assert got["pos"].tolist() == [5, 2 ** 32 - 1, 1 << 30] and got["id"].tolist() == [3, 7, 10000]
    big = np.random.default_rng(1).integers(0, 1 << 31, (bench.DUMP_MAX_RECORDS + 1, 2)).astype(np.int32)
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, big)
    files = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert len(rows) == bench.DUMP_MAX_RECORDS and (np.diff(rows) > 0).all()
    assert np.array_equal(np.load(tmp_path / "a" / "pos.npy"), big[rows, 0].astype(np.float64))
    assert np.load(tmp_path / "a" / "count.npy").tolist() == [bench.DUMP_MAX_RECORDS + 1]


def test_shared_config_is_a_function_of_the_command_line():
    import bench
    a = SimpleNamespace(scaling="weak", bytes=0, streams=4)
    c = bench.shared_config(a, "w", 1 << 30, None, 8)
    assert c["bytes_per_gpu"] == 1 << 30 and c["total_bytes"] == 8 << 30 and "exceeds" in c["l2"]
    s = SimpleNamespace(scaling="strong", bytes=0, streams=4)
    c = bench.shared_config(s, "w", 1 << 30, None, 8)
    assert c["bytes_per_gpu"] == 128 << 20 and c["total_bytes"] == 1 << 30 and "rotate" in c["l2"]
    # strong scaling's shard 0 follows pfac_job_plan (64 KiB granularity)
    import phfpfac_b200 as pf
    for total, world in ((1 << 30, 3), (1000003, 4), (65536, 8), (5 << 20, 2)):
        s = SimpleNamespace(scaling="strong", bytes=total, streams=4)
        assert bench.shared_config(s, "w", 0, None, world)["bytes_per_gpu"] == pf.plan_shard(total, world, 16, 0)[1]
    # fixtures are never cut (they are scanned whole on every rank)
    assert bench.shared_config(s, "w", 1048575, b"x", 2)["total_bytes"] == 2 * (5 << 20)
