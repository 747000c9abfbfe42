"""bench.py's host-side helpers (no GPU): byte counts of SURVEY 8(d), the clock-sampler parser, the keep-load step
count (identical on every rank by construction), and that --impl reference on a non-zero rank does no work."""
import importlib.util
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_algorithmic_byte_counts_follow_survey_8d():
    b = _bench()
    n, nnz, d = 69716, 2474518, 64  # yelp2018 shape: N = U + I, nnzA = 2 * nnz
    S = 8 * nnz + 4 * (n + 1) + 8 * n * d
    assert b.spmm_bytes(n, nnz, d) == S == 55769604          # the figure of the bench line
    assert b.step_bytes("XSimGCL", n, nnz, d, 3) == 2 * 3 * S + 28 * n * d == 459548696
    assert b.step_bytes("LightGCN", n, nnz, d, 3) == b.step_bytes("XSimGCL", n, nnz, d, 3)
    assert b.step_bytes("SimGCL", n, nnz, d, 3) == 6 * 3 * S + 28 * n * d
    assert b.step_bytes("SGL", n, nnz, d, 3, view_nnz=nnz - 1000) == 2 * 3 * S + 4 * 3 * b.spmm_bytes(n, nnz - 1000, d) + 28 * n * d


def test_keep_load_step_count_depends_only_on_the_step_time():
    b = _bench()
    fake = types.SimpleNamespace(cuda=types.SimpleNamespace(synchronize=lambda: None))
    for ms, want in ((0.33, 1212), (0.5, 800), (40.0, 50), (1e-9, 20000)):
        calls = []
        b.keep_load(calls.append, ms, fake)
        assert len(calls) == want and calls == list(range(want))


def test_clock_sampler_parses_nvidia_smi_rows(tmp_path):
    b = _bench()
    cs = b.ClockSampler(0)
    rows = ["0, 1965, 1965, 400.1, 0x0, Not Active, Not Active, Not Active, Not Active",
            "0, 1950, 1965, 950.0, 0x4, Not Active, Not Active, Not Active, Active",
            "garbage"]
    p = tmp_path / "smi.csv"
    p.write_text("\n".join(rows) + "\n")
    cs.path = str(p)
    cs.proc = types.SimpleNamespace(terminate=lambda: None, wait=lambda timeout=None: 0, kill=lambda: None)
    out = cs.stop()
    assert out["sm_mhz"] == 1957.5 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"] and out["samples"] == 2
    assert b.ClockSampler(0).stop()["reasons"] == ["nvidia-smi unavailable"]  # never started: still a dict


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_peaks_come_from_the_driver_file_when_present():
    b = _bench()
    pk = b.peaks()
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            assert pk["hbm_gbs"] == float(json.load(f)["hbm_gbs"]) and pk["source"].startswith("measured")
    else:
        assert pk["source"].startswith("fallback")


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    import numpy as np
    import pytest
    b = _bench()
    arrays = {"emb": np.arange(12, dtype=np.float32).reshape(3, 4), "losses": np.array([0.5, 1.5], dtype=np.float64)}
    b.dump_outputs(str(tmp_path / "out"), arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "out" / f"{k}.npy")
        assert got.dtype == v.dtype and np.array_equal(got, v)
    with pytest.raises(ValueError):
        b.dump_outputs(str(tmp_path / "int"), {"ids": np.arange(4, dtype=np.int32)})
    with pytest.raises(ValueError):
        b.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(b.DUMP_LIMIT_BYTES // 4 + 1, dtype=np.float32)})
    assert not (tmp_path / "int").exists() and not (tmp_path / "big").exists()


def test_dump_outputs_is_refused_where_there_is_no_single_gpu_timed_path(tmp_path):
    for extra, env in ((["--impl", "reference"], {}), (["--profile"], {}), ([], dict(RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path)] + extra,
                           capture_output=True, text=True, env=dict(os.environ, **env), timeout=120)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr and r.stdout == ""
