"""bench.py's reference arm (`--impl reference`): the JSON line the driver parses, produced here on the CPU -- the unmodified
reference (oracle/_ref, compiled from the reference's sources by oracle/Makefile) or, where it was not built, the oracle port, on the same
synthetic slots as the CUDA arm.  No GPU and nothing of libft8b200 is involved in this arm (bench.py:reference_arm)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.pop("RANK", None); env.pop("WORLD_SIZE", None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", *args],
                          capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    p = _run()
    assert p.returncode == 0, p.stderr[-800:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must carry the JSON line only"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and "unavailable" not in d
    assert d["metric"].startswith("FT8 15s-slots decoded/sec") and d["unit"] == "slots/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["vs_baseline"] is None and d["scaling"] == "weak" and d["data"].startswith("synthetic")
    assert set(d["config"]) >= {"workload", "slots_per_gpu_per_step", "max_candidates", "max_messages", "ldpc_iterations"} and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    from oracle.pyoracle import reference_dir
    if os.path.isfile(os.path.join(reference_dir(), "rtlsdr_ft8d.c")):   # build() compiles the unmodified reference from there: it is what is timed
        assert cb["kind"] == "reference"


def test_reference_arm_runs_on_rank_0_only():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29577"}, ("--gpus", "2"))
    assert p.returncode == 0 and p.stdout.strip() == "", (p.stdout[-200:], p.stderr[-400:])


def test_steps_and_dump_outputs_arguments_are_checked():
    assert "--steps must be at least 1" in _run(args=("--steps", "0")).stderr
    assert "--dump-outputs applies to the CUDA arm" in _run(args=("--dump-outputs", "x")).stderr


def test_dump_outputs_writes_the_records_a_caller_receives(tmp_path, monkeypatch):
    """bench.dump_outputs: float arrays only, records past a slot's count zeroed, and a fixed sample of slots above the size cap."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle.pyoracle import result_dtype
    res = np.zeros((6, 50), result_dtype)
    res["call"], res["loc"], res["freq"], res["snr"] = b"K1JT", b"FN20", 1234, -7
    nres = np.array([0, 1, 2, 50, -1, 3], np.int32)
    bench.dump_outputs(str(tmp_path / "all"), res, nres, result_dtype)
    d = {n: np.load(tmp_path / "all" / (n + ".npy")) for n in ("slot_index", "n_results", "freq", "snr", "call", "loc")}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert np.array_equal(d["slot_index"], np.arange(6)) and np.array_equal(d["n_results"], nres)
    valid = np.arange(50)[None, :] < nres[:, None]
    assert np.array_equal(d["freq"], np.where(valid, 1234.0, 0.0)) and np.array_equal(d["snr"], np.where(valid, -7.0, 0.0))
    assert d["call"].shape == (6, 50, 13) and bytes(d["call"][3, 49].astype(np.uint8)).rstrip(b"\0") == b"K1JT"
    assert not d["call"][0].any() and not d["loc"][4].any() and bytes(d["loc"][5, 2].astype(np.uint8)).rstrip(b"\0") == b"FN20"
    per_slot = 50 * (8 + 8 + 4 * (13 + 7)) + 16
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 3 * per_slot + 6 * bench.DUMP_HEADER_BYTES + 100)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), res, nres, result_dtype)
    idx = np.load(tmp_path / "a" / "slot_index.npy")
    assert idx.size == 3 and np.array_equal(idx, np.load(tmp_path / "b" / "slot_index.npy"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_MAX_BYTES
