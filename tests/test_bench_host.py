"""bench.py's host-side safety net (no GPU): child processes with deadlines, the reference arm's JSON line."""
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def test_run_child_returns_output_and_kills_the_whole_group_on_timeout(tmp_path):
    import bench
    rc, out, err = bench._run_child([sys.executable, "-c", "import sys; print('hello'); print('oops', file=sys.stderr); sys.exit(3)"], 30)
    assert (rc, out.strip(), err.strip()) == (3, "hello", "oops")
    pidfile = tmp_path / "grandchild.pid"
    code = ("import os, time\n"
            "pid = os.fork()\n"
            "if pid == 0:\n"
            "    time.sleep(120)\n"
            f"open({str(pidfile)!r}, 'w').write(str(pid))\n"
            "time.sleep(120)\n")
    t0 = time.time()
    with pytest.raises(subprocess.TimeoutExpired):
        bench._run_child([sys.executable, "-c", code], 2)
    assert time.time() - t0 < 30
    grandchild = int(pidfile.read_text())
    for _ in range(50):                       # (the kernel needs a moment to reap it)
        try:
            os.kill(grandchild, 0)
        except ProcessLookupError:
            break
        time.sleep(0.1)
    else:
        # still in the process table: it must at least be a zombie of a killed process, not a sleeper
        state = Path(f"/proc/{grandchild}/stat").read_text().split()[2]
        assert state == "Z", state


def test_cpu_baseline_child_reports_a_missed_deadline_instead_of_stalling():
    import bench
    t0 = time.time()
    r = bench.cpu_baseline_child(timeout_s=0.2, attempts=1)
    assert time.time() - t0 < 30
    assert r["value"] is None and "no result within" in r["unavailable"] and r["unit"] == bench.UNIT


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    """`bench.py --impl reference` (the reference's own CPU path through a child process with a deadline): one JSON line."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "bar_strategy_evals_per_sec" and line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    # a rank other than 0 of a multi-process launch does no work and prints nothing
    r2 = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2"], stdout=subprocess.PIPE,
                        stderr=subprocess.PIPE, text=True, timeout=120, cwd=str(ROOT), env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r2.returncode == 0 and r2.stdout.strip() == ""


def test_claimed_stdout_carries_only_the_result_line():
    """bench._claim_stdout: whatever the process (or a C library) prints to fd 1 afterwards lands on stderr."""
    code = ("import os, sys, json; sys.path.insert(0, %r); import bench\n"
            "fd = bench._claim_stdout()\n"
            "print('a python print'); os.system('echo a child of the shell')\n"
            "os.write(1, b'a C library writing to fd 1\\n')\n"
            "os.write(fd, (json.dumps({'value': 1}) + '\\n').encode())\n") % str(ROOT)
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout == '{"value": 1}\n'
    for s in ("a python print", "a child of the shell", "a C library writing to fd 1"):
        assert s in r.stderr


def test_dump_outputs_writes_float64_arrays_and_samples_above_the_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every array float64 and finite (inf / nan coded beside the array), trade_hash exact through
    its two halves, a seeded sample above the cap."""
    import numpy as np
    import bench
    rng = np.random.default_rng(1)
    pop, S = 300, 3
    fitness = rng.normal(size=pop)
    sortino = rng.normal(size=(pop, S))
    sortino[0, 0], sortino[5, 2], sortino[7, 1] = np.inf, -np.inf, np.nan
    stats = {"score": rng.normal(size=(pop, S)), "sortino_ratio": sortino,
             "trade_hash": rng.integers(0, 2**64, size=(pop, S), dtype=np.uint64)}
    bench.dump_outputs(str(tmp_path / "all"), fitness, stats)
    got = {p.stem: np.load(p) for p in (tmp_path / "all").glob("*.npy")}
    assert set(got) == {"fitness", "score", "sortino_ratio", "sortino_ratio_nonfinite", "trade_hash_hi", "trade_hash_lo"}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in got.values())
    assert np.array_equal(got["fitness"], fitness) and np.array_equal(got["score"], stats["score"])
    code = got["sortino_ratio_nonfinite"]
    assert (code[0, 0], code[5, 2], code[7, 1]) == (1.0, -1.0, 2.0) and np.count_nonzero(code) == 3
    finite = np.isfinite(sortino)
    assert np.array_equal(got["sortino_ratio"][finite], sortino[finite]) and not got["sortino_ratio"][~finite].any()
    hashes = (got["trade_hash_hi"].astype(np.uint64) << np.uint64(32)) | got["trade_hash_lo"].astype(np.uint64)
    assert np.array_equal(hashes, stats["trade_hash"])
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8 * (1 + 1 + 5 * S) * 100)        # room for 100 of the 300 individuals
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), fitness, stats)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    b = {p.stem: np.load(p) for p in (tmp_path / "b").glob("*.npy")}
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_LIMIT_BYTES
    idx = a["lane_index"].astype(np.int64)
    assert len(idx) == 100 and np.array_equal(a["fitness"], fitness[idx]) and np.array_equal(a["score"], stats["score"][idx])
    assert all(np.isfinite(x).all() for x in a.values())
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
