"""Host logic of bench.py's CPU arm (no GPU, no oracle): the thread count the reference arm gives the oracle.
Round 1's `--impl reference` arm was 3.8x slower than the cpu_baseline leg of the same box (cgroup CPU quota), and a
later version came out single-threaded on hosts WITHOUT a quota (OMP_PROC_BIND narrows the affinity mask of the calling
thread once libgomp is loaded): both are pinned here. Also the files --dump-outputs writes (host logic, and one small
bench.py run on the GPU whose dumped solutions are checked against the regenerated inputs)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class FakeBatch:
    def __init__(self, seconds_by_threads):
        self.t = seconds_by_threads
        self.calls = []

    def solve(self, threads):
        self.calls.append(threads)
        return self.t[threads]


def test_host_thread_count_is_read_once(monkeypatch):
    import bench

    h = bench.host_threads()
    assert h >= 1
    monkeypatch.setattr(os, "sched_getaffinity", lambda pid: {0}, raising=False)  # what libgomp's binding leaves behind
    assert bench.host_threads() == h
    cands = bench.thread_candidates()
    assert h in cands and max(1, h // 2) in cands


def test_thread_choice_uses_sustained_time_and_respects_the_quota(monkeypatch):
    import bench

    t = {16: 0.110, 32: 0.105, 64: 0.174, 128: 0.150}
    monkeypatch.setattr(bench, "cpu_quota", lambda: 16.0)
    best, tried = bench.best_thread_count(FakeBatch(t), [128, 64, 32, 16])
    assert best == 16 and set(tried) == set(t)  # 32 threads are 4.5 % faster: not enough to leave the quota's count
    best, _ = bench.best_thread_count(FakeBatch({**t, 32: 0.090}), [128, 64, 32, 16])
    assert best == 32  # 18 % faster: taken
    monkeypatch.setattr(bench, "cpu_quota", lambda: None)
    best, _ = bench.best_thread_count(FakeBatch(t), [128, 64, 32, 16])
    assert best == 32  # no quota: ties within 3 % go to fewer threads, 4.5 % is a win
    best, _ = bench.best_thread_count(FakeBatch({64: 0.100, 128: 0.099}), [128, 64])
    assert best == 64


def fake_results(B, rng):
    info = {"iter": rng.integers(0, 50, B), "status": np.zeros(B, dtype=np.int64), "pri_res": rng.random(B), "solve_time": rng.random(B)}
    return dict(x=rng.random((B, 5)), y=rng.random((B, 2)), z=rng.random((B, 3)), se=rng.random((B, 2)), si=rng.random((B, 3)), info=info)


def test_dump_outputs_writes_float64_arrays_and_a_fixed_sample_above_the_cap(tmp_path, monkeypatch):
    import bench

    res = fake_results(40, np.random.default_rng(1))
    bench.dump_outputs(str(tmp_path / "all"), res, 100)
    names = sorted(p.name for p in (tmp_path / "all").iterdir())
    assert names == sorted(["x.npy", "y.npy", "z.npy", "se.npy", "si.npy", "info_iter.npy", "info_status.npy", "info_pri_res.npy", "qp_index.npy"])
    for n in names:
        assert np.load(tmp_path / "all" / n).dtype == np.float64
    assert np.array_equal(np.load(tmp_path / "all" / "x.npy"), res["x"])
    assert np.array_equal(np.load(tmp_path / "all" / "qp_index.npy"), 100 + np.arange(40))

    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * 19 * 10)  # 19 values per row: room for 10 of the 40 rows
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res, 0)
    idx = np.load(tmp_path / "a" / "qp_index.npy").astype(np.int64)
    assert len(idx) == 10 and np.all(np.diff(idx) > 0)
    assert sum(p.stat().st_size - 128 for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES  # (128-byte .npy header)
    assert np.array_equal(np.load(tmp_path / "a" / "x.npy"), res["x"][idx])
    for n in names:
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n))


@pytest.mark.gpu
def test_bench_dumps_the_solutions_of_its_last_timed_step(tmp_path):
    import bench
    from helpers import kkt_residuals
    from proxsuite_b200 import proxqp

    B = 16
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", str(B), "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["value"] > 0
    out = {n[:-4]: np.load(tmp_path / n) for n in os.listdir(tmp_path)}
    assert np.array_equal(out["qp_index"], np.arange(B)) and (out["info_status"] == 0).all()
    st = bench.generate(0, B, proxqp.dense.random_qp)
    for i in range(B):
        pri, dua = kkt_residuals({k: st[k][i] for k in bench.KEYS}, out["x"][i], out["y"][i], out["z"][i])
        assert pri <= bench.EPS_ABS and dua <= bench.EPS_ABS, (i, pri, dua)
