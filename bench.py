#!/usr/bin/env python
"""bench.py — QPs solved per second on batched dense ProxQP (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (GPU arm, this repo)
    python bench.py --impl reference --gpus N --steps K ...  (CPU arm: the reference's
                                                              algorithm on the host cores)

Workload (the shape BASELINE.json's metric and the north-star target are quoted on: configs[1]'s QP shape at the
headline batch of 4096): per GPU a BatchQP of 4096 random dense QPs,
n=100, n_eq=50, n_in=100, fp64, generated exactly like the reference's batch
benchmark (benchmark/timings-parallel.cpp:19-54: set_seed(i) +
dense_strongly_convex_qp(sparsity 0.15, strong convexity 1e-2), eps_abs=1e-9,
eps_rel=0, NO_INITIAL_GUESS). A "step" is one solve_in_parallel over the whole
(already init-ed) batch — what timings-parallel.cpp:208-232 times. Weak scaling:
every rank owns its own 4096 QPs (--batch 1024 gives configs[1]'s literal batch), no collective in the data path.

`value`   : QPs/s with inputs resident in HBM, CUDA-event timed on the launching stream.
`e2e`     : QPs/s through the public API with HOST (pinned) inputs, every step: init (chunked H2D
            upload, a progress word behind each chunk) + solve (ONE persistent kernel that waits
            for each QP's inputs, runs its Ruiz equilibration and solves it) + D2H of x, y, z,
            se, si, info. PQP_E2E=plain|chunks selects the older separate-launch pipelines.
`roofline`: algorithmic bytes (SURVEY.md section 8(d)(ii) streamed-operand model,
            evaluated from the oracle's operation counters on a sample of the
            same workload) / measured solve-kernel time, against the measured
            HBM peak of MEASURED_PEAKS.json.

--dump-outputs DIR writes the results of the last timed device-resident step (rank 0's batch) as DIR/<name>.npy, so
that two builds can be compared output for output on the same seeded inputs (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DIM, N_EQ, N_IN = 100, 50, 100
BATCH_PER_GPU = 4096  # headline batch (north_star: 4096 QPs on 1 GPU); configs[1]'s literal batch is --batch 1024
CPU_SAMPLE = 1024     # QPs per CPU-arm step (a bounded sample of the same workload: seeds 0..1023)
SPARSITY, STRONG_CONVEXITY = 0.15, 1e-2
EPS_ABS = 1e-9
KEYS = "HgAbClu"
DUMP_BYTES = 64 << 20  # cap of --dump-outputs


def algorithmic_bytes_per_qp(cnt, n, ne, ni, ncons, batch):
    """SURVEY.md section 8(d)(ii): bytes of the operands each executed primitive
    streams, from the oracle's counters (mean per QP)."""
    nnzH = n * n
    c = {k: v / batch for k, v in cnt.items()}
    b = 8.0 * c["factor_m2"]
    b += 8.0 * (c["solve_m2"] + 4.0 * c["solve_m"])
    b += 8.0 * (c["n_resid"] * (nnzH + 2 * ne * n) + n * c["resid_nc"] + 6.0 * c["solve_m"])
    b += 16.0 * c["rank_chunk_t2"] + 16.0 * c["rank_rt"]
    b += c["insert_bytes"]
    b += 8.0 * c["delete_t2"]
    b += c["n_cdx"] * 16.0 * ni * n
    b += c["n_global_res"] * 8.0 * (nnzH + 2 * ne * n + 2 * ni * n)
    b += 8.0 * c["ls_evals"] * (2 * n + 2 * ne + 5 * ncons)
    return b


def compulsory_bytes_per_qp(n, ne, ni):
    """SURVEY.md section 8(d)(i): inputs read once + solution written once."""
    return 8.0 * (n * n + ne * n + ni * n + n + ne + 2 * ni) + 8.0 * (n + ne + ni)


def generate(first, count, gen):
    data = [gen("strongly_convex", first + i, N_DIM, N_EQ, N_IN, SPARSITY, STRONG_CONVEXITY) for i in range(count)]
    return {k: np.stack([d[k] for d in data]) for k in KEYS}


def dump_outputs(out_dir, res, first):
    """Write DenseBatch.results() as float64 .npy files: x, y, z, se, si [B, *] and one info_<field> [B] per pqp_info
    field except the wall-clock *_time ones, plus qp_index [B] (the seed of each row's QP). Above DUMP_BYTES the rows
    are a fixed sample of the batch (numpy seed 0, sorted), the same for every run with the same --batch."""
    arrays = {k: res[k] for k in ("x", "y", "z", "se", "si")}
    arrays.update({"info_" + k: v for k, v in res["info"].items() if not k.endswith("_time")})
    B = len(res["x"])
    row_bytes = 8 * (1 + sum(a.size for a in arrays.values()) // B)
    keep = min(B, DUMP_BYTES // row_bytes)
    rows = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    arrays["qp_index"] = first + np.arange(B)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(np.asarray(v, dtype=np.float64)[rows]))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            p = [x.strip() for x in s.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


_HOST_THREADS = None


def host_threads():
    """Every host thread this process may use. torchrun exports OMP_NUM_THREADS=1 to its
    workers; the CPU arm must not inherit that, so the count is passed explicitly. Read ONCE, at the first call (module
    import): with OMP_PROC_BIND=true libgomp binds the calling thread to one place when it loads, after which
    sched_getaffinity(0) says 1 - a later call would then make the CPU arm single-threaded on a host without a quota."""
    global _HOST_THREADS
    if _HOST_THREADS is None:
        try:
            _HOST_THREADS = max(1, len(os.sched_getaffinity(0)))
        except AttributeError:
            _HOST_THREADS = max(1, os.cpu_count() or 1)
    return _HOST_THREADS


def cpu_quota():
    """CPUs' worth of time the cgroup lets this process use per period (cpu.max: "quota period"), or None.
    The pool's GPU boxes show 128 logical CPUs in the affinity mask but a quota of 16: every thread beyond the quota only
    burns it faster, and CFS then stops ALL threads until the next 100 ms period - which is what made round 1's
    `--impl reference` arm 3.8x slower than the cpu_baseline leg of the same box (step times in multiples of 100 ms)."""
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            q, per = open(path).read().split()[:2]
            if q != "max":
                return float(q) / float(per)
        except (OSError, ValueError):
            pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / per
    except (OSError, ValueError):
        pass
    return None


def thread_candidates():
    """Thread counts worth trying for the CPU arm: every logical CPU, half of them (the reference's default,
    parallel/qp_solve.hpp:45-49), and - under a cgroup CPU quota - the quota and twice the quota."""
    H = host_threads()
    c = {H, max(1, H // 2)}
    q = cpu_quota()
    if q:
        c |= {max(1, min(H, int(q + 0.999))), max(1, min(H, 2 * int(q + 0.999)))}
    return sorted(c, reverse=True)


host_threads()  # (pinned down before any OpenMP runtime can narrow the affinity mask of this thread)


def gpu_numa_cpus(index):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None. Pinned host buffers are first-touched by this process: on
    the pool's two-socket boxes a buffer that lands on the far socket uploads at 15-25 GB/s instead of ~50."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        bdf = out.lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        return (node, cpus) if cpus else None
    except Exception:
        return None


def pin_openmp_env(threads):
    """OpenMP environment of the CPU arm, set BEFORE libgomp is loaded (it reads the environment once): one thread per
    logical CPU, no migration, spinning workers. torchrun / the driver may export OMP_NUM_THREADS=1; the CPU arm must not
    inherit that."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ["OMP_DYNAMIC"] = "false"
    os.environ.pop("OMP_THREAD_LIMIT", None)
    if cpu_quota() is None:  # (under a quota fewer threads than CPUs run: let the kernel place them; spinning would burn quota)
        os.environ["OMP_PROC_BIND"] = "true"
        os.environ["OMP_PLACES"] = "threads"
        os.environ["OMP_WAIT_POLICY"] = "active"
    else:
        os.environ["OMP_WAIT_POLICY"] = "passive"


def make_oracle_batch(sample):
    """`sample` QPs of the workload (seeds 0..sample-1) set up in the oracle (C++ restatement of the reference, kind
    "port", rebuilt with -march=native on this machine), ready for solve_in_parallel."""
    from oracle import oracle as O

    flags = O.use_native()
    st = generate(0, sample, O.generate_qp)
    b = O.OracleBatch(sample, N_DIM, N_EQ, N_IN)
    for i in range(sample):
        q = b[i]
        q.set(eps_abs=EPS_ABS, eps_rel=0, initial_guess=O.NO_INITIAL_GUESS)
        q.init(**{k: st[k][i] for k in KEYS})
    return b, flags


def best_thread_count(batch, candidates):
    """The CPU arm gets the thread count that serves it best on this host: every logical CPU, or
    half of them (the reference's own default, parallel/qp_solve.hpp:45-49; SMT siblings can hurt), or - under a cgroup
    quota - the quota. Judged on the SUSTAINED time of four back-to-back solves after one untimed solve, not on the best of
    them: under a CFS quota an over-subscribed run fits one solve into a fresh 100 ms period now and then (best-of-three said
    106 ms for 128 threads on a 16-CPU quota) while its steady state is twice that (the timed steps then took 195-199 ms).
    Ties within 3 % go to the smaller thread count (fewer threads = less quota burnt by spinning / waking)."""
    best_t, best_time, tried = None, None, {}
    q = cpu_quota()
    for t in sorted(candidates):
        batch.solve(t)
        dt = sum(batch.solve(t) for _ in range(4)) / 4
        tried[t] = dt
        # more threads than the quota's CPUs must win by 10 % to be taken: they run into the throttle now and then (one
        # 165 ms step among 110 ms ones with 32 threads on a 16-CPU quota), the quota's own count does not
        margin = 0.90 if (q and best_t is not None and t > int(q + 0.999) >= best_t) else 0.97
        if best_time is None or dt < margin * best_time:
            best_t, best_time = t, dt
    return best_t, tried


def cpu_baseline(sample, reps, threads=0):
    """The oracle on the host cores: OpenMP schedule(dynamic) over QPs with all threads, batch already
    init-ed (benchmark/timings-parallel.cpp:208-232)."""
    b, flags = make_oracle_batch(sample)
    H = host_threads()
    tried = {}
    if threads:
        T = threads
    else:
        T, tried = best_thread_count(b, thread_candidates())
    b.solve(T)  # warm-up
    b.counters(reset=True)
    times = [b.solve(T) for _ in range(reps)]
    cnt = b.counters()
    cnt = {k: v / reps for k, v in cnt.items()}
    solved = sum(1 for i in range(sample) if b[i].results().info.status == 0)
    return dict(qps=sample / min(times), best_s=min(times), total_s=sum(times), times=times, cores=T, host_threads=H, tried=tried, sample=sample,
                reps=reps, solved=solved, counters=cnt, flags=flags)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path. The reference itself cannot be
    compiled here (Eigen 3 absent, DESIGN.md section 6), so this is the oracle
    port (rebuilt with -march=native on this machine) with every host thread; rank 0 alone runs.
    Each step = solve_in_parallel over a CPU_SAMPLE-QP sample of the workload; `value` = QPs of the K timed
    steps / their total time. Per-step times, the thread count tried / chosen and the load average are printed
    so that an outlier run can be recognised (`steps_ms`, `threads_tried_ms`, `loadavg`)."""
    if rank != 0:
        return
    sample = CPU_SAMPLE
    H = host_threads()
    pin_openmp_env(H)
    b, flags = make_oracle_batch(sample)
    T, tried = best_thread_count(b, thread_candidates())
    for _ in range(max(args.warmup, 3)):
        b.solve(T)
    times = [b.solve(T) for _ in range(args.steps)]  # orc_batch_solve returns the wall time of the parallel region
    dt = sum(times)
    qps = sample * args.steps / dt
    try:
        load = os.getloadavg()[0]
    except OSError:
        load = None
    line = {
        "impl": "reference", "metric": "QPs solved/sec (batch dense, n=100)", "value": qps, "unit": "QPs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"BatchQP dense n={N_DIM} n_eq={N_EQ} n_in={N_IN} eps_abs=1e-9 NO_INITIAL_GUESS; step = solve_in_parallel over a {sample}-QP sample (seeds 0..{sample - 1}) of the {BATCH_PER_GPU}-QP batch, OpenMP schedule(dynamic)",
                   "batch_per_step": sample, "compiler_flags": flags},
        "cpu_baseline": {"value": qps, "unit": "QPs/s", "cores": T, "kind": "port", "sample": f"{sample} QPs x {args.steps} steps, seeds 0..{sample - 1}"},
        "e2e": {"value": qps, "unit": "QPs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "steps_ms": [round(1e3 * t, 2) for t in times], "best_step_qps": sample / min(times), "host_threads": H,
        "threads_tried_ms": {str(k): round(1e3 * v, 2) for k, v in tried.items()}, "loadavg": load, "cgroup_cpu_quota": cpu_quota(),
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="QPs per GPU (default 4096, the north-star batch; BASELINE.json configs[1] literally: 1024)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed device-resident step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; proxsuite_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    from proxsuite_b200 import proxqp

    B = args.batch
    n, ne, ni = N_DIM, N_EQ, N_IN
    # synthetic inputs of this rank (seeds rank*B .. rank*B+B-1), in pinned host memory allocated on the GPU's NUMA node
    full_mask = os.sched_getaffinity(0)
    numa = None if os.environ.get("BENCH_NO_NUMA") == "1" else gpu_numa_cpus(local_rank)  # (BENCH_NO_NUMA=1: A/B hook)
    if numa:
        os.sched_setaffinity(0, numa[1])
    host = generate(rank * B, B, proxqp.dense.random_qp)
    pinned = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
    host = {k: v.numpy() for k, v in pinned.items()}
    h2d_bytes = sum(v.nbytes for v in host.values())

    db = proxqp.dense.DenseBatch(B, n, ne, ni, device=local_rank)
    db.settings.eps_abs = EPS_ABS
    db.settings.eps_rel = 0
    db.settings.initial_guess = proxqp.InitialGuess.NO_INITIAL_GUESS
    db.init(**host)
    db.solve()
    chk = db.results()
    assert (chk["info"]["status"] == 0).all(), "not every QP was solved"
    x = chk["x"]
    cx = np.einsum("bij,bj->bi", host["C"], x)
    pri = max(np.abs(np.einsum("bij,bj->bi", host["A"], x) - host["b"]).max(), np.abs(np.maximum(cx - host["u"], 0) + np.minimum(cx - host["l"], 0)).max())
    dua = np.abs(np.einsum("bij,bj->bi", host["H"], x) + host["g"] + np.einsum("bji,bj->bi", host["A"], chk["y"]) + np.einsum("bji,bj->bi", host["C"], chk["z"])).max()
    assert pri <= 1e-9 and dua <= 1e-9, (pri, dua)

    # a dedicated non-default stream: kernels, memsets and the timing events
    # all go to THIS stream (handle 0 would select the batch's own stream)
    stream = torch.cuda.Stream()
    assert stream.cuda_stream != 0

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident throughput ("value") --------------------------------
    for _ in range(args.warmup):
        db.solve_async(stream.cuda_stream)
    db.sync()
    launches0 = db.timings()["kernel_launches"]
    sampler = ClockSampler(local_rank)
    sync_all()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        db.solve_async(stream.cuda_stream)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    db.sync()
    outputs = db.results() if args.dump_outputs and rank == 0 else None  # the last timed step's results
    launches = db.timings()["kernel_launches"] - launches0
    kernel_ms = db.timings()["solve_ms"]  # last solve kernel alone (events around the launch)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * args.steps / (ms_max * 1e-3)

    # ---- end to end through the public API ("e2e") ---------------------------
    gathered = torch.empty((world * B, n + ne + ni + 20), dtype=torch.float64, device="cuda") if world > 1 else None

    def e2e_step():
        db.init(**host)          # H2D from pinned memory (chunked, progress words); the set-up is fused into the solve kernel
        db.solve()               # persistent solve kernel
        if world > 1:            # the one exchange step: gather (x, y, z, info) of every rank FROM THE DEVICE BUFFERS (NCCL)
            rd = db.results_device()
            dist.all_gather_into_tensor(gathered, torch.cat([rd["x"], rd["y"], rd["z"], rd["info"]], dim=1))
        return db.results()      # D2H of this rank's x, y, z, se, si + info
    d2h_bytes = 8 * B * (n + 2 * ne + 2 * ni) + B * 20 * 8
    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t.item())

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        cpu = None
        b_alg = None
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, full_mask)  # the CPU leg gets every CPU of the box again
            pin_openmp_env(host_threads())
            cpu = cpu_baseline(sample=CPU_SAMPLE, reps=5)
            b_alg = algorithmic_bytes_per_qp(cpu["counters"], n, ne, ni, ni, cpu["sample"])
        else:
            try:
                with open(os.path.join(ROOT, "profiles", "algorithmic_bytes.json")) as f:
                    b_alg = json.load(f)["bytes_per_qp"]
            except Exception:
                b_alg = None
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            pass
        ncu = {}
        try:  # utilisation figures of the committed ncu --set full capture of this kernel (profiles/, per round)
            with open(os.path.join(ROOT, "profiles", "ncu_solve_metrics.json")) as f:
                ncu = json.load(f)
        except Exception:
            pass
        roof = None
        if b_alg is not None and kernel_ms > 0:
            achieved = b_alg * B / (kernel_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                    "peak_source": peak_src, "kernel": "pqp_solve_kernel", "kernel_ms": kernel_ms,
                    "algorithmic_bytes_per_qp": b_alg, "compulsory_bytes_per_qp": compulsory_bytes_per_qp(n, ne, ni),
                    "achieved_compulsory_gbs": compulsory_bytes_per_qp(n, ne, ni) * B / (kernel_ms * 1e-3) / 1e9,
                    "note": "three figures, never mixed: `achieved` uses the streamed-operand model B_alg of SURVEY 8(d)(ii) (what the CPU algorithm streams), "
                            "`achieved_compulsory_gbs` the compulsory floor B_min, `traffic` the ncu-measured DRAM bytes per launch. The kernel keeps its factors on chip, "
                            "so HBM is not its roof; `ncu` gives issue-slot / FP64-pipe utilisation of the same kernel",
                    "ncu": ncu or None}
        line = {
            "metric": "QPs solved/sec (batch dense, n=100)", "value": value, "unit": "QPs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"BatchQP {B} random dense QPs per GPU, n={n} n_eq={n_eq_str()} n_in={ni}, fp64, eps_abs=1e-9 eps_rel=0 NO_INITIAL_GUESS (BASELINE.json configs[1]'s QP shape at the north-star batch of 4096; generator of benchmark/timings-parallel.cpp)",
                       "batch_per_gpu": B, "global_batch": world * B, "parallelism": f"batch sharded over {world} GPU(s), no collective in the iteration",
                       "e2e_mode": os.environ.get("PQP_E2E", "fused") + " (init uploads, the solve kernel equilibrates + solves each QP as its inputs arrive)",
                       "host_buffers": "pinned, first-touched on the GPU's NUMA node %s" % (numa[0] if numa else "(unknown: default placement)"),
                       "l2": "inputs larger than L2 (scaled+model data %.0f MB per GPU per step)" % (2 * h2d_bytes / 1e6)},
            "e2e": {"value": e2e_value, "unit": "QPs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": None if cpu is None else {"value": cpu["qps"], "unit": "QPs/s", "cores": cpu["cores"], "kind": "port",
                                                      "sample": f"{cpu['sample']} QPs of the same workload x {cpu['reps']} repetitions (best), OpenMP schedule(dynamic), {cpu['solved']}/{cpu['sample']} solved; {cpu['flags']}",
                                                      "times_ms": [round(1e3 * t, 2) for t in cpu["times"]], "threads_tried_ms": {str(k): round(1e3 * v, 2) for k, v in cpu["tried"].items()},
                                                      "host_threads": cpu["host_threads"], "cgroup_cpu_quota": cpu_quota()},
        }
        print(json.dumps(line))
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs, rank * B)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def n_eq_str():
    return str(N_EQ)


if __name__ == "__main__":
    main()
