#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native interior-point path.

    python bench.py --gpus N --steps K --warmup W [--workload C1|C2|C3] [--impl reference] [--dump-outputs DIR]

A "step" is ONE COMPLETE SOLVE (blind start -> Optimal) of the workload LP, i.e. one pass of the
hot path (`InteriorPoint::solve`, /root/reference/src/solvers/interior_point/mod.rs:161-240) over
one synthetic problem.  metric = IPM iterations per second (BASELINE.json: "time-to-solve & IPM
iterations/s"); ms_per_step is the time-to-solve.

  value : iterations/s with the problem already resident in HBM (lpb_solve on a live context),
          timed with CUDA events on the stream the kernels are launched on, max over ranks.
  e2e   : the same through the public reference-shaped API (`InteriorPoint.solve(problem)`):
          context creation, H2D of A/b/c from pinned host memory, solve, D2H of x, teardown.
  roofline : the dominant kernel (K1, DMMA SYRK): m(m+1)n algorithmic flop per launch / its mean
          launch duration (CUDA events inside the library, on the launching stream); `peak` is the nominal
          B200 FP64 figure, `peak_measured` the DMMA issue peak measured in this very run.
  cpu_baseline : the oracle (NumPy/OpenBLAS restatement of the reference) on the host cores: REAL
          iterations of its loop on the same workload, as many as fit a bounded budget.
  c5 : every product line also carries a short record of config C5 (32768 x 131072, generated on the device
          per column shard, 3 iterations): per-iteration time and phases at this N -- the configuration the
          north star quotes the multi-GPU target on.

`--impl reference` times the oracle's own loop (real iterations, all host threads); its `config` equals the
product arm's.  Both arms report `ms_per_iteration`; `ms_per_step` is one complete solve in the product arm and
one bounded sample of iterations in the reference arm (`details.step`).

N > 1: strong scaling -- the same LP with A column-sharded over the ranks (SURVEY.md 8e), NCCL
all-reduce of M and of the A.w products.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned to its caller as
DIR/<name>.npy in float64: `x`, `fun` and `iteration` of the solve (C4: `x`, `fun`, `iteration` and `status` of
every LP, rows in batch order, with `lp_index`).  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

if "reference" in sys.argv[1:]:
    # The CPU arm uses every host thread -- also under torchrun, which exports OMP_NUM_THREADS=1 to its ranks.
    # Must happen before NumPy loads its BLAS.
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {  # slack-form (m, n); BASELINE.json configs[0..4]
    "C1": (512, 1024),
    "C2": (4096, 8192),
    "C3": (16384, 32768),
    "C4": (64, 128),        # batched: 8192 independent LPs, one CTA per problem, batch sharded over ranks
    "C5": (32768, 131072),  # A generated on the device per column shard (never on the host)
}
C4_BATCH = 8192
DEFAULT_WORKLOAD = "C3"
NOMINAL_FP64_TFLOPS = 40.0  # B200 FP64 (tensor == vector), NVIDIA HGX B200 spec sheet


def workload_label(name, m, n, seed):
    return "%s dense LP slack-form m=%d n=%d seed=%d (ub+eq, SURVEY 8d generator)" % (name, m, n, seed)


def bench_config(workload, m, n, seed, world, potrf_dist=2):
    """`config` of the JSON line: the SAME dict in the product and the reference arm."""
    if workload == "C4":
        wl = "C4 batched: %d independent dense LPs slack-form m=%d n=%d, seeds 1000+i, one CTA per problem" % (
            C4_BATCH, m, n)
        par = "batch sharded over %d GPU(s), no collective" % world
    else:
        wl = workload_label(workload, m, n, seed)
        if workload == "C5":
            wl += ", generated on the device per column shard (counter-based N(0,1))"
        par = "1 GPU" if world == 1 else "A column-sharded over %d GPUs, NCCL all-reduce of M, %s Cholesky" % (
            world, "panel-broadcast distributed" if potrf_dist else "replicated")
    a_mb = m * n * 8 / 1e6
    l2 = ("inputs larger than L2 (A = %.0f MB, streamed from HBM by every sweep and SYRK)" % a_mb if a_mb > 126.0 else
          "inputs fit in L2 (A = %.0f MB), no flush between iterations: a parity-test configuration, not a bench line"
          % a_mb)
    return {"workload": wl, "parallelism": par, "l2": l2}


def synthetic_lp(m, n, seed):
    """SURVEY.md 8(d) generator (same bits as oracle.ipm_oracle.synthetic_lp; duplicated here so the
    product arm never imports the oracle)."""
    mh = m // 2
    n0 = n - mh
    rng = np.random.default_rng(seed)
    A0 = rng.standard_normal((m, n0))
    x0 = rng.uniform(0.5, 1.5, n0)
    s0 = rng.uniform(0.5, 1.5, mh)
    b = A0.dot(x0)
    b[:mh] += s0
    y0 = rng.standard_normal(m)
    y0[:mh] = -np.abs(y0[:mh])
    z0 = rng.uniform(0.5, 1.5, n0)
    c = A0.T.dot(y0) + z0
    return c, A0[:mh], b[:mh], A0[mh:], b[mh:]


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled every 100 ms during the timed region (NVML)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# --------------------------------------------------------------------------- CPU baseline / reference arm
def cpu_problem(m, n, seed):
    """The workload LP as the oracle's Problem (built once per process: generation is not what is timed)."""
    from oracle import ipm_oracle as o
    return o.build_problem(*synthetic_lp(m, n, seed))


def cpu_iterations(pb, budget_s, min_iters=1, max_iters=200):
    """Run the oracle's loop (interior_point/mod.rs:199-240 restated) from the blind start and time REAL
    iterations until `budget_s` is used up (at least `min_iters`).  Returns (iterations, seconds) of the timed
    iterations; the blind-start residuals before the first iteration are not counted."""
    from oracle import ipm_oracle as o

    class _Stop(Exception):
        pass

    stamps = []

    def on_iteration(iteration, pt, ind):
        stamps.append(time.perf_counter())
        if (iteration >= min_iters and stamps[-1] - t_start >= budget_s) or iteration >= max_iters:
            raise _Stop()

    t_start = time.perf_counter()
    box = {}

    def first_tick(*a):
        box.setdefault("t0", time.perf_counter())

    # the clock starts when blind_start() has produced the first iterate (its 2 GEMVs are set-up, not an iteration)
    orig = o.blind_start
    try:
        def timed_blind_start(p):
            pt = orig(p)
            first_tick()
            return pt
        o.blind_start = timed_blind_start
        try:
            o.InteriorPoint().solve(pb, on_iteration=on_iteration)
        except (_Stop, o.LinearProgramError):
            pass
    finally:
        o.blind_start = orig
    its = len(stamps)
    if its == 0:
        return 0, 0.0
    return its, stamps[-1] - box["t0"]


def cpu_sample(m, n, seed, budget_s=25.0, pb=None):
    """Time the oracle (the reference's algorithm on host cores, OpenBLAS threads) on a bounded sample of the
    workload: REAL consecutive iterations of its loop.  Returns (iterations_per_s, sample_description, cores)."""
    cores = os.cpu_count() or 1
    if pb is None:
        pb = cpu_problem(m, n, seed)
    its, dt = cpu_iterations(pb, budget_s)
    desc = "oracle loop on %d host threads: the first %d real iteration(s) of the %dx%d solve in %.1f s" % (
        cores, its, m, n, dt)
    return its / dt, desc, cores


def run_reference_arm(args, m, n):
    """The reference's own CPU implementation of the path (the oracle port: no Rust toolchain here) on the box's
    host cores.  One continuous run of its loop; the first `warmup` samples are untimed, the next `steps` samples
    are timed; a sample is `k` consecutive real iterations (k sized so the whole run stays within minutes)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    if args.workload in ("C4", "C5"):
        print(json.dumps({"impl": "reference", "unavailable":
                          "the CPU port of %s is not run by this arm (C4: see the product line's cpu_baseline; C5: "
                          "A does not fit the host)" % args.workload}), flush=True)
        return
    pb = cpu_problem(m, n, args.seed)
    # calibrate one iteration, then choose k so that (warmup + steps) * k iterations take <= ~4 minutes
    its1, dt1 = cpu_iterations(pb, 0.0, min_iters=1)
    t_it = dt1 / max(1, its1)
    n_samples = args.warmup + args.steps
    k = int(max(1, min(8, 240.0 / max(t_it, 1e-3) / max(1, n_samples))))
    total_its = n_samples * k
    from oracle import ipm_oracle as o
    stamps = []

    class _Stop(Exception):
        pass

    def on_iteration(iteration, pt, ind):
        stamps.append(time.perf_counter())
        if iteration >= total_its:
            raise _Stop()

    t0 = time.perf_counter()
    finished = None
    try:
        res = o.InteriorPoint().solve(pb, on_iteration=on_iteration)
        finished = res.iteration
    except _Stop:
        pass
    except o.LinearProgramError:
        pass
    done = len(stamps)
    w_its = min(args.warmup * k, max(0, done - 1))
    t_begin = stamps[w_its - 1] if w_its > 0 else t0
    timed_its = done - w_its
    dt = stamps[-1] - t_begin
    value = timed_its / dt
    steps_done = max(1, timed_its // k) if finished is None else args.steps
    sample = ("oracle loop on %d host threads: %d consecutive real iterations of the %dx%d solve timed (%.1f s) after %d "
              "untimed ones; a step is a sample of %d iteration(s)%s" % (
                  cores, timed_its, m, n, dt, w_its, k,
                  "" if finished is None else "; the solve converged after %d iterations inside the run" % finished))
    line = {
        "impl": "reference", "metric": "ipm_iterations_per_s", "value": value, "unit": "iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / steps_done * 1e3,
        "ms_per_iteration": 1e3 / value,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.workload, m, n, args.seed, args.gpus, args.potrf_dist),
        "details": {"step": "%d real iterations of the CPU loop" % k, "iterations_timed": timed_its,
                    "calibration_s_per_iteration": t_it},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- shared pieces of the product arm
def _sync_max_ms(torch, dist, ms):
    if dist is None:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as <out_dir>/<name>.npy in float64 (64 MB at most in all)."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError("--dump-outputs: %d bytes exceed the limit of %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_solve(out_dir, res):
    dump_outputs(out_dir, {"x": res.x(), "fun": res.fun(), "iteration": res.iteration()})


def _gather_rows(torch, dist, t, per, total):
    """Rows of a batch sharded over the ranks in blocks of `per`, on the host in batch order (every rank calls)."""
    if dist is None:
        return t.cpu().numpy()
    pad = torch.zeros((per,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[: t.shape[0]] = t
    parts = [torch.empty_like(pad) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, pad)
    return torch.cat(parts)[:total].cpu().numpy()


def _roofline(prof_sum, m, n_loc, peak_measured=None):
    """K1 roofline.  `achieved` counts the flop the kernel EXECUTES: m(m+1) * syrk_cols, where syrk_cols
    is n minus the trailing slack columns that liblpb200 folds into the diagonal of M instead of
    contracting over them (lpb_profile.syrk_cols).  SURVEY 8(d)'s algorithmic figure m(m+1)n -- what a
    structure-blind SYRK would execute -- divided by the same time is reported beside it."""
    launches = max(1, prof_sum.get("syrk_launches", 1))
    solves = max(1, prof_sum.get("solves", 1))
    n_exec = prof_sum.get("syrk_cols", 0) / solves or n_loc
    f_alg = float(m) * (m + 1) * n_loc
    f_syrk = float(m) * (m + 1) * n_exec
    f_chol = float(m) ** 3 / 3.0
    syrk_ms = prof_sum.get("syrk_ms", 0.0) / launches
    potrf_ms = prof_sum.get("potrf_ms", 0.0) / max(1, prof_sum.get("potrf_launches", 1))
    achieved = f_syrk / (syrk_ms * 1e-3) * 1e-12 if syrk_ms > 0 else None
    return {
        "bound": "tensor", "kernel": "syrk_dmma_kernel (K1, A.diag(x/z).A^T, FP64 DMMA)",
        "achieved": achieved, "peak": NOMINAL_FP64_TFLOPS, "unit": "TFLOP/s",
        "frac": (achieved / NOMINAL_FP64_TFLOPS) if achieved else None,
        "traffic": SYRK_TRAFFIC.get((m, int(n_exec)), (None, None))[0],
        "traffic_source": SYRK_TRAFFIC.get((m, int(n_exec)), (None, None))[1],
        "peak_source": "nominal B200 FP64 (MEASURED_PEAKS.json has no FP64 entry)",
        "peak_measured": peak_measured,
        "peak_measured_source": "DMMA issue peak measured in this run (lpb_measure_dmma_peak: register-only "
                                "mma.sync.m8n8k4.f64 loop on every SM, ~0.3 s)",
        "frac_of_measured": (achieved / peak_measured) if (achieved and peak_measured) else None,
        "flop_per_launch": f_syrk, "ms_per_launch": syrk_ms, "syrk_cols": n_exec,
        "algorithmic_flop_per_launch": f_alg,
        "algorithmic_tflops": (f_alg / (syrk_ms * 1e-3) * 1e-12) if syrk_ms > 0 else None,
        "phase_syrk_plus_cholesky_tflops": ((f_syrk + f_chol) / ((syrk_ms + potrf_ms) * 1e-3) * 1e-12
                                            if syrk_ms + potrf_ms > 0 else None),
        "potrf_ms_per_launch": potrf_ms,
        "potrf_tflops": (f_chol / (potrf_ms * 1e-3) * 1e-12) if potrf_ms > 0 else None,
    }


# dram__bytes_read.sum + dram__bytes_write.sum of ONE syrk_dmma_kernel launch, from the committed
# `ncu --set full` captures (profiles/); keyed by (m, n_local).
SYRK_TRAFFIC = {
    # C3 on 1 GPU, banded tile order, K summed in blocks of 512 columns: 38.58 GB read + 2.84 GB written
    # (profiles/ncu_syrk_C3_r02_blocked.txt; round 1 without the blocked sum: 46.05 + 1.08); algorithmic bytes: 3.22 GB of
    # A (dense columns) + 1.07 GB of M.  The kernel is DMMA-bound (DRAM at 2.6 % of peak); the re-reads are operand tiles
    # streamed once per wave of 148 tiles.
    # NOT measured in the run (ncu cannot run inside a timed bench): the value of the committed capture.
    (16384, 24576): (38.577897e9 + 2.840231e9, "profiles/ncu_syrk_C3_r02_blocked.txt (ncu --set full, one launch)"),
}


def measure_peak(rp):
    """DMMA issue peak of this GPU, measured now through the library (None if the call fails)."""
    from lp_b200 import _ffi
    out = C.c_double(0.0)
    rc = _ffi.load().lpb_measure_dmma_peak(rp.handle, C.c_double(0.3), C.byref(out))
    return float(out.value) if rc == 0 and out.value > 0 else None


C5_RECORD_ITERS = 3


def c5_record(args, torch, dist, rank, world, stream):
    """Config C5 (32768 x 131072, A generated on the device per column shard) for C5_RECORD_ITERS iterations at
    this N: per-iteration time and phases.  Rides along in every product line so the scaling run shows the
    configuration the north star quotes the multi-GPU target on (its full solve is `--workload C5`)."""
    import lp_b200
    from lp_b200.api import SyntheticShardedProblem
    m5, n5 = WORKLOADS["C5"]
    solver = lp_b200.InteriorPoint.custom().max_iter(C5_RECORD_ITERS).build()
    rec = None
    try:
        with SyntheticShardedProblem(m5, n5, args.seed, rank, world, dist, stream=stream) as sp:
            sp.set_option("potrf_dist", args.potrf_dist)
            status = "IterationLimitExceeded"
            try:
                solver.solve_resident(sp)
                status = "Optimal"
            except lp_b200.IterationLimitExceeded:
                pass
            p = sp.profile()
            n_loc = sp.n
        its = max(1, int(p["iterations"]))
        ms = _sync_max_ms(torch, dist, p["total_ms"])
        f_syrk = float(m5) * (m5 + 1) * p["syrk_cols"]
        rec = {"workload": bench_config("C5", m5, n5, args.seed, world, args.potrf_dist)["workload"],
               "n_gpus": world, "iterations": its, "status_after_%d_iterations" % C5_RECORD_ITERS: status,
               "ms_per_iteration": ms / its, "iterations_per_s": its / (ms * 1e-3),
               "phases_ms_per_iteration": {k: p[k] / its for k in ("syrk_ms", "potrf_ms", "solve_ms", "sweep_ms",
                                                                   "vector_ms", "comm_ms")},
               "syrk_tflops_this_gpu": (f_syrk / (p["syrk_ms"] / max(1, p["syrk_launches"]) * 1e-3) * 1e-12
                                        if p["syrk_ms"] > 0 else None),
               "a_shard_gb": m5 * n_loc * 8 / 1e9,
               "note": "times include the blind-start residuals; CUDA events on the launching stream, max over ranks"}
    except Exception as e:  # noqa: BLE001 -- the record must never take the headline line down with it
        rec = {"error": "%s: %s" % (type(e).__name__, e)}
    return rec


def _timed_solves(args, torch, dist, solver, rp, local_rank):
    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        solver.solve_resident(rp)
    barrier()
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_sum, launches, total_iters, res = {}, 0, 0, None
    sampler.start()
    barrier()
    e0.record()
    for _ in range(args.steps):
        res = solver.solve_resident(rp)
        total_iters += res.iteration()
        p = rp.profile()
        launches += p["launches"]
        for k, v in p.items():
            prof_sum[k] = prof_sum.get(k, 0) + v
        prof_sum["solves"] = prof_sum.get("solves", 0) + 1
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = _sync_max_ms(torch, dist, e0.elapsed_time(e1))
    return ms, total_iters, launches, prof_sum, clocks, res


def run_device_synthetic(args, torch, dist, rank, local_rank, world, stream, m, n):
    """C5 (and any size with --device-synthetic): A is generated per column shard on the device."""
    import lp_b200
    from lp_b200.api import SyntheticShardedProblem
    solver = lp_b200.InteriorPoint.default()
    t0 = time.perf_counter()
    rp = SyntheticShardedProblem(m, n, args.seed, rank, world, dist, stream=stream)
    rp.set_option("potrf_dist", args.potrf_dist)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    ms, total_iters, launches, prof_sum, clocks, res = _timed_solves(args, torch, dist, solver, rp, local_rank)
    if args.dump_outputs and rank == 0:
        dump_solve(args.dump_outputs, res)
    value = total_iters / (ms * 1e-3)
    peak_holder = [measure_peak(rp) if rank == 0 else None]
    rp.close()
    # e2e: context creation + on-device generation of the shard + solve + D2H / gather of x
    e2e = None
    if not args.no_e2e:
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        it_e2e = 0
        for _ in range(args.steps):
            with SyntheticShardedProblem(m, n, args.seed, rank, world, dist, stream=stream) as sp:
                it_e2e += solver.solve_resident(sp).iteration()
        torch.cuda.synchronize()
        dt = _sync_max_ms(torch, dist, (time.perf_counter() - t0) * 1e3) * 1e-3
        e2e = {"value": it_e2e / dt, "unit": "iterations/s", "h2d_bytes_per_step": 0,
               "d2h_bytes_per_step": int(rp.n * 8 + 16), "ms_per_step": dt / args.steps * 1e3,
               "note": "inputs are generated on the device (the %.1f GB matrix never exists on the host); "
                       "the timed region covers generation + solve + D2H of x" % (m * n * 8 / 1e9)}
    n_loc = rp.n
    if rank == 0:
        steps = args.steps
        phases = {k: prof_sum.get(k, 0.0) / steps for k in
                  ("total_ms", "syrk_ms", "potrf_ms", "solve_ms", "sweep_ms", "vector_ms", "comm_ms")}
        line = {
            "metric": "ipm_iterations_per_s", "value": value, "unit": "iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "ms_per_iteration": ms / max(1, total_iters), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.workload, m, n, args.seed, world, args.potrf_dist),
            "details": {"iterations_per_solve": total_iters / args.steps, "objective": res.fun(),
                        "device_generation_s": gen_s, "step": "one complete solve (blind start -> Optimal)"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": _roofline(prof_sum, m, n_loc, peak_holder[0]),
            "phases_ms_per_solve": phases, "cpu_baseline": None,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        _ffi_finalize()
        dist.destroy_process_group()


def run_batched(args, torch, dist, rank, local_rank, world, stream):
    """C4: `batch` independent 64x128 LPs, one CTA per problem; the batch is sharded over the ranks
    with no collective on the data path (SURVEY.md 8e)."""
    import lp_b200
    from lp_b200 import _ffi
    lib = _ffi.load()
    m, n = WORKLOADS["C4"]
    batch = args.batch
    per = -(-batch // world)
    lo, hi = min(batch, rank * per), min(batch, (rank + 1) * per)
    nb = hi - lo
    t0 = time.perf_counter()
    A = lp_b200.pinned_empty((nb, m, n))  # host inputs of the e2e leg live in pinned memory (H2D at PCIe rate)
    b = lp_b200.pinned_empty((nb, m))
    c = lp_b200.pinned_empty((nb, n))
    for i in range(nb):  # SURVEY 8(d): seeds 1000 + i
        cc, A_ub, b_ub, A_eq, b_eq = synthetic_lp(m, n, 1000 + lo + i)
        pb = lp_b200.Problem.target(cc).ub(A_ub, b_ub).eq(A_eq, b_eq).build()
        A[i], b[i], c[i] = pb.A(), pb.b(), pb.c()
    gen_s = time.perf_counter() - t0
    solver = lp_b200.InteriorPoint.default()
    dA, db, dc = torch.from_numpy(A).cuda(), torch.from_numpy(b).cuda(), torch.from_numpy(c).cuda()
    dx = torch.zeros((nb, n), dtype=torch.float64, device="cuda")
    dfun = torch.zeros(nb, dtype=torch.float64, device="cuda")
    dit = torch.zeros(nb, dtype=torch.int64, device="cuda")
    dst = torch.zeros(nb, dtype=torch.int32, device="cuda")

    def resident():
        rc = lib.lpb_solve_batched(nb, m, n, dA.data_ptr(), db.data_ptr(), dc.data_ptr(), C.byref(solver._o),
                                   dx.data_ptr(), dfun.data_ptr(), dit.data_ptr(), dst.data_ptr(),
                                   _ffi.LPB_MEM_DEVICE, C.c_void_p(stream))
        assert rc == 0, _ffi.last_error()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        resident()
    barrier()
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    barrier()
    e0.record()
    for _ in range(args.steps):
        resident()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = _sync_max_ms(torch, dist, e0.elapsed_time(e1))
    its = dit.sum().to(torch.float64).reshape(1)
    n_ok = (dst == 0).sum().to(torch.float64).reshape(1)
    if dist is not None:
        dist.all_reduce(its)
        dist.all_reduce(n_ok)
    total_iters = float(its.item())
    value = total_iters * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        outs = [_gather_rows(torch, dist, t, per, batch) for t in (dx, dfun, dit, dst)]
        if rank == 0:
            rows = np.arange(batch)
            if batch * (n + 4) * 8 > DUMP_LIMIT_BYTES:  # a fixed, seeded sample of the LPs
                rows = np.sort(np.random.default_rng(0).choice(batch, DUMP_LIMIT_BYTES // ((n + 4) * 8), replace=False))
            dump_outputs(args.dump_outputs, dict(zip(("lp_index", "x", "fun", "iteration", "status"),
                                                     [rows] + [o[rows] for o in outs])))
    # e2e: host arrays in, host arrays out through lp_b200.solve_batched (H2D of A, b, c + D2H of x, fun, ...)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = lp_b200.solve_batched(A, b, c, n_slack=m // 2, solver=solver, stream=stream)
    torch.cuda.synchronize()
    dt = _sync_max_ms(torch, dist, (time.perf_counter() - t0) * 1e3) * 1e-3
    e2e = {"value": total_iters * args.steps / dt, "unit": "iterations/s",
           "h2d_bytes_per_step": int((A.size + b.size + c.size) * 8), "d2h_bytes_per_step": int(nb * (n * 8 + 8 + 8 + 4)),
           "ms_per_step": dt / args.steps * 1e3}
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import ipm_oracle as o
            k = min(nb, 256)
            t0 = time.perf_counter()
            it_cpu = 0
            for i in range(k):
                it_cpu += o.InteriorPoint().solve(o.Problem(A[i], b[i], c[i], 0.0, m // 2)).iteration
            dtc = time.perf_counter() - t0
            cpu = {"value": it_cpu / dtc, "unit": "iterations/s", "cores": os.cpu_count() or 1, "kind": "port",
                   "sample": "oracle looped over the first %d of the %d LPs" % (k, batch)}
        # one-time load of each LP into shared memory is the only HBM traffic of the kernel
        bytes_per_lp = (m * n + m + n) * 8 + n * 8 + 24
        line = {
            "metric": "ipm_iterations_per_s", "value": value, "unit": "iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(bench_config("C4", m, n, args.seed, world),
                           l2="whole batch (%.0f MB) larger than L2" % (batch * bytes_per_lp / 1e6)),
            "details": {"lps_per_s": batch * args.steps / (ms * 1e-3), "optimal": int(n_ok.item()), "batch": batch,
                        "iterations_per_lp": total_iters / batch, "host_generation_s": gen_s},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(args.steps),
            "roofline": {"bound": "hbm", "kernel": "batched_ipm_kernel (K6): latency / shared-memory bound; HBM only "
                                                   "for the one-time load of each LP",
                         "achieved": batch * bytes_per_lp / (ms / args.steps * 1e-3) / 1e9 / world, "peak": _hbm_peak(),
                         "unit": "GB/s", "frac": batch * bytes_per_lp / (ms / args.steps * 1e-3) / 1e9 / world / _hbm_peak(),
                         "traffic": None},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        _ffi_finalize()
        dist.destroy_process_group()


def _ffi_finalize():
    from lp_b200 import _ffi
    _ffi.load().lpb_comm_finalize()


def _hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0  # B200_PROFILING.md fallback


# --------------------------------------------------------------------------- product arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the short C5 record that rides along with the C3 line")
    ap.add_argument("--device-synthetic", action="store_true",
                    help="generate the LP on the device per column shard (always on for C5)")
    ap.add_argument("--batch", type=int, default=C4_BATCH)
    ap.add_argument("--potrf-dist", type=int, default=2, choices=[0, 1, 2],
                    help="N > 1: 2 = distributed Cholesky, two broadcasts per panel + side-stream potf2 (default), "
                         "1 = one broadcast per panel, 0 = replicated on every rank")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the product arm (--impl b200)")
    m, n = WORKLOADS[args.workload]

    if args.impl == "reference":
        run_reference_arm(args, m, n)
        return

    import torch
    import lp_b200
    from lp_b200 import _ffi
    from lp_b200.api import ResidentProblem, ShardedProblem

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d" % args.gpus)
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    lib = _ffi.load()
    stream = torch.cuda.current_stream().cuda_stream

    if args.workload == "C4":
        run_batched(args, torch, dist, rank, local_rank, world, stream)
        return
    if args.workload == "C5" or args.device_synthetic:
        run_device_synthetic(args, torch, dist, rank, local_rank, world, stream, m, n)
        return

    # ---- build the workload on the host (identical bits on every rank)
    t0 = time.perf_counter()
    c, A_ub, b_ub, A_eq, b_eq = synthetic_lp(m, n, args.seed)
    problem = lp_b200.Problem.target(c).ub(A_ub, b_ub).eq(A_eq, b_eq).build()
    del A_ub, A_eq
    gen_s = time.perf_counter() - t0
    solver = lp_b200.InteriorPoint.default()

    if world > 1:
        rp = ShardedProblem(problem, rank, world, dist, stream=stream)
        rp.set_option("potrf_dist", args.potrf_dist)
        peer_panels = bool(rp.peer_panels)
    else:
        rp = ResidentProblem(problem, stream=stream)
        peer_panels = False
    for kv in filter(None, os.environ.get("LPB_BENCH_OPTS", "").split(",")):  # experiments: "key=value,key=value"
        k, v = kv.split("=")
        rp.set_option(k, int(v))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    iters = 0
    for _ in range(args.warmup):
        res = solver.solve_resident(rp)
        iters = res.iteration()
    barrier()

    # ---- timed region: EXACTLY K solves, CUDA events on the launching stream
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_sum = {}
    launches = 0
    total_iters = 0
    sampler.start()
    barrier()
    e0.record()
    for _ in range(args.steps):
        res = solver.solve_resident(rp)
        total_iters += res.iteration()
        p = rp.profile()
        launches += p["launches"]
        for k, v in p.items():
            prof_sum[k] = prof_sum.get(k, 0) + v
        prof_sum["solves"] = prof_sum.get("solves", 0) + 1
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_solve(args.dump_outputs, res)
    value = total_iters / (ms * 1e-3)
    fun = res.fun()
    n_loc_rank = rp.n
    peak_measured = measure_peak(rp) if rank == 0 else None

    # ---- e2e through the public API (host buffers, H2D + D2H inside the timed region)
    e2e = None
    if not args.no_e2e and world == 1:
        rp.close()
        torch.cuda.synchronize()
        solver.solve(problem)  # warm (allocator, pinned pages)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        it_e2e = 0
        for _ in range(args.steps):
            r2 = solver.solve(problem)
            it_e2e += r2.iteration()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e2e = {"value": it_e2e / dt, "unit": "iterations/s", "h2d_bytes_per_step": int((m * n + m + n) * 8),
               "d2h_bytes_per_step": int(n * 8 + 16), "ms_per_step": dt / args.steps * 1e3}
    elif world > 1:
        # sharded: the public call is ShardedProblem(...) + solve_resident; time upload + solve + download
        rp.close()
        barrier()
        t0 = time.perf_counter()
        it_e2e = 0
        for _ in range(args.steps):
            with ShardedProblem(problem, rank, world, dist, stream=stream) as sp:
                it_e2e += solver.solve_resident(sp).iteration()
        barrier()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": it_e2e / dt, "unit": "iterations/s",
               "h2d_bytes_per_step": int((m * (n // world) + m + n // world) * 8),
               "d2h_bytes_per_step": int((n // world) * 8 + 16), "ms_per_step": dt / args.steps * 1e3}

    # ---- C5 record (device-generated, 3 iterations) at this N: after the headline numbers, nothing above depends on it
    c5 = None
    if not args.no_c5 and args.workload == DEFAULT_WORKLOAD:
        torch.cuda.empty_cache()
        c5 = c5_record(args, torch, dist, rank, world, stream)

    if rank == 0:
        roofline = _roofline(prof_sum, m, n_loc_rank, peak_measured)
        steps = args.steps
        phases = {k: prof_sum.get(k, 0.0) / steps for k in
                  ("total_ms", "syrk_ms", "potrf_ms", "solve_ms", "sweep_ms", "vector_ms", "comm_ms")}
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            v, desc, cores = cpu_sample(m, n, args.seed)
            cpu = {"value": v, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": desc}
        line = {
            "metric": "ipm_iterations_per_s", "value": value, "unit": "iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "ms_per_iteration": ms / max(1, total_iters), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args.workload, m, n, args.seed, world, args.potrf_dist),
            "details": {"iterations_per_solve": total_iters / args.steps, "objective": fun, "host_generation_s": gen_s,
                        "step": "one complete solve (blind start -> Optimal)",
                        "peer_panels": peer_panels},  # first panel rows handed over through cudaIpc-mapped peer memory
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "phases_ms_per_solve": phases, "cpu_baseline": cpu, "c5": c5,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        _ffi_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
