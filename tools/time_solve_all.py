"""Throughput of the ragged batched mode (lpb_solve_many_ragged / InteriorPoint.solve_all) (GPU only).

    python tools/time_solve_all.py [--out profiles/time_solve_all.json] [--batch 8192] [--reps 3]

SURVEY 8(d) generator (oracle.synthetic_lp), seeds 1000 + i.  All timings are taken in one run:
  * uniform control: `batch` LPs of 128 x 256 from device inputs; lpb_solve_many_ragged and lpb_solve_many alternate,
    CUDA events, one warm-up call each.  The packed arrays of a uniform list are the stacked arrays of the batch, so
    both calls read the same device buffers: the difference is what the descriptors, the structure scan per LP and the
    order array cost where the uniform path already works;
  * mixed list: `batch` LPs whose shapes are drawn (seeded) from 8 shapes spanning the three launch groups (K6 two
    CTAs per SM, K6 one per SM, K8), in shuffled order, from device inputs: lpb_solve_many_ragged against the
    workaround without it (one lpb_solve_many per shape group, back to back on one stream), CUDA events around each;
    and InteriorPoint.solve looped over the first 64 LPs (host clock);
  * end to end from a list of Problems through InteriorPoint.solve_all (host clock), with the packing into the
    page-locked staging buffer timed on its own.
The outputs of the ragged call are compared with the per-group workaround (bit for bit) and with the single-problem
path on the first 64 LPs (status equal, iterations +-1, x 1e-6, fun 1e-8 relative).
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np

import lp_b200
from lp_b200 import _ffi
from lp_b200.api import _pack_problems, _staging
from oracle import ipm_oracle as o
from time_solve_many import card

NLOOP = 64
# (m, n) slack form, m // 2 slack columns: K6 two per SM, K6 two per SM, K6 two per SM, K6 one per SM, K8 (m <= 64,
# A does not fit beside M), K8, K8, K8
MIXED = [(32, 96), (48, 128), (64, 128), (64, 256), (64, 400), (96, 192), (100, 174), (128, 256)]


def gen(shapes, seed0):
    raw, slack = [], []
    for i, (m, n) in enumerate(shapes):
        args = o.synthetic_lp(m, n, seed0 + i)
        raw.append(args)
        slack.append(o.build_problem(*args))
    return raw, slack


def to_dev(*arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to("cuda") for a in arrs]


def outputs(nx, batch):
    import torch
    return (torch.zeros(nx, dtype=torch.float64, device="cuda"), torch.zeros(batch, dtype=torch.float64, device="cuda"),
            torch.zeros(batch, dtype=torch.int64, device="cuda"), torch.zeros(batch, dtype=torch.int32, device="cuda"))


def timed(call, reps):
    """CUDA-event times (ms) of `reps` calls after one warm-up call."""
    import torch
    stream = torch.cuda.current_stream()
    call()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        call()
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


class Ragged:
    """lpb_solve_many_ragged on device copies of a packed list."""

    def __init__(self, slack):
        import torch
        self.batch = len(slack)
        self.m = np.array([p.A.shape[0] for p in slack], dtype=np.int64)
        self.n = np.array([p.A.shape[1] for p in slack], dtype=np.int64)
        self.dA, self.db, self.dc = to_dev(np.concatenate([p.A.reshape(-1) for p in slack]),
                                           np.concatenate([p.b for p in slack]), np.concatenate([p.c for p in slack]))
        self.out = outputs(int(self.n.sum()), self.batch)
        self.opts = lp_b200.InteriorPoint.default()._o
        self.stream = torch.cuda.current_stream().cuda_stream

    def __call__(self):
        dx, df, dit, dst = self.out
        rc = _ffi.load().lpb_solve_many_ragged(self.batch, self.m.ctypes.data, self.n.ctypes.data, self.dA.data_ptr(),
                                               self.db.data_ptr(), self.dc.data_ptr(), C.byref(self.opts),
                                               dx.data_ptr(), df.data_ptr(), dit.data_ptr(), dst.data_ptr(),
                                               _ffi.LPB_MEM_DEVICE, C.c_void_p(self.stream))
        assert rc == _ffi.LPB_OK, _ffi.last_error()

    def result(self):
        x, f, it, st = (t.cpu().numpy() for t in self.out)
        off = np.concatenate([[0], np.cumsum(self.n)])
        return [x[off[i]: off[i + 1]] for i in range(self.batch)], f, it, st


class Uniform:
    """lpb_solve_many on one shape group (device arrays; A, b, c may be given already on the device)."""

    def __init__(self, batch, m, n, dA=None, db=None, dc=None, slack=None):
        import torch
        self.batch, self.m, self.n = batch, m, n
        if dA is None:
            dA, db, dc = to_dev(np.stack([p.A for p in slack]), np.stack([p.b for p in slack]),
                                np.stack([p.c for p in slack]))
        self.dA, self.db, self.dc = dA, db, dc
        self.out = outputs(batch * n, batch)
        self.opts = lp_b200.InteriorPoint.default()._o
        self.stream = torch.cuda.current_stream().cuda_stream

    def __call__(self):
        dx, df, dit, dst = self.out
        rc = _ffi.load().lpb_solve_many(self.batch, self.m, self.n, self.dA.data_ptr(), self.db.data_ptr(),
                                        self.dc.data_ptr(), C.byref(self.opts), dx.data_ptr(), df.data_ptr(),
                                        dit.data_ptr(), dst.data_ptr(), _ffi.LPB_MEM_DEVICE, C.c_void_p(self.stream))
        assert rc == _ffi.LPB_OK, _ffi.last_error()

    def result(self):
        x, f, it, st = (t.cpu().numpy() for t in self.out)
        return list(x.reshape(self.batch, self.n)), f, it, st


def bits_equal(a, b):
    return bool(all(np.array_equal(x, y) for x, y in zip(a[0], b[0])) and np.array_equal(a[1], b[1])
                and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]))


def parity(res, single, slack):
    k = len(single)
    ok = bool((res[3][:k] == _ffi.LPB_OK).all())
    dit = max(abs(int(res[2][i]) - single[i].iteration()) for i in range(k))
    dx = max(float(np.abs(res[0][i][: len(res[0][i]) - slack[i].A.shape[0] // 2] - single[i].x()).max())
             for i in range(k))
    dfun = max(abs(res[1][i] - single[i].fun()) / max(1.0, abs(single[i].fun())) for i in range(k))
    return {"all_optimal": ok, "max_diter": dit, "max_dx": dx, "max_rel_dfun": dfun,
            "within_bar": bool(ok and dit <= 1 and dx < 1e-6 and dfun <= 1e-8)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "time_solve_all.json"))
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    res = {"card": card(), "batch": args.batch, "seeds": "1000 + i"}
    print(json.dumps(res["card"]), flush=True)

    # uniform control: the same device buffers through both entry points, alternating
    _, slack = gen([(128, 256)] * args.batch, 1000)
    rg = Ragged(slack)
    un = Uniform(args.batch, 128, 256, rg.dA.view(args.batch, 128, 256), rg.db.view(args.batch, 128),
                 rg.dc.view(args.batch, 256))
    rg(), un()
    ms_r, ms_u = [], []
    for _ in range(args.reps):
        ms_r += timed(rg, 1)
        ms_u += timed(un, 1)
    res["uniform_128x256"] = {
        "ragged_ms": ms_r, "solve_many_ms": ms_u,
        "ragged_lps_per_s": args.batch / (np.median(ms_r) * 1e-3),
        "solve_many_lps_per_s": args.batch / (np.median(ms_u) * 1e-3),
        "ragged_over_solve_many_time": float(np.median(ms_r) / np.median(ms_u)),
        "bit_identical": bits_equal(rg.result(), un.result())}
    print("uniform", json.dumps(res["uniform_128x256"]), flush=True)
    del rg, un, slack
    torch.cuda.empty_cache()

    # mixed list
    rng = np.random.default_rng(1)
    shapes = [MIXED[k] for k in rng.integers(0, len(MIXED), args.batch)]
    raw, slack = gen(shapes, 1000)
    rg = Ragged(slack)
    ms_r = timed(rg, args.reps)
    ragged_out = rg.result()
    groups = {s: [i for i in range(args.batch) if shapes[i] == s] for s in MIXED}
    calls = [Uniform(len(ix), m, n, slack=[slack[i] for i in ix]) for (m, n), ix in groups.items() if ix]

    def workaround():
        for cl in calls:
            cl()
    ms_w = timed(workaround, args.reps)
    work = [None] * args.batch, np.zeros(args.batch), np.zeros(args.batch, np.int64), np.zeros(args.batch, np.int32)
    for cl, ix in zip(calls, [ix for ix in groups.values() if ix]):
        x, f, it, st = cl.result()
        for k, i in enumerate(ix):
            work[0][i], work[1][i], work[2][i], work[3][i] = x[k], f[k], it[k], st[k]
    del calls
    solver = lp_b200.InteriorPoint.default()
    pbs_loop = [lp_b200.Problem.target(a[0]).ub(a[1], a[2]).eq(a[3], a[4]).build() for a in raw[:NLOOP]]
    solver.solve(pbs_loop[0])
    t0 = time.perf_counter()
    single = [solver.solve(p) for p in pbs_loop]
    loop_s = time.perf_counter() - t0
    res["mixed"] = {
        "shapes": ["%dx%d" % s for s in MIXED], "lps_per_shape": {"%dx%d" % s: len(ix) for s, ix in groups.items()},
        "A_bytes": int(rg.dA.numel() * 8), "iterations_mean": float(ragged_out[2].mean()),
        "optimal": int((ragged_out[3] == 0).sum()),
        "ragged_ms": ms_r, "ragged_lps_per_s": args.batch / (np.median(ms_r) * 1e-3),
        "per_shape_solve_many_ms": ms_w, "per_shape_solve_many_lps_per_s": args.batch / (np.median(ms_w) * 1e-3),
        "speedup_ragged_vs_per_shape": float(np.median(ms_w) / np.median(ms_r)),
        "single_problem_loop_lps_per_s": NLOOP / loop_s, "single_problem_loop_lps": NLOOP,
        "bit_identical_to_per_shape_solve_many": bits_equal(ragged_out, work),
        "parity_vs_single_problem_path": parity(ragged_out, single, slack)}
    print("mixed", json.dumps(res["mixed"]), flush=True)
    del rg
    torch.cuda.empty_cache()

    # end to end from Problems
    pbs = [lp_b200.Problem.target(a[0]).ub(a[1], a[2]).eq(a[3], a[4]).build() for a in raw]
    pack_s, e2e_s = [], []
    solver.solve_all(pbs)
    for _ in range(args.reps):
        t0 = time.perf_counter()
        _pack_problems(pbs, _staging)
        pack_s.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        out = solver.solve_all(pbs)
        e2e_s.append(time.perf_counter() - t0)
    same = all(np.array_equal(r.x(), ragged_out[0][i][: len(ragged_out[0][i]) - shapes[i][0] // 2])
               and r.fun() == ragged_out[1][i] and r.iteration() == ragged_out[2][i] for i, r in enumerate(out))
    res["mixed_end_to_end_solve_all"] = {
        "pack_ms": [v * 1e3 for v in pack_s], "solve_all_ms": [v * 1e3 for v in e2e_s],
        "solve_all_lps_per_s": args.batch / float(np.median(e2e_s)),
        "bit_identical_to_device_ragged": bool(same)}
    print("e2e", json.dumps(res["mixed_end_to_end_solve_all"]), flush=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1, default=float)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
