"""Throughput of lp_b200.solve_many against the single-problem path looped over the same LPs (GPU only).

    python tools/time_solve_many.py [--out profiles/time_solve_many.json] [--batch 8192]

For each shape (128 x 256: K8; 96 x 192: K8), batch 8192, seeds 1000 + i, SURVEY 8(d) generator:
  * solve_many with device-resident inputs, CUDA events around lpb_solve_many after one warm-up call;
  * solve_many end to end from page-locked host memory (upload, kernel, download), host clock;
  * InteriorPoint.solve on a cached context (one warm-up solve), looped over the first 64 LPs;
and, as a regression guard, C4 (8192 LPs of 64 x 128) through lpb_solve_batched with device inputs.
A of one shape is batch * m * n * 8 bytes (2.1 GB at 128 x 256), far above the 126 MB of L2, so only the A of the
LPs resident on the SMs sits in L2.  The outputs of both paths on the first 64 seeds are saved next to the JSON and
checked against each other with the parity bar (status equal, iterations +-1, x 1e-6, fun 1e-8 relative).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np

import lp_b200
from lp_b200 import _ffi
from oracle import ipm_oracle as o

NLOOP = 64


def gen(batch, m, n, seed0, pinned):
    alloc = lp_b200.pinned_empty if pinned else np.empty
    A, b, c = alloc((batch, m, n)), alloc((batch, m)), alloc((batch, n))
    raw = []
    for i in range(batch):
        args = o.synthetic_lp(m, n, seed0 + i)
        pb = o.build_problem(*args)
        A[i], b[i], c[i] = pb.A, pb.b, pb.c
        if i < NLOOP:
            raw.append(args)
    return A, b, c, raw


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # the number is still printed, without the card's limit
        q = "unknown (%s)" % e
    return {"name": name, "power_limit_and_max_sm_clock": q,
            "l2_bytes": torch.cuda.get_device_properties(0).L2_cache_size}


def device_rate(entry, A, b, c, reps):
    """LPs/s of one call on device-resident inputs (CUDA events, after one warm-up call); returns outputs too."""
    import torch
    lib = _ffi.load()
    batch, m, n = A.shape
    dev = torch.device("cuda", 0)
    dA, db, dc = (torch.from_numpy(np.asarray(v)).to(dev) for v in (A, b, c))
    dx = torch.zeros((batch, n), dtype=torch.float64, device=dev)
    df = torch.zeros(batch, dtype=torch.float64, device=dev)
    dit = torch.zeros(batch, dtype=torch.int64, device=dev)
    dst = torch.zeros(batch, dtype=torch.int32, device=dev)
    opts = lp_b200.InteriorPoint.default()._o
    stream = torch.cuda.current_stream()
    torch.cuda.synchronize()

    def call():
        rc = getattr(lib, entry)(batch, m, n, dA.data_ptr(), db.data_ptr(), dc.data_ptr(), C.byref(opts),
                                 dx.data_ptr(), df.data_ptr(), dit.data_ptr(), dst.data_ptr(), _ffi.LPB_MEM_DEVICE,
                                 C.c_void_p(stream.cuda_stream))
        assert rc == _ffi.LPB_OK, _ffi.last_error()

    call()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        call()
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    out = dict(x=dx.cpu().numpy(), fun=df.cpu().numpy(), it=dit.cpu().numpy(), st=dst.cpu().numpy())
    del dA, db, dc, dx, df, dit, dst
    torch.cuda.empty_cache()
    return batch / (np.median(ms) * 1e-3), ms, out


def host_rate(A, b, c, n_slack, reps):
    lp_b200.solve_many(A, b, c, n_slack=n_slack)
    s = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = lp_b200.solve_many(A, b, c, n_slack=n_slack)
        s.append(time.perf_counter() - t0)
    return A.shape[0] / np.median(s), [v * 1e3 for v in s], r


def single_rate(raw):
    solver = lp_b200.InteriorPoint.default()
    pbs = [lp_b200.Problem.target(a[0]).ub(a[1], a[2]).eq(a[3], a[4]).build() for a in raw]
    solver.solve(pbs[0])  # warm-up: context creation for the shape
    x, fun, it = [], [], []
    t0 = time.perf_counter()
    for pb in pbs:
        r = solver.solve(pb)
        x.append(r.x())
        fun.append(r.fun())
        it.append(r.iteration())
    dt = time.perf_counter() - t0
    return len(pbs) / dt, dict(x=np.array(x), fun=np.array(fun), it=np.array(it))


def parity(many, single, n_slack):
    k = len(single["it"])
    ok = bool((many["st"][:k] == _ffi.LPB_OK).all())
    dit = int(np.abs(many["it"][:k] - single["it"]).max())
    dx = float(np.abs(many["x"][:k, : many["x"].shape[1] - n_slack] - single["x"]).max())
    dfun = float((np.abs(many["fun"][:k] - single["fun"]) / np.maximum(1.0, np.abs(single["fun"]))).max())
    return {"all_optimal": ok, "max_diter": dit, "max_dx": dx, "max_rel_dfun": dfun,
            "within_bar": bool(ok and dit <= 1 and dx < 1e-6 and dfun <= 1e-8)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "time_solve_many.json"))
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    res = {"card": card(), "batch": args.batch, "seeds": "1000 + i", "shapes": {}}
    print(json.dumps(res["card"]), flush=True)
    for m, n in [(128, 256), (96, 192)]:
        A, b, c, raw = gen(args.batch, m, n, 1000, pinned=True)
        n_slack = m // 2
        dev_rate, dev_ms, many = device_rate("lpb_solve_many", A, b, c, args.reps)
        e2e_rate, e2e_ms, _ = host_rate(A, b, c, n_slack, args.reps)
        loop_rate, single = single_rate(raw)
        par = parity(many, single, n_slack)
        np.savez(os.path.splitext(args.out)[0] + "_outputs_%dx%d.npz" % (m, n),
                 many_x=many["x"][:NLOOP], many_fun=many["fun"][:NLOOP], many_it=many["it"][:NLOOP],
                 single_x=single["x"], single_fun=single["fun"], single_it=single["it"])
        r = {"A_bytes": A.nbytes, "iterations_mean": float(many["it"].mean()),
             "optimal": int((many["st"] == 0).sum()),
             "solve_many_device_lps_per_s": float(dev_rate), "solve_many_device_ms": dev_ms,
             "solve_many_pinned_e2e_lps_per_s": float(e2e_rate), "solve_many_pinned_e2e_ms": e2e_ms,
             "single_problem_loop_lps_per_s": loop_rate, "single_problem_loop_lps": NLOOP,
             "speedup_device_vs_loop": float(dev_rate / loop_rate), "parity_vs_single_problem_path": par}
        res["shapes"]["%dx%d" % (m, n)] = r
        print("%dx%d" % (m, n), json.dumps(r), flush=True)
        del A, b, c
    A, b, c, _ = gen(args.batch, 64, 128, 1000, pinned=False)
    c4_rate, c4_ms, c4 = device_rate("lpb_solve_batched", A, b, c, args.reps)
    res["C4_solve_batched_device"] = {"lps_per_s": float(c4_rate), "ms": c4_ms, "optimal": int((c4["st"] == 0).sum())}
    print("C4", json.dumps(res["C4_solve_batched_device"]), flush=True)
    res["bar_10x_at_128x256"] = bool(res["shapes"]["128x256"]["speedup_device_vs_loop"] >= 10.0)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
