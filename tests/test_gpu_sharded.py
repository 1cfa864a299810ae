"""K7: the column-sharded path (SURVEY.md 8e) on real GPUs, one process per GPU, NCCL all-reduces of
M / the A.w products / the reduction scalars inside liblpb200.so.

* world = 1 cases run on any GPU box (they cover the device-side synthetic generator, config C5's
  data path, against the CPU oracle on the downloaded problem).
* world = 2 cases need two GPUs; they are skipped on a one-GPU machine.  The same
  decomposition is covered on the CPU with gloo in tests/test_sharded_gloo.py.
"""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

CASES = [(64, 128, 0), (130, 301, 2), (256, 512, 1)]
SYN = (256, 640, 7)
BIG = (1300, 3000, 4)   # 11 panels of 128 (ragged last one): exercises the distributed factorisation


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_device_synthetic_generator_world1_matches_oracle():
    """lpb_create_sharded_synthetic on one rank: the downloaded LP has the slack structure of
    linear_program.rs:145-156, is solved to Optimal, and the GPU solve agrees with the oracle on it."""
    import lp_b200
    from lp_b200.api import SyntheticShardedProblem
    from oracle import ipm_oracle as o
    m, n, seed = SYN
    with SyntheticShardedProblem(m, n, seed) as sp:
        A, b, c = sp.download()
        res = lp_b200.InteriorPoint.default().solve_resident(sp)
    mh, n0 = m // 2, n - m // 2
    np.testing.assert_array_equal(A[:mh, n0:], np.eye(mh))
    np.testing.assert_array_equal(A[mh:, n0:], 0.0)
    np.testing.assert_array_equal(c[n0:], 0.0)
    a0 = A[:, :n0]
    assert abs(a0.mean()) < 0.02 and abs(a0.std() - 1.0) < 0.02          # N(0,1) entries
    assert abs(np.corrcoef(a0[0], a0[1])[0, 1]) < 0.2                    # rows are not copies of one another
    ref = o.InteriorPoint().solve(o.Problem(A, b, c, 0.0, mh))
    assert abs(res.iteration() - ref.iteration) <= 1
    assert np.abs(res.x() - ref.x).max() < 1e-6
    assert abs(res.fun() - ref.fun) <= 1e-8 * max(1.0, abs(ref.fun))


def test_peer_memory_entry_points_refuse_unsharded_contexts():
    """lpb_peer_export / lpb_peer_import (the cudaIpc panel ring of the distributed factorisation) only make sense on
    a context of 2..8 ranks: a world-1 context gets LPB_ERR_BAD_ARGUMENT, keeps working, and "peer_panels" = 1 is
    refused while nothing is mapped."""
    import ctypes as C
    import lp_b200
    from lp_b200 import _ffi
    from lp_b200.api import SyntheticShardedProblem
    lib = _ffi.load()
    m, n, seed = SYN
    with SyntheticShardedProblem(m, n, seed) as sp:
        assert sp.peer_panels is False
        buf = (C.c_ubyte * 64)()
        state = C.c_int(-1)
        assert lib.lpb_peer_export(sp.handle, buf, C.byref(state)) == _ffi.LPB_ERR_BAD_ARGUMENT
        assert lib.lpb_peer_import(sp.handle, (C.c_ubyte * 64)(), 1) == _ffi.LPB_ERR_BAD_ARGUMENT
        assert lib.lpb_set_option(sp.handle, b"peer_panels", 1) == _ffi.LPB_ERR_BAD_ARGUMENT
        assert lib.lpb_set_option(sp.handle, b"peer_panels", 0) == _ffi.LPB_OK
        res = lp_b200.InteriorPoint.default().solve_resident(sp)
        assert res.iteration() > 0


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group(backend="nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import lp_b200
        from lp_b200.api import ShardedProblem, SyntheticShardedProblem
        from oracle import ipm_oracle as o
        out = {}
        solver = lp_b200.InteriorPoint.default()
        for (m, n, seed) in CASES:
            c, A_ub, b_ub, A_eq, b_eq = o.synthetic_lp(m, n, seed)
            pb = lp_b200.Problem.target(c).ub(A_ub, b_ub).eq(A_eq, b_eq).build()
            with ShardedProblem(pb, rank, world, dist) as sp:
                res = solver.solve_resident(sp)
                prof = sp.profile()
            out[(m, n, seed)] = (res.x(), res.fun(), res.iteration(), prof["comm_ms"])
        m, n, seed = SYN
        with SyntheticShardedProblem(m, n, seed, rank, world, dist) as sp:
            A_k, b, c_k = sp.download()
            res = solver.solve_resident(sp)
        out["syn"] = (A_k, b, c_k, sp.col0, res.x(), res.fun(), res.iteration())
        # distributed factorisation (2: two broadcasts per panel + side-stream potf2 + packed panels, the default;
        # 1: one broadcast per panel) vs the replicated one (0) on the same all-reduced M
        from lp_b200 import _ffi
        lib = _ffi.load()
        m, n, seed = BIG
        c, A_ub, b_ub, A_eq, b_eq = o.synthetic_lp(m, n, seed)
        pb = lp_b200.Problem.target(c).ub(A_ub, b_ub).eq(A_eq, b_eq).build()
        ldm = (m + 15) // 16 * 16
        big = {}
        for mode in (2, "nccl", 1, 0):   # 2: first panel rows through peer memory (cudaIpc) | "nccl": through ncclBroadcast
            with ShardedProblem(pb, rank, world, dist) as sp:
                if mode == 2:
                    assert sp.peer_panels, "the peers' panel rings were not mapped: " + _ffi.last_error()
                if mode == "nccl":
                    sp.set_option("peer_panels", 0)
                sp.set_option("potrf_dist", 2 if mode == "nccl" else mode)
                sp.set_option("check_replicas", 1)
                assert lib.lpb_blind_start(sp.handle) == 0
                assert lib.lpb_form_and_factor(sp.handle) == 0, _ffi.last_error()
                L = np.tril(sp.debug_read("M").reshape(m, ldm)[:, :m])
                res = solver.solve_resident(sp)
            big[mode] = (L, res.x(), res.fun(), res.iteration())
        with ShardedProblem(pb, rank, world, dist) as sp:   # all-reduce of the full square instead of the packed triangle
            sp.set_option("packed_allreduce", 0)
            assert lib.lpb_blind_start(sp.handle) == 0
            assert lib.lpb_form_and_factor(sp.handle) == 0, _ffi.last_error()
            big["square"] = np.tril(sp.debug_read("M").reshape(m, ldm)[:, :m])
        out["big"] = big
        q.put((rank, out))
        dist.barrier()
        lib.lpb_comm_finalize()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_gpu_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_column_sharded_solve_matches_oracle_and_one_gpu():
    import torch.multiprocessing as mp
    import lp_b200
    from lp_b200.api import SyntheticShardedProblem
    from oracle import ipm_oracle as o
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for key in CASES:
        ref = o.InteriorPoint().solve(o.build_problem(*o.synthetic_lp(*key)))
        for rank in (0, 1):
            x, fun, it, comm_ms = results[rank][key]
            assert abs(it - ref.iteration) <= 1
            assert np.abs(x - ref.x).max() < 1e-6
            assert abs(fun - ref.fun) <= 1e-8 * max(1.0, abs(ref.fun))
            assert comm_ms > 0.0                                          # the NCCL all-reduces did run
        np.testing.assert_array_equal(results[0][key][0], results[1][key][0])   # ranks agree bit for bit
        assert results[0][key][1] == results[1][key][1]
    # distributed factorisation: every entry of L is computed by exactly one rank with the same kernels and
    # the same order of updates as the replicated run -> identical bits across ranks AND across the two modes
    ref = o.InteriorPoint().solve(o.build_problem(*o.synthetic_lp(*BIG)))
    for rank in (0, 1):
        for mode in (2, "nccl", 1, 0):
            L, x, fun, it = results[rank]["big"][mode]
            np.testing.assert_array_equal(L, results[0]["big"][0][0])
            assert abs(it - ref.iteration) <= 1
            assert np.abs(x - ref.x).max() < 1e-6
            assert abs(fun - ref.fun) <= 1e-8 * max(1.0, abs(ref.fun))
    for rank in (0, 1):  # packed-triangle all-reduce vs the plain one: same M up to the order of the sums
        Lsq = results[rank]["big"]["square"]
        assert np.abs(Lsq - results[0]["big"][1][0]).max() <= 1e-12 * np.abs(Lsq).max()
    Lref = np.linalg.cholesky((lambda A: A @ A.T)(o.build_problem(*o.synthetic_lp(*BIG)).A))
    L = results[0]["big"][1][0]
    assert np.abs(L - Lref).max() <= 1e-10 * np.abs(Lref).max()
    # device-side generator: the two shards tile the world-1 problem exactly (counter-based entries)
    m, n, seed = SYN
    with SyntheticShardedProblem(m, n, seed) as sp:
        A1, b1, c1 = sp.download()
        res1 = lp_b200.InteriorPoint.default().solve_resident(sp)
    A2 = np.concatenate([results[0]["syn"][0], results[1]["syn"][0]], axis=1)
    c2 = np.concatenate([results[0]["syn"][2], results[1]["syn"][2]])
    np.testing.assert_array_equal(A2, A1)
    np.testing.assert_allclose(results[0]["syn"][1], b1, rtol=1e-13, atol=1e-12)   # b is an all-reduced sum
    np.testing.assert_array_equal(results[0]["syn"][1], results[1]["syn"][1])
    np.testing.assert_allclose(c2, c1, rtol=1e-13, atol=1e-12)
    for rank in (0, 1):
        x, fun, it = results[rank]["syn"][4:7]
        assert abs(it - res1.iteration()) <= 1
        assert np.abs(x - res1.x()).max() < 1e-6
        assert abs(fun - res1.fun()) <= 1e-8 * max(1.0, abs(res1.fun()))
