"""InteriorPoint.solve_all on the B200: a list of problems of different shapes in one lpb_solve_many_ragged call.
Each LP must give the bits lp_b200.solve_many gives a batch of that LP alone, whatever else is in the list and in
whatever order; problems outside solve_many's limits get the bits of InteriorPoint.solve.  Parity bar against the
oracle: status equal, iterations +-1, x 1e-6, fun 1e-8 rel."""
import ctypes as C

import numpy as np
import pytest

import lp_b200
from lp_b200 import _ffi
from lp_b200.api import _pack_problems
from oracle import ipm_oracle as o

pytestmark = pytest.mark.gpu


def raw_lp(m, n, seed, dtype=np.float64):
    """SURVEY 8(d) construction (as tests/test_gpu_solve_many.py): m // 2 inequality rows, the rest equalities, n
    slack-form columns; strictly primal- and dual-feasible.  Returns the ProblemBuilder inputs."""
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
    c = A0.T.dot(y0) + rng.uniform(0.5, 1.5, n0)
    return [v.astype(dtype) for v in (c, A0[:mh], b[:mh], A0[mh:], b[mh:])]


def build(m, n, seed, dtype=np.float64):
    c, A_ub, b_ub, A_eq, b_eq = raw_lp(m, n, seed, dtype)
    return lp_b200.Problem.target(c).ub(A_ub, b_ub).eq(A_eq, b_eq).build()


# K6 footprint of an LP (batched.cu: batched_smem_doubles), in bytes
def k6_bytes(m, n, ns):
    mp = (m + 15) // 16 * 16
    lda = (n - ns + 15) // 16 * 16 + 4
    vec = mp * (mp + 1) + 10 * n + 5 * m + 2 * mp + 2 * 64 + 8 * 8 + (mp // 16) * 16 * 17 + (4 * 16 + 16 * 17) + 2
    return 8 * (m * lda + vec)


def group(m, n, ns):
    """The launch group of a ragged call: K8, K6 one CTA per SM, or K6 two per SM.  The library asks the occupancy
    API for the two-per-SM limit; on a B200 (228 KB of shared memory per SM, 1 KB reserved per CTA) it is 113 KB."""
    b = k6_bytes(m, n, ns)
    if m > 64 or b > 227 * 1024:
        return "K8"
    return "K6-two" if b <= 113 * 1024 else "K6-one"


SHAPES = [(64, 128), (64, 256), (64, 400), (96, 192), (100, 173), (65, 70), (128, 768), (37, 91), (16, 40)]


def mixed_list():
    return [build(m, n, 5000 + 10 * k + r) for k, (m, n) in enumerate(SHAPES) for r in range(4 if m < 128 else 2)]


def ragged(problems, solver=None):
    """lpb_solve_many_ragged on host arrays: (x_slack list, fun, iterations, status)."""
    pk = _pack_problems(problems)
    solver = solver or lp_b200.InteriorPoint.default()
    rc = _ffi.load().lpb_solve_many_ragged(len(problems), pk.m.ctypes.data, pk.n.ctypes.data, pk.A.ctypes.data,
                                           pk.b.ctypes.data, pk.c.ctypes.data, C.byref(solver._o), pk.x.ctypes.data,
                                           pk.fun.ctypes.data, pk.it.ctypes.data, pk.st.ctypes.data,
                                           _ffi.LPB_MEM_HOST, None)
    assert rc == _ffi.LPB_OK, _ffi.last_error()
    xs = [pk.x[pk.c_off[k]: pk.c_off[k] + pk.n[k]].copy() for k in range(len(problems))]
    return xs, pk.fun.copy(), pk.it.copy(), pk.st.copy()


def alone(p, solver=None):
    """solve_many on a batch of this problem alone: (x_slack, fun, iteration, status)."""
    r = lp_b200.solve_many(p.A()[None], p.b()[None], p.c()[None], n_slack=p.n_slack(), solver=solver)
    return r.x_slack[0], r.fun[0], r.iteration[0], r.status[0]


def assert_same_bits(got, want, what=""):
    np.testing.assert_array_equal(got[0], want[0], err_msg=what)
    assert (got[1], got[2], got[3]) == (want[1], want[2], want[3]), what


def test_shapes_cover_the_three_launch_groups():
    groups = {group(m, n, m // 2) for m, n in SHAPES}
    assert groups == {"K8", "K6-one", "K6-two"}
    assert group(64, 128, 32) == "K6-two" and group(64, 256, 32) == "K6-one" and group(64, 400, 32) == "K8"


def test_mixed_list_matches_oracle_and_batch_of_one():
    pbs = mixed_list()
    res = lp_b200.InteriorPoint.default().solve_all(pbs)
    xs, fun, it, st = ragged(pbs)
    for k, (p, r) in enumerate(zip(pbs, res)):
        assert isinstance(r, lp_b200.OptimizeResult), (k, r)
        ref = o.InteriorPoint().solve(o.Problem(p.A(), p.b(), p.c(), 0.0, p.n_slack()))
        assert abs(r.iteration() - ref.iteration) <= 1, k
        assert np.abs(r.x() - ref.x).max() < 1e-6, k  # the oracle's x is de-normalised already
        assert abs(r.fun() - ref.fun) <= 1e-8 * max(1.0, abs(ref.fun)), k
        one = alone(p)
        assert_same_bits((xs[k], fun[k], it[k], st[k]), one, "LP %d %s" % (k, p.A().shape))
        np.testing.assert_array_equal(r.x(), one[0][: p.A().shape[1] - p.n_slack()])
        assert r.fun() == one[1] + p.c0() and r.iteration() == one[2]


def test_order_does_not_change_the_bits():
    pbs = mixed_list()
    base = ragged(pbs)
    perm = np.random.default_rng(7).permutation(len(pbs))
    got = ragged([pbs[i] for i in perm])
    for j, i in enumerate(perm):
        assert_same_bits((got[0][j], got[1][j], got[2][j], got[3][j]),
                         (base[0][i], base[1][i], base[2][i], base[3][i]), "LP %d" % i)


def test_each_lp_keeps_its_own_slack_structure():
    """One LP without the identity block does not make the others store and contract their slack columns."""
    pbs = mixed_list()
    base = ragged(pbs)
    k = 5  # a 64 x 256 LP (K6, one per SM)
    p = pbs[k]
    A2 = p.A().copy()
    nd = A2.shape[1] - p.n_slack()
    A2[5, nd + 5] = 2.0  # that slack column is 2 e_5 now: a different, still valid LP
    broken = lp_b200.Problem.target(p.c()).eq(A2, p.b()).build()
    pbs2 = list(pbs)
    pbs2[k] = broken
    got = ragged(pbs2)
    for i in range(len(pbs)):
        row = (got[0][i], got[1][i], got[2][i], got[3][i])
        if i != k:
            assert_same_bits(row, (base[0][i], base[1][i], base[2][i], base[3][i]), "LP %d" % i)
        assert_same_bits(row, alone(pbs2[i]), "LP %d alone" % i)
    ref = o.InteriorPoint().solve(o.Problem(A2, p.b(), p.c(), 0.0, 0))
    assert abs(int(got[2][k]) - ref.iteration) <= 1 and np.abs(got[0][k] - ref.x).max() < 1e-6


def test_uniform_list_equals_solve_many_on_the_stack():
    pbs = [build(96, 192, 6000 + i) for i in range(12)] + [build(64, 128, 6100 + i) for i in range(12)]
    xs, fun, it, st = ragged(pbs)
    for lo in (0, 12):
        grp = pbs[lo: lo + 12]
        r = lp_b200.solve_many(np.stack([p.A() for p in grp]), np.stack([p.b() for p in grp]),
                               np.stack([p.c() for p in grp]), n_slack=grp[0].n_slack())
        np.testing.assert_array_equal(np.stack(xs[lo: lo + 12]), r.x_slack)
        np.testing.assert_array_equal(fun[lo: lo + 12], r.fun)
        np.testing.assert_array_equal(it[lo: lo + 12], r.iteration)
        np.testing.assert_array_equal(st[lo: lo + 12], r.status)


def status_problems():
    """The three LPs of test_solve_many_statuses_and_limits (infeasible, unbounded, fine): 96 x (n + 3), K8."""
    c, A_ub, b_ub, A_eq, b_eq = raw_lp(95, 150, 77)
    big = o.build_problem(c, A_ub, b_ub, A_eq, b_eq)
    small_A = [np.array([[1.0, 1.0, 1.0]]), np.array([[1.0, -1.0, 1.0]]), np.array([[1.0, 1.0, 1.0]])]
    small_b = [np.array([-1.0]), np.array([1.0]), np.array([2.0])]
    small_c = [np.array([1.0, 1.0, 0.0]), np.array([-1.0, 0.0, 0.0]), np.array([-1.0, -2.0, 0.0])]
    m0, n0 = big.A.shape
    out = []
    for k in range(3):
        A = np.zeros((m0 + 1, n0 + 3))
        A[:m0, :n0] = big.A
        A[m0:, n0:] = small_A[k]
        out.append(lp_b200.Problem.target(np.concatenate([big.c, small_c[k]]))
                   .eq(A, np.concatenate([big.b, small_b[k]])).build())
    return out


def test_statuses_come_back_as_the_exceptions_solve_raises():
    pbs = status_problems() + [build(64, 128, 42)]
    for solver in (lp_b200.InteriorPoint.default(), lp_b200.InteriorPoint.custom().max_iter(1).build()):
        res = solver.solve_all(pbs)
        for p, r in zip(pbs, res):
            try:
                want = solver.solve(p)
            except lp_b200.LinearProgramError as e:
                want = e
            assert type(r) is type(want), (type(r), type(want))
            if isinstance(want, lp_b200.IterationLimitExceeded):
                assert r.x is not None and r.x.shape == (p.A().shape[1],) and np.isfinite(r.x).all()
    res = lp_b200.InteriorPoint.default().solve_all(pbs)
    assert [type(r) for r in res] == [lp_b200.Infeasible, lp_b200.Unbounded, lp_b200.OptimizeResult,
                                      lp_b200.OptimizeResult]
    limited = lp_b200.InteriorPoint.custom().max_iter(1).build().solve_all(pbs)
    assert isinstance(limited[3], lp_b200.IterationLimitExceeded)


def test_problems_outside_the_limits_fall_back_to_solve():
    pbs = mixed_list()[:8]
    base = ragged(pbs)
    big = [build(200, 400, 9001), build(128, 1000, 9002)]
    lst = pbs[:4] + [big[0]] + pbs[4:] + [big[1]]
    solver = lp_b200.InteriorPoint.default()
    res = solver.solve_all(lst)
    for p, r in ((big[0], res[4]), (big[1], res[-1])):
        want = solver.solve(p)
        np.testing.assert_array_equal(r.x(), want.x())
        assert (r.fun(), r.iteration()) == (want.fun(), want.iteration())
    for k, r in enumerate(res[:4] + res[5:-1]):
        p = pbs[k]
        np.testing.assert_array_equal(r.x(), base[0][k][: p.A().shape[1] - p.n_slack()])
        assert r.fun() == base[1][k] and r.iteration() == base[2][k]


def test_float32_problems_come_back_as_float32():
    pbs = [build(m, n, 7000 + k, np.float32) for k, (m, n) in enumerate([(64, 128), (96, 192)])]
    assert all(p.dtype() == np.float32 for p in pbs)
    res = lp_b200.InteriorPoint.default().solve_all(pbs)
    for p, r in zip(pbs, res):
        assert r.x().dtype == np.float32
        one = alone(p)
        np.testing.assert_array_equal(r.x(), one[0][: p.A().shape[1] - p.n_slack()].astype(np.float32))
        assert r.fun() == float(np.float32(one[1]))


def test_staging_host_pinned_and_device_inputs():
    """1024 LPs: the four-chunk pipeline, with one chunk all K8 and another all K6.  Host inputs, page-locked inputs
    (solve_all) and device inputs give the same bits, also after lpb_release_workspaces."""
    import torch
    shapes = [(96, 192)] * 256 + [(24, 48)] * 512 + [(64, 256)] * 256
    pbs = [build(m, n, 8000 + i) for i, (m, n) in enumerate(shapes)]
    lib = _ffi.load()
    host = ragged(pbs)
    assert (host[3] == _ffi.LPB_OK).all()
    for k in (0, 300, 1000):
        assert_same_bits((host[0][k], host[1][k], host[2][k], host[3][k]), alone(pbs[k]), "LP %d" % k)
    solver = lp_b200.InteriorPoint.default()
    for rnd in range(2):
        res = solver.solve_all(pbs)
        for k, (p, r) in enumerate(zip(pbs, res)):
            np.testing.assert_array_equal(r.x(), host[0][k][: p.A().shape[1] - p.n_slack()])
            assert r.fun() == host[1][k] and r.iteration() == host[2][k]
        assert lib.lpb_release_workspaces() == 0
        lp_b200.release_cached_contexts()

    pk = _pack_problems(pbs)
    dev = torch.device("cuda", 0)
    dA, db, dc = (torch.from_numpy(np.array(v)).to(dev) for v in (pk.A, pk.b, pk.c))
    dx = torch.zeros(pk.x.size, dtype=torch.float64, device=dev)
    df = torch.zeros(len(pbs), dtype=torch.float64, device=dev)
    dit = torch.zeros(len(pbs), dtype=torch.int64, device=dev)
    dst = torch.zeros(len(pbs), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    rc = lib.lpb_solve_many_ragged(len(pbs), pk.m.ctypes.data, pk.n.ctypes.data, dA.data_ptr(), db.data_ptr(),
                                   dc.data_ptr(), C.byref(solver._o), dx.data_ptr(), df.data_ptr(), dit.data_ptr(),
                                   dst.data_ptr(), _ffi.LPB_MEM_DEVICE,
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == _ffi.LPB_OK, _ffi.last_error()
    np.testing.assert_array_equal(dx.cpu().numpy(), np.concatenate(host[0]))
    np.testing.assert_array_equal(df.cpu().numpy(), host[1])
    np.testing.assert_array_equal(dit.cpu().numpy(), host[2])
    np.testing.assert_array_equal(dst.cpu().numpy(), host[3])
