"""solve_many on the B200: K8 (A read through L2, up to 128 rows) and K6 where K6 takes the shape, against the oracle
looped over the batch and against the single-problem path.  Parity bar per problem: status equal, iterations +-1,
x 1e-6, fun 1e-8 rel."""
import ctypes as C

import numpy as np
import pytest

import lp_b200
from lp_b200 import _ffi
from oracle import ipm_oracle as o

pytestmark = pytest.mark.gpu


def lp(m, n, seed):
    """SURVEY 8(d) construction for any m (oracle.synthetic_lp takes even m only): m // 2 inequality rows,
    the rest equalities, n slack-form columns; strictly primal- and dual-feasible."""
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
    return o.build_problem(c, A0[:mh], b[:mh], A0[mh:], b[mh:])


def make_batch(batch, m, n, seed0):
    pbs = [lp(m, n, seed0 + i) for i in range(batch)]
    return np.stack([p.A for p in pbs]), np.stack([p.b for p in pbs]), np.stack([p.c for p in pbs]), m // 2


def oracle_status(A, b, c, n_slack, **kw):
    try:
        ref = o.InteriorPoint(**kw).solve(o.Problem(A, b, c, 0.0, n_slack))
        return _ffi.LPB_OK, ref
    except o.Infeasible:
        return _ffi.LPB_ERR_INFEASIBLE, None
    except o.Unbounded:
        return _ffi.LPB_ERR_UNBOUNDED, None
    except o.IterationLimitExceeded:
        return _ffi.LPB_ERR_ITERATION_LIMIT_EXCEEDED, None


def assert_matches_oracle(res, A, b, c, n_slack):
    for i in range(A.shape[0]):
        ref = o.InteriorPoint().solve(o.Problem(A[i], b[i], c[i], 0.0, n_slack))
        assert res.status[i] == _ffi.LPB_OK, (i, res.status[i])
        assert abs(int(res.iteration[i]) - ref.iteration) <= 1, (i, res.iteration[i], ref.iteration)
        assert np.abs(res.x[i] - ref.x).max() < 1e-6, i
        assert abs(res.fun[i] - ref.fun) <= 1e-8 * max(1.0, abs(ref.fun)), i


@pytest.mark.parametrize("batch,m,n", [
    (64, 128, 256), (16, 128, 768),                  # K8 at full size
    (33, 96, 192), (9, 100, 173), (5, 65, 70),       # K8, m and n not multiples of 16
    (8, 64, 1024),                                   # K8: m <= 64, but A does not fit beside M
])
def test_solve_many_matches_oracle(batch, m, n):
    A, b, c, n_slack = make_batch(batch, m, n, 1000)
    assert_matches_oracle(lp_b200.solve_many(A, b, c, n_slack=n_slack), A, b, c, n_slack)


def test_solve_many_takes_k6_where_k6_fits():
    A, b, c, n_slack = make_batch(64, 64, 128, 1000)
    many = lp_b200.solve_many(A, b, c, n_slack=n_slack)
    batched = lp_b200.solve_batched(A, b, c, n_slack=n_slack)
    for name in ("x_slack", "fun", "iteration", "status"):
        np.testing.assert_array_equal(getattr(many, name), getattr(batched, name))
    assert_matches_oracle(many, A, b, c, n_slack)


def test_solve_many_equals_single_problem_path():
    A, b, c, n_slack = make_batch(8, 128, 256, 2000)
    res = lp_b200.solve_many(A, b, c, n_slack=n_slack)
    nu = 256 - n_slack
    for i in range(8):
        pb = (lp_b200.Problem.target(c[i][:nu]).ub(A[i][:n_slack, :nu], b[i][:n_slack])
              .eq(A[i][n_slack:, :nu], b[i][n_slack:]).build())
        single = lp_b200.InteriorPoint.default().solve(pb)
        assert abs(int(res.iteration[i]) - single.iteration()) <= 1
        np.testing.assert_allclose(res.x[i], single.x(), rtol=0, atol=1e-7)
        assert abs(res.fun[i] - single.fun()) <= 1e-8 * max(1.0, abs(single.fun()))


def test_solve_many_slack_structure_is_detected_from_the_data():
    """As for solve_batched: columns permuted (no trailing identity, K8 reads every column) give the same solutions,
    and one problem that breaks the identity block makes the whole batch read every column."""
    A, b, c, n_slack = make_batch(6, 128, 256, 4000)
    ref = lp_b200.solve_many(A, b, c, n_slack=n_slack)
    assert all(ref.status == _ffi.LPB_OK)
    perm = np.concatenate([np.arange(256 - n_slack, 256), np.arange(256 - n_slack)])
    got = lp_b200.solve_many(A[:, :, perm], b, c[:, perm])
    assert np.abs(got.iteration - ref.iteration).max() <= 1
    np.testing.assert_allclose(got.x_slack[:, np.argsort(perm)], ref.x_slack, rtol=0, atol=1e-7)
    np.testing.assert_allclose(got.fun, ref.fun, rtol=1e-9)
    A2 = A.copy()
    A2[3, 5, 256 - n_slack + 5] = 2.0             # problem 3: that slack column is 2 e_5 now, a different (still valid) LP
    mixed = lp_b200.solve_many(A2, b, c, n_slack=n_slack)
    one = o.InteriorPoint().solve(o.Problem(A2[3], b[3], c[3], 0.0, n_slack))
    assert abs(int(mixed.iteration[3]) - one.iteration) <= 1 and np.abs(mixed.x[3] - one.x).max() < 1e-6
    keep = [i for i in range(6) if i != 3]
    np.testing.assert_allclose(mixed.x_slack[keep], ref.x_slack[keep], rtol=0, atol=1e-7)


def test_solve_many_statuses_and_limits():
    """The three 1 x 3 LPs of test_batched_statuses_and_limits (infeasible, unbounded, fine), each block-diagonal
    beside the same feasible 95-row LP: 96 x (n + 3), K8."""
    big = lp(95, 150, 77)
    small_A = [np.array([[1.0, 1.0, 1.0]]), np.array([[1.0, -1.0, 1.0]]), np.array([[1.0, 1.0, 1.0]])]
    small_b = [np.array([-1.0]), np.array([1.0]), np.array([2.0])]
    small_c = [np.array([1.0, 1.0, 0.0]), np.array([-1.0, 0.0, 0.0]), np.array([-1.0, -2.0, 0.0])]
    m0, n0 = big.A.shape
    A = np.zeros((3, m0 + 1, n0 + 3))
    A[:, :m0, :n0] = big.A
    for k in range(3):
        A[k, m0:, n0:] = small_A[k]
    b = np.stack([np.concatenate([big.b, small_b[k]]) for k in range(3)])
    c = np.stack([np.concatenate([big.c, small_c[k]]) for k in range(3)])
    res = lp_b200.solve_many(A, b, c)
    want = [oracle_status(A[k], b[k], c[k], 0) for k in range(3)]
    assert [w[0] for w in want] == [_ffi.LPB_ERR_INFEASIBLE, _ffi.LPB_ERR_UNBOUNDED, _ffi.LPB_OK]
    assert list(res.status) == [w[0] for w in want]
    ref = want[2][1]
    assert abs(int(res.iteration[2]) - ref.iteration) <= 1
    assert np.abs(res.x[2] - ref.x).max() < 1e-6
    assert abs(res.fun[2] - ref.fun) <= 1e-8 * max(1.0, abs(ref.fun))
    res = lp_b200.solve_many(A, b, c, solver=lp_b200.InteriorPoint.custom().max_iter(1).build())
    assert res.status[2] == _ffi.LPB_ERR_ITERATION_LIMIT_EXCEEDED and res.iteration[2] == 1


def test_solve_many_staging_host_pinned_and_device_inputs():
    """Host inputs (staged through the cached arena), page-locked host inputs and device inputs give the same bits,
    also on a second call and after lpb_release_workspaces."""
    import torch
    A, b, c, n_slack = make_batch(16, 128, 256, 3000)
    r1 = lp_b200.solve_many(A, b, c, n_slack=n_slack)
    r2 = lp_b200.solve_many(A, b, c, n_slack=n_slack)
    assert _ffi.load().lpb_release_workspaces() == 0
    r3 = lp_b200.solve_many(A[:5], b[:5], c[:5], n_slack=n_slack)       # smaller batch: arena re-created
    Ap, bp, cp = lp_b200.pinned_empty(A.shape), lp_b200.pinned_empty(b.shape), lp_b200.pinned_empty(c.shape)
    Ap[:], bp[:], cp[:] = A, b, c
    r4 = lp_b200.solve_many(Ap, bp, cp, n_slack=n_slack)
    for r in (r2, r4):
        np.testing.assert_array_equal(r.x_slack, r1.x_slack)
        np.testing.assert_array_equal(r.fun, r1.fun)
        np.testing.assert_array_equal(r.iteration, r1.iteration)
    np.testing.assert_array_equal(r3.x_slack, r1.x_slack[:5])
    assert (r1.status == _ffi.LPB_OK).all()

    dev = torch.device("cuda", 0)
    dA, db, dc = (torch.from_numpy(v).to(dev) for v in (A, b, c))
    dx = torch.zeros((16, 256), dtype=torch.float64, device=dev)
    df = torch.zeros(16, dtype=torch.float64, device=dev)
    dit = torch.zeros(16, dtype=torch.int64, device=dev)
    dst = torch.zeros(16, dtype=torch.int32, device=dev)
    opts = lp_b200.InteriorPoint.default()._o
    torch.cuda.synchronize()
    rc = _ffi.load().lpb_solve_many(16, 128, 256, dA.data_ptr(), db.data_ptr(), dc.data_ptr(), C.byref(opts),
                                    dx.data_ptr(), df.data_ptr(), dit.data_ptr(), dst.data_ptr(), _ffi.LPB_MEM_DEVICE,
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == _ffi.LPB_OK, _ffi.last_error()
    np.testing.assert_array_equal(dx.cpu().numpy(), r1.x_slack)
    np.testing.assert_array_equal(df.cpu().numpy(), r1.fun)
    np.testing.assert_array_equal(dit.cpu().numpy(), r1.iteration)
    np.testing.assert_array_equal(dst.cpu().numpy(), r1.status)
