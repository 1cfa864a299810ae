"""Each phase of the single-problem IPM iteration on the B200, checked against tests/phase_check.py after every call:
the host loop drives lpb_blind_start ... lpb_extract_x, snapshots the device state before each call and compares the
call's outputs with a reference computed from that state, within worst-case rounding bounds.  The cases sit at the
edges of the sweeps, the reductions and the slack-column shortcut; a converged run must also reproduce
InteriorPoint.solve_resident bit for bit."""
import ctypes as C
import time

import numpy as np
import pytest

import lp_b200
from lp_b200 import _ffi
from lp_b200.api import ResidentProblem
from tests import phase_check as pc

pytestmark = pytest.mark.gpu


def lp(m, n, seed):
    """SURVEY 8(d) construction for any m: m // 2 inequality rows, the rest equalities, n slack-form columns;
    strictly primal- and dual-feasible (the generator of test_gpu_solve_many.py)."""
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
    return lp_b200.Problem.target(c).ub(A0[:mh], b[:mh]).eq(A0[mh:], b[mh:]).build()


def structured(A, seed):
    """An LP on a given A, as in test_structure_detection_edge_cases: b = A x0, c = A^T y0 + U(0.5, 1.5)."""
    rng = np.random.default_rng(seed)
    m, n = A.shape
    b = A @ rng.uniform(0.5, 1.5, n)
    c = A.T @ rng.standard_normal(m) + rng.uniform(0.5, 1.5, n)
    bufs = [lp_b200.api._HostBuffer(s) for s in (A.shape, b.shape, c.shape)]
    bufs[0].array[:], bufs[1].array[:], bufs[2].array[:] = A, b, c
    return lp_b200.Problem(bufs[0], bufs[1], bufs[2], 0.0, 0)


def singleton_tail(m, n0, k, seed, scale=True):
    """m x n0 Gaussian block followed by k singleton columns on rows 0..k-1 (scaled 1 + 0.25 j if `scale`)."""
    rng = np.random.default_rng(seed)
    tail = np.zeros((m, k))
    tail[np.arange(k), np.arange(k)] = 1.0 + 0.25 * np.arange(k) if scale else 1.0
    return np.hstack([rng.standard_normal((m, n0)), tail])


class Checked:
    """The phase calls with a snapshot of the state before each one and the checks of phase_check after it."""

    def __init__(self, rp, pb, check=True, refined=False):
        self.lib, self.rp, self.h = _ffi.load(), rp, rp.handle
        self.P = pc.Ref(pb.A(), pb.b(), pb.c(), pb.c0())
        self.check, self.refined = check, refined
        self.worst = {}
        self.state = None

    def snap(self):
        return {k: self.rp.debug_read(k) for k in pc.STATE}

    def call(self, fn, *args):
        assert fn(self.h, *args) == 0, _ffi.last_error()
        pre, self.state = self.state, (self.snap() if self.check else None)
        return pre, self.state

    def record(self, ratios):
        for k, v in ratios.items():
            self.worst[k] = max(self.worst.get(k, 0.0), v)

    def blind_start(self):
        self.state = self.snap() if self.check else None
        _, post = self.call(self.lib.lpb_blind_start)
        if self.check:
            self.record(pc.check_blind_start(self.P, post))

    def residuals(self, tau, kappa):
        rs = _ffi.lpb_residual_scalars()
        pre, post = self.call(self.lib.lpb_residuals, tau, kappa, C.byref(rs))
        if self.check:
            out = {k: getattr(rs, k) for k in ("nrm_rp", "nrm_rd", "cx", "by", "xz")}
            self.record(pc.check_residuals(self.P, pre, post, tau, out))
        return rs

    def form_and_factor(self):
        pre, post = self.call(self.lib.lpb_form_and_factor)
        if self.check:
            self.record(pc.check_form_and_factor(self.P, pre, post))

    def direction(self, corrector, ip, eta, gamma, mu, alpha, tau, kappa):
        din = _ffi.lpb_direction_in(corrector, int(ip), eta, gamma, mu, alpha)
        dout = _ffi.lpb_direction_out()
        steps = self.rp.debug_counter("refine_steps")
        pre, post = self.call(self.lib.lpb_direction, C.byref(din), tau, kappa, C.byref(dout))
        if self.refined:
            assert self.rp.debug_counter("refine_steps") >= steps + 1
        self.din = dict(corrector=corrector, ip=int(ip), eta=eta, gamma=gamma, mu=mu, alpha=alpha)
        out = {k: getattr(dout, k) for k in ("cu", "bv", "cp", "bq", "nan_pq")}
        if self.check:
            self.record(pc.check_direction(self.P, pre, post, self.din, out,
                                           pred_out=None if not corrector else self.pred_out, refined=self.refined))
        if not corrector:
            self.pred_out = out
        return dout

    def assemble_delta(self, d_tau):
        axz = (C.c_double * 2)()
        pre, post = self.call(self.lib.lpb_assemble_delta, d_tau, axz)
        if self.check:
            self.record(pc.check_assemble_delta(self.P, pre, post, d_tau, [axz[0], axz[1]], self.din))
        return axz

    def do_step(self, alpha, ip):
        pre, post = self.call(self.lib.lpb_do_step, alpha, int(ip))
        if self.check:
            self.record(pc.check_do_step(self.P, pre, post, alpha, ip))

    def extract_x(self, tau):
        x = np.zeros(self.P.n)
        fun = C.c_double()
        pre, _ = self.call(self.lib.lpb_extract_x, tau, x.ctypes.data, C.byref(fun))
        if self.check:
            self.record(pc.check_extract_x(self.P, pre, tau, x, fun.value))
        return x, fun.value


def drive(dev, n, ip, max_iter=50, check_iters=None):
    """The host loop of test_host_driven_phase_calls_equal_lpb_solve (ipm_driver.hpp), on `dev`."""
    tau = kappa = 1.0
    dev.check = check_iters is None or 0 in check_iters
    dev.blind_start()
    rs = dev.residuals(tau, kappa)
    ini = (rs.nrm_rp, rs.nrm_rd)
    it = 0
    converged = False
    while it < max_iter:
        it += 1
        dev.check = check_iters is None or it in check_iters
        if dev.check and dev.state is None:
            dev.state = dev.snap()
        gamma = 1.0 if ip else 0.0
        eta = 1.0 if ip else 1.0 - gamma
        r_G = rs.cx - rs.by + kappa
        mu = (rs.xz + tau * kappa) / (n + 1)
        dev.form_and_factor()
        dout = dev.direction(0, ip, eta, gamma, mu, 0.0, tau, kappa)
        assert dout.nan_pq == 0
        tk = gamma * mu - tau * kappa

        def dscal(g_hat, tk):
            d_tau = (g_hat + 1.0 / tau * tk - (-dout.cu + dout.bv)) / (1.0 / tau * kappa + (-dout.cp + dout.bq))
            return d_tau, 1.0 / tau * (tk - kappa * d_tau)

        def step(axz, d_tau, d_kappa, a0):
            at = min(1.0, tau / -d_tau) if d_tau < 0 else 1.0
            ak = min(1.0, kappa / -d_kappa) if d_kappa < 0 else 1.0
            return min(1.0, axz[0], at, axz[1], ak) * a0

        d_tau, d_kappa = dscal(r_G * eta, tk)
        axz = dev.assemble_delta(d_tau)
        alpha = step(axz, d_tau, d_kappa, 1.0)
        one_m = 1.0 - alpha  # (one_m * one_m), not pow(): libm's pow is not correctly rounded
        gamma = 10.0 if ip else (one_m * one_m) * min(0.1, one_m)
        eta = 1.0 if ip else 1.0 - gamma
        if ip:
            tk = (1.0 - alpha) * gamma * mu - tau * kappa - alpha * alpha * d_tau * d_kappa
        else:
            tk = gamma * mu - tau * kappa - d_tau * d_kappa
        dout = dev.direction(1, ip, eta, gamma, mu, alpha, tau, kappa)
        d_tau, d_kappa = dscal(r_G * eta, tk)
        axz = dev.assemble_delta(d_tau)
        alpha = 1.0 if ip else step(axz, d_tau, d_kappa, 0.99995)
        dev.do_step(alpha, ip)
        tau, kappa = tau + d_tau * alpha, kappa + d_kappa * alpha
        if ip:
            tau, kappa = max(tau, 1.0), max(kappa, 1.0)
        ip = False
        rs = dev.residuals(tau, kappa)
        rho_p = rs.nrm_rp / max(ini[0], 1.0)
        rho_d = rs.nrm_rd / max(ini[1], 1.0)
        rho_A = abs(rs.cx - rs.by) / (tau + abs(rs.by))
        if rho_p < 1e-8 and rho_d < 1e-8 and rho_A < 1e-8:
            converged = True
            break
    x, fun = dev.extract_x(tau)
    return converged, it, x, fun


def run_case(name, pb, n_dense, ip=True, structure=1, options=(), max_iter=50, check_iters=None):
    t0 = time.time()
    opts = dict(options, structure=structure)
    with ResidentProblem(pb) as rp:
        for k, v in opts.items():
            rp.set_option(k, v)
        dev = Checked(rp, pb, refined=bool(opts.get("refine", 0)))
        converged, it, x, fun = drive(dev, rp.n, ip, max_iter, check_iters)
        assert rp.profile()["syrk_cols"] == n_dense
    worst_key = max(dev.worst, key=dev.worst.get)
    print("\n[phases] %-34s %5d x %-8d n_dense %-8d it %2d  worst %.3g (%s)  %.1f s" % (
        name, pb.A().shape[0], pb.A().shape[1], n_dense, it, dev.worst[worst_key], worst_key, time.time() - t0))
    for k in sorted(dev.worst):
        print("    %-40s %.3g" % (k, dev.worst[k]))
    bad = {k: v for k, v in dev.worst.items() if not v <= 1.0}
    assert not bad, bad
    solver = lp_b200.InteriorPoint.custom().ip(ip).max_iter(max_iter).build()
    with ResidentProblem(pb) as rp:
        for k, v in opts.items():
            rp.set_option(k, v)
        if converged:
            res = solver.solve_resident(rp)
            assert res.iteration() == it
            np.testing.assert_array_equal(x[:rp.n - rp.n_slack], res.x())
            assert fun == res.fun()
        else:
            with pytest.raises(lp_b200.IterationLimitExceeded) as e:
                solver.solve_resident(rp)
            assert rp.last_iterations == it
            np.testing.assert_array_equal(x, e.value.x)
    return dev.worst


def test_tiny_odd_shape():
    """3 x 7 (1 inequality row, 2 equality rows): n < 16, so no structure; odd n (lane-0 tail of gemv_n, odd last
    column of gemv_t); m < 16 (ldm padding)."""
    run_case("3x7", lp(3, 7, 1), 7)


@pytest.mark.parametrize("structure", [1, 0])
@pytest.mark.parametrize("ip", [True, False])
def test_standard_slack_block(ip, structure):
    """64 x 128: 32 slack columns, n_dense = 96."""
    run_case("64x128 ip=%d structure=%d" % (ip, structure), lp(64, 128, 2), 96 if structure else 128,
             ip=ip, structure=structure)


@pytest.mark.parametrize("structure", [1, 0])
def test_odd_dense_part(structure):
    """97 x 229: n_dense = 181 is odd (the odd dense tail beside TailCols, the (nd + 1) & ~1 pitch); m is not a
    multiple of 16."""
    run_case("97x229 structure=%d" % structure, lp(97, 229, 3), 181 if structure else 229, structure=structure)


@pytest.mark.parametrize("structure", [1, 0])
def test_ragged_row_chunks(structure):
    """1025 x 2049: gemv_t_shape gives colblocks 9 (n = 2049) or 7 (n_dense = 1537), both want 64 chunks, so 17 rows
    per chunk and ceil(1025 / 17) = 61 chunks, the last of 5 rows; 61 = 4 * 15 + 1 sends sum_chunks into its
    remainder loop.  The Cholesky runs 8 panels of 128 plus one row."""
    run_case("1025x2049 structure=%d" % structure, lp(1025, 2049, 4), 1537 if structure else 2049,
             structure=structure)


def test_wide_reductions():
    """16 x 1 050 000, the first 4 iterations (checked in the first and the last): vec_blocks reaches the cap of 1024
    blocks, finalize_reduce_kernel folds 1024 partials, the thin epilogues loop about 4 times per thread.  Its 8
    slack columns are fewer than the 16 the shortcut needs, so A is dense."""
    run_case("16x1050000", lp(16, 1_050_000, 5), 1_050_000, ip=False, max_iter=4, check_iters=(1, 4))


def test_scaled_singletons_with_zero_column():
    """m = 40: 24 singleton columns scaled 1 + 0.25 j, one of them all zero (col_row = -1 in at_dot, col_val != 1)."""
    A = singleton_tail(40, 60, 24, 11)
    A[:, 60 + 3] = 0.0
    run_case("40x84 scaled + zero column", structured(A, 12), 60)


def test_singletons_sharing_a_row():
    """m = 40: the last singleton repeats row 5, so the run stops there and n_dense = n0 + 6 keeps singleton columns
    in the dense part."""
    A = singleton_tail(40, 60, 24, 11)
    A[:, -1] = 0.0
    A[5, -1] = 3.0
    run_case("40x84 shared row", structured(A, 13), 66)


def test_diagonal_problem():
    """A = diag(s), 40 x 40: n_dense = 0 (the memset paths of sweep_n and form_normal_matrix, no row chunks)."""
    A = np.diag(np.random.default_rng(14).uniform(0.5, 2.0, 40))
    run_case("40x40 diagonal", structured(A, 15), 0)


@pytest.mark.parametrize("k", [16, 15])
def test_run_length_threshold(k):
    """A trailing run of exactly 16 singletons is folded, one of 15 is not (n - nd < 16)."""
    A = singleton_tail(40, 60, k, 16, scale=False)
    run_case("40x%d run of %d" % (60 + k, k), structured(A, 17), 60 if k == 16 else 60 + k)


@pytest.mark.parametrize("refine", [(1, 0), (1, 3)])
@pytest.mark.parametrize("m,n,nd", [(64, 128, 96), (1025, 2049, 1537)])
def test_refined_directions(m, n, nd, refine):
    """With iterative refinement (refine = 1, and refine_max = 3) the u / p relations hold for the final v / q and
    every direction call takes at least one step; t then holds A u of the previous step and is not checked."""
    opts = {"refine": refine[0]}
    if refine[1]:
        opts["refine_max"] = refine[1]
    run_case("%dx%d refine=%d refine_max=%d" % (m, n, *refine), lp(m, n, 6), nd, options=opts)
