"""The per-phase checkers of tests/phase_check.py on a CPU-built state: they accept each phase's exact output and
reject each of a set of subtly wrong kernels (a dropped column, slack row, row chunk, K-block or reduction tail, a
swapped slack mapping, a wrong partials pitch or diagonal fold, a wrong ratio-test exclusion, a clamp on y).

The state is a 97 x 229 LP whose last 48 columns are scaled singletons on rows 0..47 (the slack block, values
in [0.5, 0.9] so that s d and s^2 d differ), leaving n_dense = 181 odd, with x and z spanning 1e-8 .. 1e8.  Each
mutation is applied where its dropped term is at least 1e-6 of the checked quantity's scale."""
import numpy as np
import pytest
from scipy.linalg import solve_triangular

from tests import phase_check as pc

LD = np.longdouble
M_ROWS, N_DENSE, N_SLACK = 97, 181, 48
TAU = 1.7
NUM_SMS = 148  # kNumSMs (common.cuh): sets the row chunks of gemv_t


def gemv_t_chunks(m, n):
    """Row chunks of gemv_t_kernel: gemv_t_shape in vec_kernels.cu."""
    cb = -(-(-(-n // 2)) // 128)
    want = min(max(-(-NUM_SMS * 8 // cb), 1), 64)
    rpc = min(max(-(-m // want), 8), 1024)
    nc = -(-m // rpc)
    if nc > 64:
        nc, rpc = -(-m // 1024), 1024
    return nc, rpc


def make_state(m, n_dense, n_slack, seed):
    rng = np.random.default_rng(seed)
    n = n_dense + n_slack
    A = np.zeros((m, n))
    A[:, :n_dense] = rng.standard_normal((m, n_dense))
    s = rng.uniform(0.5, 0.9, n_slack)
    A[np.arange(n_slack), n_dense + np.arange(n_slack)] = s
    x0 = rng.uniform(0.5, 1.5, n)
    b = A @ x0
    c = A.T @ rng.standard_normal(m) + rng.uniform(0.5, 1.5, n)
    P = pc.Ref(A, b, c, c0=0.25)
    st = {"x": np.exp(rng.uniform(-18, 18, n)), "z": np.exp(rng.uniform(-18, 18, n)), "y": rng.standard_normal(m),
          "c": c.copy(), "b": b.copy(), "rD": rng.standard_normal(n), "rP": rng.standard_normal(m),
          "dx": rng.standard_normal(n), "dz": rng.standard_normal(n), "dy": rng.standard_normal(m),
          "u": rng.standard_normal(n), "p": rng.standard_normal(n), "t": rng.standard_normal(2 * m),
          "W": rng.standard_normal(2 * m)}
    st["x"][n_dense - 1] = 1e6      # the last dense column carries weight in A x
    st["dinv"] = st["x"] / st["z"]
    st["M"] = sim_form(P, st)[0]["M"]
    return P, st, s


def f64(a):
    return np.asarray(a, dtype=LD).astype(np.float64)


def dot(a, b):
    return float((np.asarray(a, dtype=LD) * b).sum())


# ----------------------------------------------------------------------------- exact phase outputs
def sim_residuals(P, pre, tau):
    post = {k: v.copy() for k, v in pre.items()}
    m = P.m
    post["t"][:m] = f64(P.Aw(pre["x"]))
    post["rP"] = f64(P.b.astype(LD) * LD(tau) - post["t"][:m])
    post["rD"] = f64(P.c.astype(LD) * LD(tau) - P.ATv(pre["y"]) - pre["z"])
    out = {"nrm_rd": float(np.sqrt((post["rD"].astype(LD) ** 2).sum())),
           "nrm_rp": float(np.sqrt((post["rP"].astype(LD) ** 2).sum())),
           "cx": dot(P.c, pre["x"]), "xz": dot(pre["x"], pre["z"]), "by": dot(P.b, pre["y"])}
    return post, out


def sim_form(P, pre, M_exact=None):
    post = {k: v.copy() for k, v in pre.items()}
    post["dinv"] = d = pre["x"] / pre["z"]
    if M_exact is None:
        M_exact = f64((P.A.astype(LD) * d) @ P.A.T.astype(LD))
    L = np.linalg.cholesky(M_exact)
    Mbuf = np.full((P.m, P.ldm), 7.0)              # the potrf leaves the upper triangle and the padding as it was
    Mbuf[:, :P.m] = L + np.triu(M_exact, 1)
    post["M"] = Mbuf.ravel()
    return post, None


def sim_direction(P, pre, din, pred_out=None):
    post = {k: v.copy() for k, v in pre.items()}
    m, d = P.m, pre["dinv"]
    _, _, r1, _ = pc.rhat(pre, din)
    r1 = f64(r1)
    pq = not din["corrector"]
    L = P.L(pre["M"])
    post["t"][:m] = f64(P.Aw(d.astype(LD) * r1))
    rhs = [f64(pre["rP"].astype(LD) * LD(din["eta"]) + post["t"][:m])]
    if pq:
        post["t"][m:] = f64(P.Aw(d.astype(LD) * P.c))
        rhs.append(f64(P.b.astype(LD) + post["t"][m:]))
    for k, f in enumerate(rhs):
        post["W"][k * m:(k + 1) * m] = solve_triangular(L.T, solve_triangular(L, f, lower=True), lower=False)
    v, q = post["W"][:m], post["W"][m:]
    post["u"] = f64(d.astype(LD) * (P.ATv(v) - r1))
    out = {"cu": dot(P.c, post["u"]), "bv": dot(P.b, v)}
    if pq:
        post["p"] = f64(d.astype(LD) * (P.ATv(q) - P.c))
        out.update(cp=dot(P.c, post["p"]), bq=dot(P.b, q), nan_pq=0)
    else:
        out.update(cp=pred_out["cp"], bq=pred_out["bq"], nan_pq=0)
    return post, out


def sim_assemble(P, pre, d_tau, din):
    post = {k: v.copy() for k, v in pre.items()}
    m = P.m
    post["dx"] = f64(pre["u"].astype(LD) + pre["p"] * LD(d_tau))
    post["dy"] = f64(pre["W"][:m].astype(LD) + pre["W"][m:] * LD(d_tau))
    xs, _, _, _ = pc.rhat(pre, din)
    post["dz"] = f64((xs - pre["z"].astype(LD) * post["dx"]) / pre["x"])
    axz = [pc.ratio_test(pre["x"], post["dx"]), pc.ratio_test(pre["z"], post["dz"])]
    return post, axz


def sim_step(P, pre, alpha, ip):
    post = {k: v.copy() for k, v in pre.items()}
    for k, clamp in (("x", ip), ("z", ip), ("y", False)):
        s, rest = pc.step_exact(pre[k], pre["d" + k], alpha)
        post[k] = f64(s.astype(LD) + rest)
        if clamp:
            post[k] = np.maximum(post[k], 1.0)
    return post


def sim_extract(P, pre, tau):
    x_out = pre["x"] / tau
    return x_out, float((P.c.astype(LD) * x_out).sum() + LD(P.c0))


# ----------------------------------------------------------------------------- fixtures
PRED = dict(corrector=0, ip=0, eta=1.0, gamma=0.0, mu=3.0, alpha=0.0)
CORR_IP = dict(corrector=1, ip=1, eta=1.0, gamma=10.0, mu=3.0, alpha=0.6)
CORR = dict(corrector=1, ip=0, eta=0.9, gamma=0.1, mu=3.0, alpha=0.6)


@pytest.fixture(scope="module")
def state():
    return make_state(M_ROWS, N_DENSE, N_SLACK, seed=5)


def accepts(r):
    assert pc.worst(r) <= 1.0, r


def rejects(r, key):
    assert r[key] > 1.0, r


def significant(mut, ref, scale):
    """The mutation moves some entry by at least 1e-6 of that entry's scale."""
    d = np.abs(np.asarray(mut, dtype=np.float64) - np.asarray(ref, dtype=np.float64)) / np.asarray(scale)
    assert np.nanmax(d) >= 1e-6


# ----------------------------------------------------------------------------- acceptance
def test_exact_outputs_pass_every_check(state):
    P, pre, _ = state
    blind = {k: v.copy() for k, v in pre.items()}
    blind["x"][:], blind["z"][:], blind["y"][:] = 1.0, 1.0, 0.0
    accepts(pc.check_blind_start(P, blind))
    post, out = sim_residuals(P, pre, TAU)
    accepts(pc.check_residuals(P, pre, post, TAU, out))
    post, _ = sim_form(P, pre)
    accepts(pc.check_form_and_factor(P, pre, post))
    pred, pout = sim_direction(P, pre, PRED)
    accepts(pc.check_direction(P, pre, pred, PRED, pout))
    for din in (CORR_IP, CORR):
        post, out = sim_direction(P, pred, din, pout)
        accepts(pc.check_direction(P, pred, post, din, out, pred_out=pout))
        post2, axz = sim_assemble(P, post, -0.3, din)
        accepts(pc.check_assemble_delta(P, post, post2, -0.3, axz, din))
    for ip in (True, False):
        accepts(pc.check_do_step(P, pre, sim_step(P, pre, 0.7, ip), 0.7, ip))
    # the damped step of the iteration, 0.99995 of the ratio-test limit: x + dx alpha cancels to 5e-5 x
    alpha = 0.99995 * min(pc.ratio_test(pre["x"], pre["dx"]), pc.ratio_test(pre["z"], pre["dz"]))
    post = sim_step(P, pre, alpha, False)
    accepts(pc.check_do_step(P, pre, post, alpha, False))
    j = int(np.argmin(post["x"] / pre["x"]))
    bad = dict(post, x=post["x"].copy())
    bad["x"][j] = np.nextafter(np.nextafter(post["x"][j], 0.0), 0.0)   # two ulps off where it cancels
    rejects(pc.check_do_step(P, pre, bad, alpha, False), "do_step x")
    x_out, fun = sim_extract(P, pre, TAU)
    accepts(pc.check_extract_x(P, pre, TAU, x_out, fun))


# ----------------------------------------------------------------------------- rejection
def test_residuals_rejects_dropped_terms(state):
    P, pre, s = state
    m, nd = P.m, N_DENSE
    post, out = sim_residuals(P, pre, TAU)
    x, y = pre["x"], pre["y"]
    scale_t = P.absAw(x)
    # the last (odd) dense column left out of A x
    bad = {k: v.copy() for k, v in post.items()}
    bad["t"][:m] -= P.A[:, nd - 1] * x[nd - 1]
    significant(bad["t"][:m], post["t"][:m], scale_t)
    rejects(pc.check_residuals(P, pre, bad, TAU, out), "residuals t = A x")
    # one slack row's s w left out of A x
    share = s * x[nd:] / scale_t[:N_SLACK]
    r = int(np.argmax(share))
    bad = {k: v.copy() for k, v in post.items()}
    bad["t"][r] -= s[r] * x[nd + r]
    significant(bad["t"][:m], post["t"][:m], scale_t)
    rejects(pc.check_residuals(P, pre, bad, TAU, out), "residuals t = A x")
    # the last row chunk of gemv_t left out of A^T y
    nc, rpc = gemv_t_chunks(m, nd)
    rows = slice((nc - 1) * rpc, m)
    bad = {k: v.copy() for k, v in post.items()}
    bad["rD"][:nd] += y[rows] @ P.A[rows, :nd]
    significant(bad["rD"], post["rD"], np.abs(P.c) * TAU + P.absATv(y) + np.abs(pre["z"]))
    rejects(pc.check_residuals(P, pre, bad, TAU, out), "residuals rD = c tau - A^T y - z")


def test_form_and_factor_rejects_wrong_normal_matrix(state):
    P, pre, s = state
    m, nd = P.m, N_DENSE
    d = pre["x"] / pre["z"]
    M = f64((P.A.astype(LD) * d) @ P.A.T.astype(LD))
    S = (P.absA * d) @ P.absA.T
    rows = np.arange(N_SLACK)
    fold = s ** 2 * d[nd + rows]
    # the slack fold with s d instead of s^2 d
    Mb = M.copy()
    Mb[rows, rows] += s * d[nd + rows] - fold
    significant(np.diag(Mb), np.diag(M), np.diag(S))
    rejects(pc.check_form_and_factor(P, pre, sim_form(P, pre, Mb)[0]), "form L L^T = A D A^T")
    # the fold missing for one row: the one where it is smallest but still above 1e-6 of M_rr
    share = fold / np.diag(S)[rows]
    r = int(np.argmin(np.where(share >= 1e-6, share, np.inf)))
    Mb = M.copy()
    Mb[r, r] -= fold[r]
    significant(np.diag(Mb), np.diag(M), np.diag(S))
    rejects(pc.check_form_and_factor(P, pre, sim_form(P, pre, Mb)[0]), "form L L^T = A D A^T")
    # one 16-column K-block of the dense part left out: the block with the largest share of some M_ii
    shares = [np.max(((P.A[:, k:k + 16] ** 2) @ d[k:k + 16]) / np.diag(S)) for k in range(0, nd - 15, 16)]
    k = 16 * int(np.argmax(shares))
    Mb = M - (P.A[:, k:k + 16] * d[k:k + 16]) @ P.A[:, k:k + 16].T
    significant(np.diag(Mb), np.diag(M), np.diag(S))
    rejects(pc.check_form_and_factor(P, pre, sim_form(P, pre, Mb)[0]), "form L L^T = A D A^T")
    # dinv one ulp off in one entry
    post, _ = sim_form(P, pre)
    post["dinv"][7] = np.nextafter(post["dinv"][7], np.inf)
    rejects(pc.check_form_and_factor(P, pre, post), "form dinv = x / z")


def test_direction_rejects_wrong_transpose_product(state):
    P, pre, s = state
    m, nd, n = P.m, N_DENSE, P.n
    post, out = sim_direction(P, pre, PRED)
    d, v, q = pre["dinv"], post["W"][:m], post["W"][m:]
    _, _, r1, sr1 = pc.rhat(pre, PRED)
    r1 = f64(r1)
    scale_u = np.abs(d) * (P.absATv(v) + sr1)
    # two slack columns' col_row swapped: pick the pair whose swap moves u the most
    j = nd + np.arange(N_SLACK)
    moved = np.abs(s * (v[:N_SLACK] - v[np.roll(np.arange(N_SLACK), 1)]) * d[j]) / scale_u[j]
    a = int(np.argmax(moved))
    b = (a - 1) % N_SLACK
    bad = {k: v_.copy() for k, v_ in post.items()}
    bad["u"][nd + a] = d[nd + a] * (s[a] * v[b] - r1[nd + a])
    bad["u"][nd + b] = d[nd + b] * (s[b] * v[a] - r1[nd + b])
    significant(bad["u"], post["u"], scale_u)
    rejects(pc.check_direction(P, pre, bad, PRED, out), "predictor u = dinv (A^T v - r1)")
    # the partials of A^T (v, q) read with pitch round_up(n, 2) instead of round_up(n_dense, 2)
    nc, rpc = gemv_t_chunks(m, nd)
    pitch, wrong = nd + (nd & 1), n + (n & 1)
    buf = np.zeros(max(64, -(-m // 1024)) * 2 * wrong)        # gemv_t_partials_doubles(m, n)
    for ch in range(nc):
        rows = slice(ch * rpc, min(m, (ch + 1) * rpc))
        for k, w in enumerate((v, q)):
            buf[(ch * 2 + k) * pitch:(ch * 2 + k) * pitch + nd] = w[rows] @ P.A[rows, :nd]
    atv = np.array([sum(buf[(ch * 2) * wrong + jj] for ch in range(nc)) for jj in range(nd)])
    bad = {k: v_.copy() for k, v_ in post.items()}
    bad["u"][:nd] = d[:nd] * (atv - r1[:nd])
    significant(bad["u"], post["u"], scale_u)
    rejects(pc.check_direction(P, pre, bad, PRED, out), "predictor u = dinv (A^T v - r1)")
    # the last dense column of A (dinv r1) left out
    bad = {k: v_.copy() for k, v_ in post.items()}
    bad["t"][:m] -= P.A[:, nd - 1] * d[nd - 1] * r1[nd - 1]
    significant(bad["t"][:m], post["t"][:m], P.absAw(d * sr1))
    rejects(pc.check_direction(P, pre, bad, PRED, out), "predictor t0 = A (dinv r1)")
    # (v, q) off by 1e-12 relative: no longer a solve with the device's factor
    bad = {k: v_.copy() for k, v_ in post.items()}
    bad["W"][3] *= 1 + 1e-12
    rejects(pc.check_direction(P, pre, bad, PRED, out), "predictor L L^T (v, q) = rhs")
    # corrector: p must stay as the predictor left it
    cpost, cout = sim_direction(P, post, CORR, out)
    cpost["p"][0] = np.nextafter(cpost["p"][0], np.inf)
    rejects(pc.check_direction(P, post, cpost, CORR, cout, pred_out=out), "corrector p q t1 cp bq unchanged")


def test_assemble_delta_rejects_wrong_ratio_test(state):
    P, pre, _ = state
    pre = {k: v.copy() for k, v in pre.items()}
    pre["u"][-1], pre["p"][-1] = -1e12 * pre["x"][-1], 0.0        # the last entry sets alpha_x
    post, axz = sim_assemble(P, pre, -0.3, PRED)
    x, dx = pre["x"], post["dx"]
    assert pc.ratio_test(x[:-1], dx[:-1]) != axz[0]
    rejects(pc.check_assemble_delta(P, pre, post, -0.3, [pc.ratio_test(x[:-1], dx[:-1]), axz[1]], PRED),
            "assemble alpha_x alpha_z exact")
    let_in = np.float64(min(1.0, np.min(x / -dx)))                 # entries with dx >= 0 in the min
    assert let_in != axz[0]
    rejects(pc.check_assemble_delta(P, pre, post, -0.3, [let_in, axz[1]], PRED), "assemble alpha_x alpha_z exact")
    bad = {k: v.copy() for k, v in post.items()}
    bad["dz"][5] *= 1 + 1e-12
    rejects(pc.check_assemble_delta(P, pre, bad, -0.3, axz, PRED), "assemble dz = (xs - z dx) / x")


def test_do_step_rejects_clamped_y(state):
    P, pre, _ = state
    post = sim_step(P, pre, 0.7, True)
    assert np.any(post["y"] < 1)
    bad = {k: v.copy() for k, v in post.items()}
    bad["y"] = np.maximum(bad["y"], 1.0)
    rejects(pc.check_do_step(P, pre, bad, 0.7, True), "do_step y")
    # without any y below 1 the ip case has not tested the missing clamp
    flat = {k: v.copy() for k, v in pre.items()}
    flat["y"][:], flat["dy"][:] = 2.0, 0.0
    rejects(pc.check_do_step(P, flat, sim_step(P, flat, 0.7, True), 0.7, True), "do_step ip clamp")


def test_blind_start_and_extract_reject_one_ulp(state):
    P, pre, _ = state
    blind = {k: v.copy() for k, v in pre.items()}
    blind["x"][:], blind["z"][:], blind["y"][:] = 1.0, 1.0, 0.0
    blind["x"][-1] = np.nextafter(1.0, 2.0)
    rejects(pc.check_blind_start(P, blind), "blind_start x = z = 1, y = 0")
    x_out, fun = sim_extract(P, pre, TAU)
    x_out[4] = np.nextafter(x_out[4], 0.0)
    rejects(pc.check_extract_x(P, pre, TAU, x_out, fun), "extract x = x / tau")


def test_reductions_reject_a_dropped_tail_of_1024():
    """A wide state (8 x 3000) so that a reduction runs over more than 1024 elements: the last 1024 left out."""
    P, pre, _ = make_state(8, 2996, 4, seed=9)
    pre["x"] = np.exp(np.random.default_rng(1).uniform(-2, 2, P.n))   # no single entry dominates the sums
    n = P.n
    x_out, fun = sim_extract(P, pre, TAU)
    accepts(pc.check_extract_x(P, pre, TAU, x_out, fun))
    short = float((P.c[:n - 1024].astype(LD) * x_out[:n - 1024]).sum() + LD(P.c0))
    rejects(pc.check_extract_x(P, pre, TAU, x_out, short), "extract fun")
    post, out = sim_residuals(P, pre, TAU)
    accepts(pc.check_residuals(P, pre, post, TAU, out))
    bad = dict(out, cx=float((P.c[:n - 1024].astype(LD) * pre["x"][:n - 1024]).sum()))
    rejects(pc.check_residuals(P, pre, post, TAU, bad), "residuals scalars")
    bad = dict(out, nrm_rd=float(np.sqrt((post["rD"][:n - 1024].astype(LD) ** 2).sum())))
    rejects(pc.check_residuals(P, pre, post, TAU, bad), "residuals scalars")
