"""Per-phase references for the single-problem IPM iteration (lpb_blind_start ... lpb_extract_x), with worst-case
rounding bounds.  Pure NumPy.

Every check compares a phase's outputs with a reference computed from the device's own state BEFORE the call (the
buffers `ResidentProblem.debug_read` names), so an error cannot carry over from one iteration into the next and each
bound stays as tight as one kernel's rounding.  A sum or dot of k float64 terms, in any order and with or without FMA
contraction, is within gamma(k) * sum |terms| of the exact value, gamma(k) = k u / (1 - k u), u = 2^-53; the rounding
counts below are read off the kernels in lp_b200/csrc/vec_kernels.cu.  Reference sums run in np.longdouble (x87
extended, u = 2^-64), except the m x m products of the factor check, which run in float64 BLAS with their own
rounding added to the bound.

Each checker returns {check name: largest error / bound}; a bit-for-bit check gives 0 or inf.  A state passes when
every ratio is <= 1 (`worst`).
"""
import numpy as np

LD = np.longdouble
U = 2.0 ** -53
# diagonally scaled bound of the Cholesky factor, |L L^T - M|_ij <= FACTOR_TOL sqrt(M_ii M_jj): the one
# test_gpu_accuracy uses; 7e-15 was measured on a late iterate of C2
FACTOR_TOL = 5e-14
# normwise backward error of the two triangular solves against the device's own factor (2e-17 measured on late C2)
SOLVE_TOL = 1e-15
STATE = ("x", "z", "y", "c", "b", "rD", "rP", "dinv", "dx", "dz", "dy", "u", "p", "t", "W", "M")


def gamma(k):
    return k * U / (1.0 - k * U)


def ratio(err, bound):
    """max |err| / bound; 0 where err == 0, inf where bound == 0 < |err| or err is NaN."""
    err = np.abs(np.asarray(err, dtype=LD)).ravel()
    bound = np.asarray(bound, dtype=LD).ravel() * np.ones_like(err)
    if err.size == 0:
        return 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, LD(0), err / bound)
    r[np.isnan(r)] = np.inf
    return float(r.max())


def exact(a, b):
    """0 when a and b hold the same bits, inf otherwise."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return 0.0 if a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64)) else np.inf


def dot_ratio(val, a, b):
    """A device dot of k terms a_i b_i: within gamma(k + 1) sum |a_i b_i| (k - 1 adds plus the product)."""
    terms = np.asarray(a, dtype=LD) * np.asarray(b, dtype=LD)
    return ratio(LD(val) - terms.sum(), gamma(terms.size + 1) * np.abs(terms).sum())


def norm_ratio(val, r):
    """sqrt of a device sum of k squares: the sum is within gamma(k + 1) relative, the sqrt halves that and rounds
    once more (1 ulp)."""
    s = (np.asarray(r, dtype=LD) ** 2).sum()
    ref = np.sqrt(s)
    bound = LD(0.5 * gamma(r.size + 1) * 1.001) * ref + LD(np.spacing(np.float64(ref)))
    return ratio(LD(val) - ref, bound)


def worst(ratios):
    return max(ratios.values()) if ratios else 0.0


class Ref:
    """The problem side of the reference: the full A (slack columns included, the shortcut is never taken here),
    b, c, c0, and the products the checks need."""

    def __init__(self, A, b, c, c0=0.0, chunk=1 << 16):
        self.A = np.ascontiguousarray(A, dtype=np.float64)
        self.absA = np.abs(self.A)
        self.b, self.c, self.c0 = np.asarray(b, np.float64), np.asarray(c, np.float64), float(c0)
        self.m, self.n = self.A.shape
        self.ldm = (self.m + 15) // 16 * 16
        self.chunk = chunk

    def Aw(self, w):
        """A w in longdouble, in column chunks (the wide case does not fit a longdouble copy of A)."""
        w = np.asarray(w, dtype=LD)
        out = np.zeros(self.m, dtype=LD)
        for j0 in range(0, self.n, self.chunk):
            out += self.A[:, j0:j0 + self.chunk].astype(LD) @ w[j0:j0 + self.chunk]
        return out

    def ATv(self, v):
        v = np.asarray(v, dtype=LD)
        out = np.empty(self.n, dtype=LD)
        for j0 in range(0, self.n, self.chunk):
            out[j0:j0 + self.chunk] = v @ self.A[:, j0:j0 + self.chunk].astype(LD)
        return out

    def absAw(self, w):  # scale vectors: float64 is plenty, they only size the bounds
        return self.absA @ np.abs(np.asarray(w, dtype=np.float64))

    def absATv(self, v):
        return np.abs(np.asarray(v, dtype=np.float64)) @ self.absA

    def L(self, M):
        return np.tril(np.asarray(M).reshape(self.m, self.ldm)[:, :self.m])


# ------------------------------------------------------------------------------------------ phases
def check_blind_start(P, post):
    return {"blind_start x = z = 1, y = 0": max(exact(post["x"], np.ones(P.n)), exact(post["z"], np.ones(P.n)),
                                                exact(post["y"], np.zeros(P.m)))}


def check_residuals(P, pre, post, tau, out):
    """out: dict nrm_rp nrm_rd cx by xz (lpb_residual_scalars)."""
    m, n = P.m, P.n
    x, y, z = pre["x"], pre["y"], pre["z"]
    t, rP, rD = post["t"][:m], post["rP"], post["rD"]
    r = {"residuals x y z unchanged": max(exact(post[k], pre[k]) for k in "xyz")}
    # gemv_n: per-lane chains, a 5-level warp tree, the odd column on lane 0, the slack add: n + 2 roundings at most
    r["residuals t = A x"] = ratio(t - P.Aw(x), gamma(n + 2) * P.absAw(x))
    # resid_p: one product and one difference
    r["residuals rP = b tau - t"] = ratio(rP - (P.b.astype(LD) * LD(tau) - t), 2 * U * (np.abs(P.b) * tau + np.abs(t)))
    # resid_d: A^T y over m rows (row chunks + sum_chunks), then c tau - s - z
    r["residuals rD = c tau - A^T y - z"] = ratio(
        rD - (P.c.astype(LD) * LD(tau) - P.ATv(y) - z),
        gamma(m + 4) * (np.abs(P.c) * tau + P.absATv(y) + np.abs(z)))
    r["residuals scalars"] = max(norm_ratio(out["nrm_rd"], rD), norm_ratio(out["nrm_rp"], rP),
                                 dot_ratio(out["cx"], P.c, x), dot_ratio(out["xz"], x, z), dot_ratio(out["by"], P.b, y))
    return r


def check_form_and_factor(P, pre, post):
    m, n = P.m, P.n
    d = post["dinv"]
    r = {"form dinv = x / z": exact(d, pre["x"] / pre["z"])}
    L = P.L(post["M"])
    Mref = (P.A * d) @ P.A.T                       # float64 BLAS: the doubled gamma below covers its rounding
    S = (P.absA * np.abs(d)) @ P.absA.T
    LLt = L @ L.T
    LLt_abs = np.abs(L) @ np.abs(L).T              # rounding of the float64 L L^T itself
    dm = np.sqrt(np.clip(np.diag(Mref), 0.0, None))
    bound = 2 * gamma(n + 2) * S + gamma(m) * LLt_abs + FACTOR_TOL * np.outer(dm, dm)
    low = np.tril_indices(m)
    r["form L L^T = A D A^T"] = ratio((LLt - Mref)[low], bound[low])
    dg = np.diag(L)
    r["form diag(L) > 0"] = 0.0 if np.all(np.isfinite(dg) & (dg > 0)) else np.inf
    return r


def rhat(pre, din):
    """xs and r1 of rhat_kernel (modes 0 / 1 / 2) exactly, with the scale of the device's rounding error: xs within
    gamma(5) sxs, r1 within gamma(8) sr1."""
    gm = din["gamma"] * din["mu"]                   # host scalars, formed as CudaDev::direction forms them
    a2 = din["alpha"] * din["alpha"]
    s = (1.0 - din["alpha"]) * din["gamma"] * din["mu"]
    x, z = pre["x"].astype(LD), pre["z"].astype(LD)
    xz = x * z
    if not din["corrector"]:
        xs, sxs = LD(gm) - xz, np.abs(xz) + abs(gm)
    else:
        dxdz = pre["dx"].astype(LD) * pre["dz"]
        if din["ip"]:
            xs, sxs = -xz - dxdz * LD(a2) + LD(s), np.abs(xz) + np.abs(dxdz) * a2 + abs(s)
        else:
            xs, sxs = -xz + LD(gm) - dxdz, np.abs(xz) + abs(gm) + np.abs(dxdz)
    r1 = pre["rD"].astype(LD) * LD(din["eta"]) - xs / x
    sr1 = np.abs(pre["rD"]) * abs(din["eta"]) + np.asarray(sxs / np.abs(x), dtype=np.float64)
    return xs, np.asarray(sxs, dtype=np.float64), r1, sr1


def check_direction(P, pre, post, din, out, pred_out=None, refined=False):
    """din: dict corrector ip eta gamma mu alpha; out: dict cu bv cp bq nan_pq.  pred_out: the predictor's out (for
    the corrector).  refined: iterative refinement ran, so t holds A u of its last step and (v, q) no longer solve
    the factor's system; the u / p relations and the scalars still hold."""
    m, n = P.m, P.n
    d = pre["dinv"]
    _, _, r1, sr1 = rhat(pre, din)
    pq = not din["corrector"]
    tag = "corrector" if din["corrector"] else "predictor"
    t0, t1 = post["t"][:m], post["t"][m:]
    v, q = post["W"][:m], post["W"][m:]
    r = {}
    if not refined:
        # gemv_n over dinv * r1 (one more rounding per term) + the slack add; r1 itself is off by gamma(8) sr1
        r[tag + " t0 = A (dinv r1)"] = ratio(t0 - P.Aw(d.astype(LD) * r1), gamma(n + 10) * P.absAw(d * sr1))
        if pq:
            r[tag + " t1 = A (dinv c)"] = ratio(t1 - P.Aw(d.astype(LD) * P.c), gamma(n + 3) * P.absAw(d * P.c))
        L = P.L(pre["M"]).astype(LD)
        rhs = [pre["rP"].astype(LD) * LD(din["eta"]) + t0] + ([P.b.astype(LD) + t1] if pq else [])
        nl2 = np.sum(L * L)
        be = 0.0
        for w, f in zip((v, q), rhs):
            res = L @ (L.T @ w.astype(LD)) - f
            be = max(be, float(np.sqrt(np.sum(res * res)) /
                               (nl2 * np.sqrt(np.sum(w.astype(LD) ** 2)) + np.sqrt(np.sum(f * f)))))
        r[tag + " L L^T (v, q) = rhs"] = be / SOLVE_TOL
    # sym_back: A^T v over m rows (at_dot / TailCols / sum_chunks), minus r1, times dinv
    r[tag + " u = dinv (A^T v - r1)"] = ratio(post["u"] - d.astype(LD) * (P.ATv(v) - r1),
                                             gamma(m + 11) * np.abs(d) * (P.absATv(v) + sr1))
    r[tag + " scalars cu bv"] = max(dot_ratio(out["cu"], P.c, post["u"]), dot_ratio(out["bv"], P.b, v))
    if pq:
        r[tag + " p = dinv (A^T q - c)"] = ratio(post["p"] - d.astype(LD) * (P.ATv(q) - P.c),
                                                 gamma(m + 3) * np.abs(d) * (P.absATv(q) + np.abs(P.c)))
        r[tag + " scalars cp bq nan"] = max(dot_ratio(out["cp"], P.c, post["p"]), dot_ratio(out["bq"], P.b, q),
                                            0.0 if out["nan_pq"] == 0 else np.inf)
    else:
        r[tag + " p q t1 cp bq unchanged"] = max(
            exact(post["p"], pre["p"]), exact(q, pre["W"][m:]), exact(t1, pre["t"][m:]),
            exact([out["cp"], out["bq"]], [pred_out["cp"], pred_out["bq"]]))
    return r


def ratio_test(v, dv):
    """min(1, min over dv_j < 0 of v_j / -dv_j): correctly rounded divisions and an exact min."""
    neg = dv < 0
    return np.float64(min(1.0, np.min(v[neg] / -dv[neg], initial=1.0)))


def check_assemble_delta(P, pre, post, d_tau, axz, din):
    """din: the direction call that produced (u, p, v, q); its rhat mode decides xs."""
    m = P.m
    u, p, v, q = pre["u"], pre["p"], pre["W"][:m], pre["W"][m:]
    x, z = pre["x"], pre["z"]
    dx, dz, dy = post["dx"], post["dz"], post["dy"]
    dt = LD(d_tau)
    r = {"assemble dx = u + p d_tau": ratio(dx - (u.astype(LD) + p * dt), 2 * U * (np.abs(u) + np.abs(p) * abs(d_tau))),
         "assemble dy = v + q d_tau": ratio(dy - (v.astype(LD) + q * dt), 2 * U * (np.abs(v) + np.abs(q) * abs(d_tau)))}
    xs, sxs, _, _ = rhat(pre, din)
    # (xs - z dx) / x: xs off by gamma(5) sxs, then a product, a difference and a division
    r["assemble dz = (xs - z dx) / x"] = ratio(dz - (xs - z.astype(LD) * dx) / x,
                                               gamma(8) * (sxs + np.abs(z * dx)) / np.abs(x))
    r["assemble alpha_x alpha_z exact"] = max(exact(axz[0], ratio_test(x, dx)), exact(axz[1], ratio_test(z, dz)))
    return r


def _two_prod(a, b):
    """p + e == a * b exactly (Dekker's product with Veltkamp's split)."""
    def split(v):
        t = v * 134217729.0  # 2^27 + 1
        hi = t - (t - v)
        return hi, v - hi
    p = a * b
    ah, al = split(a)
    bh, bl = split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def step_exact(v, dv, alpha):
    """v + dv alpha as s + rest, exactly up to 2^-64 |rest|.  A longdouble product alone is not enough: at the step
    of 0.99995 times the ratio-test limit, v + dv alpha is 5e-5 v, and 2^-64 |dv alpha| is several ulps of that."""
    p, e = _two_prod(np.asarray(dv, np.float64), np.float64(alpha))
    s, t = _two_sum(np.asarray(v, np.float64), p)
    return s, t.astype(LD) + e


def check_do_step(P, pre, post, alpha, ip):
    """x, z, y = v + dv alpha (one DFMA: within 1 ulp); with ip, x and z entries below 1 are exactly 1, y is not
    clamped and some entry of it must be below 1 for that to have been tested."""
    r = {}
    worst_ip = 0.0
    for k, clamp in (("x", ip), ("z", ip), ("y", False)):
        s, rest = step_exact(pre[k], pre["d" + k], alpha)
        got = post[k]
        err = (got.astype(LD) - s) - rest
        ulp = np.spacing(np.abs(s))
        if clamp:
            low = s.astype(LD) + rest < 1
            worst_ip = max(worst_ip, exact(got[low], np.ones(int(low.sum()))))
            r["do_step " + k] = ratio(err[~low], ulp[~low])
        else:
            r["do_step " + k] = ratio(err, ulp)
            if ip and k == "y" and not np.any(s.astype(LD) + rest < 1):
                worst_ip = np.inf
    if ip:
        r["do_step ip clamp"] = worst_ip
    return r


def check_extract_x(P, pre, tau, x_out, fun):
    x = pre["x"]
    terms = P.c.astype(LD) * x_out
    return {"extract x = x / tau": exact(x_out, x / tau),
            "extract fun": ratio(LD(fun) - (terms.sum() + LD(P.c0)),
                                 gamma(P.n + 2) * np.abs(terms).sum() + U * abs(P.c0))}
