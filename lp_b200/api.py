"""Python mirror of the reference's public API over the C ABI (include/lpb200.h).

Names, argument meaning and error behaviour follow /root/reference/src:
  Problem / ProblemBuilder      linear_program.rs:24-169
  InteriorPoint(+Builder)       solvers/interior_point/mod.rs:41-197
  EquationSolverType            solvers/interior_point/newton_equations.rs:36-46
  Solver / OptimizeResult       solvers/mod.rs:12-49
  LinearProgramError variants   error.rs:7-29
Rust `Result<T, LinearProgramError>` becomes "return T or raise the variant's exception".
All numerical work happens inside liblpb200.so on the GPU; this file only marshals arrays.
"""
from __future__ import annotations

import ctypes as C
import os
import enum
from typing import Optional

import numpy as np

from . import _ffi


# --------------------------------------------------------------------------- errors (error.rs:7-29)
class LinearProgramError(Exception):
    code = None

    def __init__(self, msg: Optional[str] = None):
        super().__init__(msg if msg is not None else (_MESSAGES.get(self.code, "")))


class Unconstrained(LinearProgramError):
    code = _ffi.LPB_ERR_UNCONSTRAINED


class NumericalProblem(LinearProgramError):
    code = _ffi.LPB_ERR_NUMERICAL_PROBLEM


class InvalidParameter(LinearProgramError):
    code = _ffi.LPB_ERR_INVALID_PARAMETER


class IncompatibleInputDimensions(LinearProgramError):
    code = _ffi.LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS


class Infeasible(LinearProgramError):
    code = _ffi.LPB_ERR_INFEASIBLE


class Unbounded(LinearProgramError):
    code = _ffi.LPB_ERR_UNBOUNDED


class IterationLimitExceeded(LinearProgramError):
    """Carries the best x / tau in SLACK form, like the reference (interior_point/mod.rs:237-239)."""
    code = _ffi.LPB_ERR_ITERATION_LIMIT_EXCEEDED

    def __init__(self, x):
        super().__init__()
        self.x = x


class DeviceError(RuntimeError):
    """CUDA / NCCL / argument failures (negative lpb codes): no reference counterpart."""

    def __init__(self, code, detail=""):
        super().__init__("lpb error %d: %s" % (code, detail))
        self.code = code


_MESSAGES = {
    _ffi.LPB_ERR_UNCONSTRAINED: "The problem is unconstrained, meaning the solution is the all-zeros vector if `c` "
                                "is nonnegative, or unbounded otherwise.",
    _ffi.LPB_ERR_NUMERICAL_PROBLEM: "The solver encountered numerical problems it could not recover from. Likely "
                                    "causes are linearly dependent constraints or variables whose scale differs by "
                                    "multiple orders of magnitude.",
    _ffi.LPB_ERR_INVALID_PARAMETER: "A parameter was set to an invalid value",
    _ffi.LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS: "The dimensions of your cost- and constraint arrays do not align.",
    _ffi.LPB_ERR_INFEASIBLE: "The solver finished successfully, it appears that the problem is infeasible.",
    _ffi.LPB_ERR_UNBOUNDED: "The solver finished successfully, it appears that your problem is unbounded.",
    _ffi.LPB_ERR_ITERATION_LIMIT_EXCEEDED: "The solver failed to converge within the maximum number of iterations.",
}

_BY_CODE = {cls.code: cls for cls in (Unconstrained, NumericalProblem, InvalidParameter,
                                      IncompatibleInputDimensions, Infeasible, Unbounded)}


def _error_for(code: int, x=None) -> Exception:
    """The exception a non-zero lpb status stands for."""
    if code == _ffi.LPB_ERR_ITERATION_LIMIT_EXCEEDED:
        return IterationLimitExceeded(x)
    if code in _BY_CODE:
        return _BY_CODE[code]()
    if code == _ffi.LPB_ERR_UNSUPPORTED:
        return InvalidParameter("unsupported on the B200 path: " + _ffi.last_error())
    return DeviceError(code, _ffi.last_error())


def _raise_for(code: int, x=None):
    if code != _ffi.LPB_OK:
        raise _error_for(code, x)


# --------------------------------------------------------------------------- host buffers
class _PinnedAlloc:
    """Owner of one page-locked host allocation (lpb_host_alloc); freed when the last array over it goes away."""

    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        if getattr(self, "ptr", None) is not None:
            try:
                _ffi.load().lpb_host_free(self.ptr)
            except Exception:
                pass
            self.ptr = None


class _PinnedArray(np.ndarray):
    """ndarray over a pinned host allocation.  The keep-alive hangs on the ctypes buffer at the bottom of the
    `.base` chain, so EVERY view of the memory -- slices, reshapes, `.view(np.ndarray)` -- keeps the allocation
    alive; `_lpb_host` only makes the owner visible for debugging."""
    _lpb_host = None


class _HostBuffer:
    """A float64 array in pinned host memory when a CUDA device is visible (uploads at PCIe rate),
    else ordinary NumPy memory (building a Problem needs no GPU, exactly like the reference).
    `array` and every view derived from it own a reference to the allocation: a view that outlives the
    _HostBuffer (e.g. `A = build().A()` returned from a helper) never points at freed memory."""

    def __init__(self, shape):
        self.shape = tuple(int(s) for s in shape)
        nbytes = int(np.prod(self.shape)) * 8
        lib = _ffi.load()
        p = C.c_void_p()
        if nbytes > 0 and lib.lpb_device_count() > 0 and lib.lpb_host_alloc(C.byref(p), nbytes) == _ffi.LPB_OK:
            buf = (C.c_double * (nbytes // 8)).from_address(p.value)
            buf._lpb_alloc = _PinnedAlloc(p)  # the ctypes object is the base of every array view below
            arr = np.frombuffer(buf, dtype=np.float64).reshape(self.shape).view(_PinnedArray)
            arr._lpb_host = buf._lpb_alloc
            self.array = arr
        else:
            self.array = np.zeros(self.shape, dtype=np.float64)

    @property
    def pinned(self) -> bool:
        return isinstance(self.array, _PinnedArray)


def pinned_empty(shape) -> np.ndarray:
    """A float64 array in pinned (page-locked) host memory when a CUDA device is visible -- inputs built in
    it upload at PCIe rate (`solve_batched`, `Problem` buffers) -- else an ordinary NumPy array."""
    return _HostBuffer(shape).array


def _as_f64(a, ndim):
    arr = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if arr.ndim != ndim:
        raise IncompatibleInputDimensions()
    return arr


# --------------------------------------------------------------------------- Problem (linear_program.rs)
class Problem:
    """A linear program in slack form: min c'x st A x == b, x >= 0 (linear_program.rs:24-30)."""

    def __init__(self, A_buf, b_buf, c_buf, c0: float, n_slack: int, dtype=np.float64):
        self._A, self._b, self._c = A_buf, b_buf, c_buf
        self._c0 = float(c0)
        self._n_slack = int(n_slack)
        # `Problem<f32>` of the reference (float.rs:43): the slack form is held and solved in FP64 on the B200
        # path (inputs are widened at build); only the RESULT is narrowed back to the caller's float type.
        self._dtype = np.dtype(dtype)

    def dtype(self) -> np.dtype:
        return self._dtype

    @staticmethod
    def target(c) -> "ProblemBuilder":
        """Problem::target (linear_program.rs:37-39)."""
        return ProblemBuilder(c)

    def A(self) -> np.ndarray:
        return self._A.array

    def b(self) -> np.ndarray:
        return self._b.array

    def c(self) -> np.ndarray:
        return self._c.array

    def c0(self) -> float:
        return self._c0

    def n_slack(self) -> int:
        return self._n_slack

    def denormalize_target(self, x_slack) -> float:
        return float(self.c().dot(x_slack) + self._c0)  # linear_program.rs:61-63

    def denormalize_x(self, x_slack) -> np.ndarray:
        return np.array(x_slack[: len(x_slack) - self._n_slack])  # linear_program.rs:65-69


class ProblemBuilder:
    """ProblemBuilder (linear_program.rs:73-169)."""

    def __init__(self, c):
        self._c = c
        self._ub = None
        self._eq = None

    def ub(self, A, b) -> "ProblemBuilder":
        self._ub = (A, b)
        return self

    def eq(self, A, b) -> "ProblemBuilder":
        self._eq = (A, b)
        return self

    def build(self) -> Problem:
        """Validate + convert to slack form [[A_ub, I], [A_eq, 0]] (linear_program.rs:125-169)."""
        lib = _ffi.load()
        given = [self._c] + [a for pair in (self._ub, self._eq) if pair is not None for a in pair]
        all_f32 = all(isinstance(a, np.ndarray) and a.dtype == np.float32 for a in given)
        c = _as_f64(self._c, 1)
        n_c = c.shape[0]

        def unpack(pair):
            if pair is None:  # (0, n) placeholders, linear_program.rs:127-130
                return np.zeros((0, n_c)), np.zeros(0)
            return _as_f64(pair[0], 2), _as_f64(pair[1], 1)

        A_ub, b_ub = unpack(self._ub)
        A_eq, b_eq = unpack(self._eq)
        m = C.c_int64()
        n = C.c_int64()
        ns = C.c_int64()
        rc = lib.lpb_slack_dims(n_c, A_ub.shape[0], A_ub.shape[1], b_ub.shape[0], A_eq.shape[0], A_eq.shape[1],
                                b_eq.shape[0], C.byref(m), C.byref(n), C.byref(ns))
        _raise_for(rc)
        A_buf = _HostBuffer((m.value, n.value))
        b_buf = _HostBuffer((m.value,))
        c_buf = _HostBuffer((n.value,))
        rc = lib.lpb_build_slack_form(
            c.ctypes.data, n_c,
            A_ub.ctypes.data if A_ub.size else None, A_ub.shape[0], A_ub.shape[1], A_ub.shape[1],
            b_ub.ctypes.data if b_ub.size else None, b_ub.shape[0],
            A_eq.ctypes.data if A_eq.size else None, A_eq.shape[0], A_eq.shape[1], A_eq.shape[1],
            b_eq.ctypes.data if b_eq.size else None, b_eq.shape[0],
            A_buf.array.ctypes.data, n.value, b_buf.array.ctypes.data, c_buf.array.ctypes.data)
        _raise_for(rc)
        return Problem(A_buf, b_buf, c_buf, 0.0, ns.value, np.float32 if all_f32 else np.float64)


# --------------------------------------------------------------------------- solver config
class EquationSolverType(enum.IntEnum):
    """newton_equations.rs:36-46.  Only Cholesky runs on the B200 path."""
    Cholesky = _ffi.LPB_SOLVER_CHOLESKY
    Inverse = _ffi.LPB_SOLVER_INVERSE
    LeastSquares = _ffi.LPB_SOLVER_LEAST_SQUARES


class OptimizeResult:
    """solvers/mod.rs:19-49."""

    def __init__(self, x, fun, iteration):
        self._x, self._fun, self._iteration = x, float(fun), int(iteration)

    def x(self) -> np.ndarray:
        return self._x

    def fun(self) -> float:
        return self._fun

    def iteration(self) -> int:
        return self._iteration


class Solver:
    """solvers/mod.rs:12-16."""

    def solve(self, problem: Problem) -> OptimizeResult:  # pragma: no cover - interface
        raise NotImplementedError


class InteriorPointBuilder:
    """interior_point/mod.rs:41-138."""

    def __init__(self):
        o = _ffi.lpb_options()
        _ffi.load().lpb_options_default(C.byref(o))  # mod.rs:51-60
        self._o = o

    def tol(self, tol: float) -> "InteriorPointBuilder":
        self._o.tol = float(tol)
        return self

    def disp(self, disp: bool) -> "InteriorPointBuilder":
        self._o.disp = 1 if disp else 0
        return self

    def ip(self, ip: bool) -> "InteriorPointBuilder":
        self._o.ip = 1 if ip else 0
        return self

    def solver_type(self, solver_type: EquationSolverType) -> "InteriorPointBuilder":
        self._o.solver_type = int(solver_type)
        return self

    def alpha0(self, alpha0: float) -> "InteriorPointBuilder":
        self._o.alpha0 = float(alpha0)
        return self

    def max_iter(self, max_iter: int) -> "InteriorPointBuilder":
        self._o.max_iter = int(max_iter)
        return self

    def build(self) -> "InteriorPoint":
        """mod.rs:118-137: InvalidParameter unless 0 < alpha0 < 1 and tol > 0."""
        o = self._o
        if o.alpha0 <= 0.0 or o.alpha0 >= 1.0:
            raise InvalidParameter("A parameter was set to an invalid value: Alpha0 must be between 0 and 1 (exclusive)")
        if o.tol <= 0.0:
            raise InvalidParameter("A parameter was set to an invalid value: The tolerance must be nonnegative.")
        return InteriorPoint(o)


class InteriorPoint(Solver):
    """interior_point/mod.rs:145-197."""

    def __init__(self, opts: _ffi.lpb_options):
        self._o = _ffi.lpb_options()
        C.memmove(C.byref(self._o), C.byref(opts), C.sizeof(_ffi.lpb_options))

    @staticmethod
    def default() -> "InteriorPoint":
        return InteriorPointBuilder().build()  # mod.rs:154-159

    @staticmethod
    def custom() -> InteriorPointBuilder:
        return InteriorPointBuilder()  # mod.rs:195-197

    def _key(self):
        o = self._o
        return (o.tol, o.disp, o.ip, o.solver_type, o.alpha0, o.max_iter)

    def __eq__(self, other):  # #[derive(PartialEq)] mod.rs:140
        return isinstance(other, InteriorPoint) and self._key() == other._key()

    def __hash__(self):
        return hash(self._key())

    def solve(self, problem: Problem) -> OptimizeResult:
        """Solver::solve (mod.rs:161-169): upload, run the loop on the GPU, de-normalise.

        The device context (A, M, the vectors, the factorisation workspaces: ~1.6x the size of A) is kept per host
        thread between calls and re-used when the next problem has the same shape -- the call then costs the H2D
        of A, b, c, the solve and the D2H of x, no cudaMalloc / cudaFree.  `release_cached_contexts()` frees it."""
        cache = _solve_cache.__dict__
        rp = cache.get("rp")
        A = problem.A()
        if rp is not None and rp.handle is not None and (rp.m, rp.n) == A.shape:
            rp.reupload(problem)
        else:
            if rp is not None:
                rp.close()
            cache["rp"] = None
            rp = ResidentProblem(problem)
            cache["rp"] = rp
        rp._problem = None        # uploads are synchronous: the cache must not pin the caller's host buffers
        try:
            return self.solve_resident(rp)
        except DeviceError:
            rp.close()            # a context that reported a CUDA / NCCL failure is not re-used
            cache["rp"] = None
            raise

    def solve_resident(self, rp: "ResidentProblem") -> OptimizeResult:
        lib = _ffi.load()
        n = rp.n
        x_slack = np.empty(n, dtype=np.float64)
        fun = C.c_double()
        it = C.c_int64()
        rc = lib.lpb_solve(rp.handle, C.byref(self._o), x_slack.ctypes.data, C.byref(fun), C.byref(it))
        rp.last_iterations = it.value
        if rc in (_ffi.LPB_OK, _ffi.LPB_ERR_ITERATION_LIMIT_EXCEEDED):
            x_slack = rp.gather_x(x_slack)
        _raise_for(rc, x_slack)
        x = np.array(x_slack[: len(x_slack) - rp.n_slack])  # denormalize_x_into, linear_program.rs:65-69
        dt = getattr(rp, "result_dtype", np.dtype(np.float64))
        if dt != np.float64:  # Problem<f32>: FP64 arithmetic, result narrowed to the caller's float type
            return OptimizeResult(x.astype(dt), float(dt.type(fun.value)), it.value)
        return OptimizeResult(x, fun.value, it.value)

    def solve_all(self, problems) -> list:
        """The batched counterpart of `solve`: a list of Problems of any shapes, solved in one call.

        Element i is what `self.solve(problems[i])` returns, except that a LinearProgramError is returned as the
        exception instance instead of raised.  Problems inside `solve_many`'s limits (m <= 128 and the shared memory
        their shape needs) go through one `lpb_solve_many_ragged` call: each gets its own slack structure and kernel,
        and its bits do not depend on the rest of the list.  The others are solved one by one with `solve`.  The
        problems are packed into a page-locked staging buffer kept per host thread (`release_cached_contexts()`
        frees it)."""
        problems = list(problems)
        out = [None] * len(problems)
        if not problems:
            return out
        lib = _ffi.load()
        many = [i for i, p in enumerate(problems) if lib.lpb_solve_many_check(*p.A().shape) == _ffi.LPB_OK]
        if many:
            pk = _pack_problems([problems[i] for i in many], _staging)
            batch = len(many)
            rc = lib.lpb_solve_many_ragged(batch, pk.m.ctypes.data, pk.n.ctypes.data, pk.A.ctypes.data,
                                           pk.b.ctypes.data, pk.c.ctypes.data, C.byref(self._o), pk.x.ctypes.data,
                                           pk.fun.ctypes.data, pk.it.ctypes.data, pk.st.ctypes.data,
                                           _ffi.LPB_MEM_HOST, None)
            _raise_for(rc)
            for k, i in enumerate(many):
                p = problems[i]
                x_slack = np.array(pk.x[pk.c_off[k]: pk.c_off[k] + pk.n[k]])
                st = int(pk.st[k])
                if st != _ffi.LPB_OK:
                    out[i] = _error_for(st, x_slack)
                    continue
                x = x_slack[: len(x_slack) - p.n_slack()]
                fun = float(pk.fun[k]) + p.c0()  # the kernels leave c0 out: c.x_slack + c0, linear_program.rs:61-63
                dt = p.dtype()
                if dt != np.float64:
                    out[i] = OptimizeResult(x.astype(dt), float(dt.type(fun)), int(pk.it[k]))
                else:
                    out[i] = OptimizeResult(x, fun, int(pk.it[k]))
        for i, p in enumerate(problems):
            if out[i] is None:
                try:
                    out[i] = self.solve(p)
                except LinearProgramError as e:
                    out[i] = e
        return out


class _Packed:
    """A list of slack-form problems packed for lpb_solve_many_ragged: problem k's A (row-major m[k] x n[k]) at
    a_off[k], b at b_off[k], c and x at c_off[k]; fun / it / st hold one entry per problem."""


def _pack_problems(problems, alloc=np.empty) -> _Packed:
    """Pack `problems` back to back into one float64 buffer from `alloc(count)` (inputs, then outputs)."""
    pk = _Packed()
    shapes = np.array([p.A().shape for p in problems], dtype=np.int64).reshape(-1, 2)
    pk.m, pk.n = np.ascontiguousarray(shapes[:, 0]), np.ascontiguousarray(shapes[:, 1])
    sizes = pk.m * pk.n
    pk.a_off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    pk.b_off = np.concatenate([[0], np.cumsum(pk.m)[:-1]]).astype(np.int64)
    pk.c_off = np.concatenate([[0], np.cumsum(pk.n)[:-1]]).astype(np.int64)
    na, nb, nc, k = int(sizes.sum()), int(pk.m.sum()), int(pk.n.sum()), len(problems)
    buf = alloc(na + nb + 2 * nc + 3 * k)
    cuts = np.cumsum([0, na, nb, nc, nc, k, k, k])
    pk.A, pk.b, pk.c, pk.x = (buf[cuts[i]: cuts[i + 1]] for i in range(4))
    pk.fun = buf[cuts[4]: cuts[5]]
    pk.it = buf[cuts[5]: cuts[6]].view(np.int64)
    pk.st = buf[cuts[6]: cuts[7]].view(np.int32)[:k]
    for i, p in enumerate(problems):
        pk.A[pk.a_off[i]: pk.a_off[i] + sizes[i]] = p.A().reshape(-1)
        pk.b[pk.b_off[i]: pk.b_off[i] + pk.m[i]] = p.b()
        pk.c[pk.c_off[i]: pk.c_off[i] + pk.n[i]] = p.c()
    return pk


_solve_cache = __import__("threading").local()


def _staging(count: int) -> np.ndarray:
    """`count` float64 of the calling thread's page-locked staging buffer of `solve_all` (grow-only)."""
    cache = _solve_cache.__dict__
    buf = cache.get("stage")
    if buf is None or buf.size < count:
        cache["stage"] = None
        buf = cache["stage"] = pinned_empty((count,))
    return buf[:count]


def release_cached_contexts():
    """Free the device context `InteriorPoint.solve` and the staging buffer `InteriorPoint.solve_all` keep for the
    calling thread."""
    rp = _solve_cache.__dict__.pop("rp", None)
    if rp is not None:
        rp.close()
    _solve_cache.__dict__.pop("stage", None)


class ResidentProblem:
    """A Problem uploaded to HBM once (an `lpb_ctx`), reusable across solves."""

    def __init__(self, problem: Problem, stream: int = 0):
        lib = _ffi.load()
        A = problem.A()
        self.m, self.n = A.shape
        self.n_slack = problem.n_slack()
        self.result_dtype = problem.dtype()
        self.last_iterations = 0
        h = C.c_void_p()
        rc = lib.lpb_create(C.byref(h), self.m, self.n, A.ctypes.data, self.n, problem.b().ctypes.data,
                            problem.c().ctypes.data, problem.c0(), _ffi.LPB_MEM_HOST, C.c_void_p(stream))
        _raise_for(rc)
        self.handle = h
        self._problem = problem

    def gather_x(self, x_local):
        return x_local

    def reupload(self, problem: Problem):
        A = problem.A()
        if A.shape != (self.m, self.n):
            raise IncompatibleInputDimensions()
        rc = _ffi.load().lpb_set_problem(self.handle, A.ctypes.data, self.n, problem.b().ctypes.data,
                                         problem.c().ctypes.data, problem.c0(), _ffi.LPB_MEM_HOST)
        _raise_for(rc)
        self.n_slack = problem.n_slack()
        self.result_dtype = problem.dtype()
        self._problem = problem

    def profile(self) -> dict:
        p = _ffi.lpb_profile()
        _raise_for(_ffi.load().lpb_get_profile(self.handle, C.byref(p)))
        return {k: getattr(p, k) for k, _ in p._fields_}

    def debug_read(self, name: str) -> np.ndarray:
        """Host copy of a named device buffer (lpb_debug_read)."""
        lib = _ffi.load()
        n = lib.lpb_debug_read(self.handle, name.encode(), None, 0)
        if n < 0:
            raise KeyError(name)
        out = np.empty(n)
        lib.lpb_debug_read(self.handle, name.encode(), out.ctypes.data, n)
        return out

    def debug_counter(self, name: str) -> int:
        return int(_ffi.load().lpb_debug_counter(self.handle, name.encode()))

    def trace(self) -> np.ndarray:
        rows = np.zeros((max(1, self.last_iterations + 1), _ffi.LPB_TRACE_COLS))
        k = _ffi.load().lpb_trace(self.handle, rows.ctypes.data, rows.shape[0])
        return rows[:k]

    def set_option(self, key: str, value: int):
        _raise_for(_ffi.load().lpb_set_option(self.handle, key.encode(), int(value)))

    def close(self):
        if self.handle is not None:
            _ffi.load().lpb_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchedResult:
    """Outcome of `solve_batched` / `solve_many`: per-problem x (user variables only), fun, iteration and status code
    (0 = Optimal, else the LPB_ERR_* code of the LinearProgramError variant)."""

    def __init__(self, x, x_slack, fun, iteration, status):
        self.x, self.x_slack, self.fun, self.iteration, self.status = x, x_slack, fun, iteration, status


def _solve_batch(entry, A, b, c, n_slack, solver, stream):
    lib = _ffi.load()
    A = np.ascontiguousarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    if A.ndim != 3 or b.shape != A.shape[:2] or c.shape != (A.shape[0], A.shape[2]):
        raise IncompatibleInputDimensions()
    batch, m, n = A.shape
    solver = solver or InteriorPoint.default()
    x = np.zeros((batch, n))
    fun = np.zeros(batch)
    it = np.zeros(batch, dtype=np.int64)
    st = np.zeros(batch, dtype=np.int32)
    rc = getattr(lib, entry)(batch, m, n, A.ctypes.data, b.ctypes.data, c.ctypes.data, C.byref(solver._o),
                             x.ctypes.data, fun.ctypes.data, it.ctypes.data, st.ctypes.data, _ffi.LPB_MEM_HOST,
                             C.c_void_p(stream))
    _raise_for(rc)
    return BatchedResult(x[:, : n - n_slack].copy(), x, fun, it, st)


def solve_batched(A, b, c, n_slack: int = 0, solver: Optional["InteriorPoint"] = None, stream: int = 0):
    """Solve `batch` independent slack-form LPs (A: batch x m x n, b: batch x m, c: batch x n) with one
    CTA per problem (the whole solve_normal_form loop on device).  Host arrays in, host arrays out."""
    return _solve_batch("lpb_solve_batched", A, b, c, n_slack, solver, stream)


def solve_many(A, b, c, n_slack: int = 0, solver: Optional["InteriorPoint"] = None, stream: int = 0):
    """Like `solve_batched`, for LPs of up to 128 rows: problems of up to 64 rows whose A fits beside M in shared
    memory run on `solve_batched`'s kernel, the others on one that reads A through L2.  n is limited by the shared
    memory the rest of a problem needs (n = 768 fits at m = 128); a shape beyond the limits raises InvalidParameter
    naming the limit."""
    return _solve_batch("lpb_solve_many", A, b, c, n_slack, solver, stream)


class Presolved:
    """Outcome of `presolve`: `.problem` is the reduced / scaled slack-form Problem to hand to any Solver;
    `.restore(result)` maps its OptimizeResult back to the original variables (x = C y; the objective is unchanged
    by the scaling).  `dropped_empty` / `dropped_duplicate` count the constraint rows removed."""

    def __init__(self, problem, original, col_scale, dropped_empty, dropped_duplicate, kept_rows):
        self.problem, self._original, self._col_scale = problem, original, col_scale
        self.dropped_empty, self.dropped_duplicate, self.rows = dropped_empty, dropped_duplicate, kept_rows

    def restore(self, result: "OptimizeResult") -> "OptimizeResult":
        n_user = len(result.x())
        x = self._col_scale[:n_user] * result.x()
        return OptimizeResult(x, result.fun(), result.iteration())


def presolve(problem: Problem, scale_passes: int = 2) -> Presolved:
    """Opt-in presolve (no reference counterpart: the crate lists it as a TODO, CONTRIBUTING.md:8): drop empty and
    duplicated constraint rows, then `scale_passes` rounds of power-of-two geometric equilibration -- the two
    causes of NumericalProblem the reference's error message names (error.rs:12-14).  Host only.
    Raises Infeasible when a dropped row contradicts the one it duplicates (or an empty row has b != 0)."""
    lib = _ffi.load()
    A = problem.A()
    m, n = A.shape
    h = C.c_void_p()
    rc = lib.lpb_presolve_create(C.byref(h), m, n, A.ctypes.data, n, problem.b().ctypes.data, problem.c().ctypes.data,
                                 problem.n_slack(), int(scale_passes))
    _raise_for(rc)
    try:
        m2, n2, ns2, de, dd = (C.c_int64() for _ in range(5))
        st = C.c_int32()
        _raise_for(lib.lpb_presolve_info(h, C.byref(m2), C.byref(n2), C.byref(ns2), C.byref(de), C.byref(dd), C.byref(st)))
        _raise_for(st.value)
        A_buf, b_buf, c_buf = _HostBuffer((m2.value, n2.value)), _HostBuffer((m2.value,)), _HostBuffer((n2.value,))
        _raise_for(lib.lpb_presolve_get(h, A_buf.array.ctypes.data, n2.value, b_buf.array.ctypes.data,
                                        c_buf.array.ctypes.data))
        ones = np.ones(n2.value)
        scale = np.empty(n2.value)
        _raise_for(lib.lpb_presolve_restore_x(h, ones.ctypes.data, scale.ctypes.data))
    finally:
        lib.lpb_presolve_destroy(h)
    reduced = Problem(A_buf, b_buf, c_buf, problem.c0(), ns2.value, problem.dtype())
    return Presolved(reduced, problem, scale, de.value, dd.value, m2.value)


def shard_columns(n: int, world: int, n_slack: int = 0):
    """Contiguous column blocks [col0, col0 + n_local) per rank (even widths keep 16-byte alignment).

    The trailing `n_slack` columns of the slack form cost nothing in the SYRK (liblpb200 folds them into
    the diagonal of M), so only the n - n_slack dense columns are balanced over the ranks; the slack
    block rides along with the last rank."""
    n_dense = max(0, n - max(0, int(n_slack)))
    if n_dense == 0:
        n_dense = n
    per = -(-n_dense // world)
    per += per & 1
    out = []
    for r in range(world):
        c0 = min(n_dense, r * per)
        nl = max(0, min(per, n_dense - c0))
        if r == world - 1:
            nl = n - c0
        out.append((c0, nl))
    return out


class ShardedProblem(ResidentProblem):
    """Column shard of a slack-form Problem on this rank's GPU (SURVEY.md 8e).  One process per GPU;
    `dist` is torch.distributed (plumbing: it carries the ncclUniqueId and gathers x)."""

    def __init__(self, problem: Problem, rank: int, world: int, dist, stream: int = 0):
        lib = _ffi.load()
        A = problem.A()
        self.m, n_global = A.shape
        self.n_global = n_global
        self.n_slack = problem.n_slack()
        self.rank, self.world, self._dist = rank, world, dist
        self.shards = shard_columns(n_global, world, self.n_slack)
        self.col0, self.n = self.shards[rank]
        if any(nl <= 0 for _, nl in self.shards):  # the same verdict on every rank, before any collective
            raise ValueError("more ranks than column blocks")
        self.last_iterations = 0
        self._problem = problem
        uid = self._broadcast_unique_id(lib)
        h = C.c_void_p()
        a_ptr = A.ctypes.data + 8 * self.col0
        c_ptr = problem.c().ctypes.data + 8 * self.col0
        rc = lib.lpb_create_sharded(C.byref(h), self.m, n_global, self.col0, self.n, a_ptr, n_global,
                                    problem.b().ctypes.data, c_ptr, problem.c0(), _ffi.LPB_MEM_HOST, rank, world,
                                    uid, C.c_void_p(stream))
        _raise_for(rc)
        self.handle = h
        self._map_peer_memory(lib)

    def _map_peer_memory(self, lib):
        """Peer-memory hand-off of the distributed factorisation (include/lpb200.h: lpb_peer_export / _import).  The
        ring and the mappings belong to the process: the first sharded context exports the cudaIpc handle of its ring,
        the handles are all-gathered and every rank maps the others (~0.4 s, once); later contexts of the same shape
        just attach.  All ranks take the same decision: unless EVERY rank exported and imported successfully, the ring
        is given up and the ncclBroadcast path stays.  LPB_PEER_PANELS=0 switches it off; a gloo (CPU) group has no
        device memory to map."""
        self.peer_panels = False
        if self.world < 2 or self.world > 8 or self._dist.get_backend() != "nccl":
            return
        if os.environ.get("LPB_PEER_PANELS", "1") == "0":
            return
        import torch
        buf = (C.c_ubyte * 64)()
        state = C.c_int(-1)
        exported = lib.lpb_peer_export(self.handle, buf, C.byref(state)) == _ffi.LPB_OK
        if exported and state.value == 0:   # attached to what this process mapped before (same verdict on every rank:
            self.peer_panels = True         # the ranks share the history of contexts)
            return
        if exported and state.value == 2:
            return
        mine = torch.zeros(65, dtype=torch.uint8)
        if exported:
            mine[0] = 1
            mine[1:] = torch.tensor(list(buf), dtype=torch.uint8)
        outs = [torch.zeros(65, dtype=torch.uint8, device="cuda") for _ in range(self.world)]
        self._dist.all_gather(outs, mine.cuda())
        outs = [o.cpu() for o in outs]
        ok = all(int(o[0]) == 1 for o in outs)
        if ok:
            allh = (C.c_ubyte * (64 * self.world))(*[int(v) for o in outs for v in o[1:].tolist()])
            ok = lib.lpb_peer_import(self.handle, allh, self.world) == _ffi.LPB_OK
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        self._dist.all_reduce(flag, op=self._dist.ReduceOp.MIN)
        self.peer_panels = bool(int(flag.item()))
        if not self.peer_panels:             # somebody failed: every rank gives the ring up
            lib.lpb_set_option(self.handle, b"peer_panels", -1)

    def _broadcast_unique_id(self, lib):
        if self.world == 1 or lib.lpb_comm_ready(self.rank, self.world):
            return None  # the process communicator exists already (ncclCommInitRank costs seconds)
        import torch
        buf = (C.c_ubyte * 128)()
        if self.rank == 0:
            _raise_for(lib.lpb_nccl_unique_id(buf))
        t = torch.tensor(list(buf), dtype=torch.uint8)
        on_gpu = self._dist.get_backend() == "nccl"
        if on_gpu:
            t = t.cuda()
        self._dist.broadcast(t, src=0)
        data = bytes(t.cpu().tolist())
        self._uid = (C.c_ubyte * 128).from_buffer_copy(data)
        return C.cast(self._uid, C.c_void_p)

    def gather_x(self, x_local):
        if self.world == 1:
            return x_local
        import torch
        per = max(nl for _, nl in self.shards)
        t = torch.zeros(per, dtype=torch.float64)
        t[: self.n] = torch.from_numpy(np.ascontiguousarray(x_local[: self.n]))
        on_gpu = self._dist.get_backend() == "nccl"
        if on_gpu:
            t = t.cuda()
        outs = [torch.zeros_like(t) for _ in range(self.world)]
        self._dist.all_gather(outs, t)
        return np.concatenate([o.cpu().numpy()[:nl] for o, (_, nl) in zip(outs, self.shards)])

    def reupload(self, problem: Problem):
        raise NotImplementedError


class SyntheticShardedProblem(ShardedProblem):
    """Column shard of the SURVEY.md 8(d) synthetic LP generated ON THE DEVICE (config C5: the
    34 GB matrix never exists on the host).  Slack-form m x n_global with m/2 inequality rows; the
    generator is counter-based, so every (seed, row, column) entry is independent of the sharding and
    any world size sees the same LP."""

    def __init__(self, m: int, n_global: int, seed: int, rank: int = 0, world: int = 1, dist=None, stream: int = 0):
        lib = _ffi.load()
        self.m, self.n_global = int(m), int(n_global)
        self.n_slack = self.m // 2
        self.rank, self.world, self._dist = rank, world, dist
        self.shards = shard_columns(self.n_global, world, self.n_slack)
        self.col0, self.n = self.shards[rank]
        if any(nl <= 0 for _, nl in self.shards):
            raise ValueError("more ranks than column blocks")
        self.last_iterations = 0
        self._problem = None
        uid = self._broadcast_unique_id(lib)
        h = C.c_void_p()
        rc = lib.lpb_create_sharded_synthetic(C.byref(h), self.m, self.n_global, self.col0, self.n, int(seed), rank,
                                              world, uid, C.c_void_p(stream))
        _raise_for(rc)
        self.handle = h
        self._map_peer_memory(lib)

    def download(self):
        """(A_local, b, c_local) as host arrays -- parity tests hand these to the CPU oracle."""
        A = np.empty((self.m, self.n))
        b = np.empty(self.m)
        c = np.empty(self.n)
        _raise_for(_ffi.load().lpb_download_problem(self.handle, A.ctypes.data, self.n, b.ctypes.data,
                                                    c.ctypes.data))
        return A, b, c
