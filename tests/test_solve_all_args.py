"""CPU checks of the ragged batched mode (lpb_solve_many_ragged / InteriorPoint.solve_all): argument and shape checks
happen before any device is touched, and the packing of a list of problems round-trips."""
import os

import numpy as np
import pytest

import lp_b200
from lp_b200 import _ffi
from lp_b200.api import _pack_problems


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_ffi.LIB_PATH):
        from lp_b200 import build
        build.build(verbose=False)
    return _ffi.load()


def _ragged(lib, ms, ns, batch=None, null=None):
    """Call lpb_solve_many_ragged on zero host arrays of the given shapes; `null` names one pointer to pass as NULL."""
    m = np.array(ms, dtype=np.int64)
    n = np.array(ns, dtype=np.int64)
    na, nb, nc = int(max(1, (m * n).sum())), int(max(1, m.sum())), int(max(1, n.sum()))
    arrs = dict(A=np.zeros(na), b=np.zeros(nb), c=np.zeros(nc), x=np.zeros(nc), fun=np.zeros(len(ms) or 1),
                it=np.zeros(len(ms) or 1, dtype=np.int64), st=np.zeros(len(ms) or 1, dtype=np.int32), m=m, n=n)
    ptr = {k: (None if k == null else v.ctypes.data) for k, v in arrs.items()}
    return lib.lpb_solve_many_ragged(len(ms) if batch is None else batch, ptr["m"], ptr["n"], ptr["A"], ptr["b"],
                                     ptr["c"], None, ptr["x"], ptr["fun"], ptr["it"], ptr["st"], _ffi.LPB_MEM_HOST,
                                     None)


def test_bad_arguments(lib):
    assert _ragged(lib, [4], [8], batch=0) == _ffi.LPB_ERR_BAD_ARGUMENT
    assert _ragged(lib, [4], [8], batch=-1) == _ffi.LPB_ERR_BAD_ARGUMENT
    for name in ("m", "n", "A", "b", "c", "x", "fun", "it", "st"):
        assert _ragged(lib, [4, 6], [8, 9], null=name) == _ffi.LPB_ERR_BAD_ARGUMENT, name
    assert _ragged(lib, [4, 0], [8, 9]) == _ffi.LPB_ERR_BAD_ARGUMENT
    assert _ragged(lib, [4, 6], [8, 0]) == _ffi.LPB_ERR_BAD_ARGUMENT
    assert "LP 1" in _ffi.last_error()


@pytest.mark.parametrize("shape,limit", [((129, 200), "m <= 128"), ((128, 1000), "227 KB")])
def test_shapes_outside_the_limits_refuse_the_whole_call(lib, shape, limit):
    ms, ns = [8, 64, shape[0], 16], [16, 128, shape[1], 40]
    assert _ragged(lib, ms, ns) == _ffi.LPB_ERR_UNSUPPORTED
    err = _ffi.last_error()
    assert "LP 2" in err and limit in err, err


def test_shapes_inside_the_limits_reach_the_device_check(lib):
    if lib.lpb_device_count() > 0:
        pytest.skip("a GPU is visible")
    assert _ragged(lib, [128, 64, 1, 100], [768, 1024, 2, 173]) == _ffi.LPB_ERR_NO_DEVICE


@pytest.mark.parametrize("m,n", [(129, 200), (128, 1000), (2, 3000), (128, 768), (64, 1024), (1, 2), (0, 5), (5, 0)])
def test_check_agrees_with_solve_many(lib, m, n):
    """lpb_solve_many_check refuses exactly what solve_many refuses (the shapes of test_solve_many_limits)."""
    rc = lib.lpb_solve_many_check(m, n)
    if m <= 0 or n <= 0:
        assert rc == _ffi.LPB_ERR_BAD_ARGUMENT
        return
    if rc == _ffi.LPB_OK:
        if lib.lpb_device_count() == 0:  # solve_many accepts the shape: it gets as far as the device check
            with pytest.raises(lp_b200.api.DeviceError):
                lp_b200.solve_many(np.zeros((1, m, n)), np.zeros((1, m)), np.zeros((1, n)))
    else:
        assert rc == _ffi.LPB_ERR_UNSUPPORTED
        with pytest.raises(lp_b200.InvalidParameter):
            lp_b200.solve_many(np.zeros((1, m, n)), np.zeros((1, m)), np.zeros((1, n)))


def _problems(seed, shapes):
    rng = np.random.default_rng(seed)
    out = []
    for m_ub, m_eq, nu in shapes:
        b = lp_b200.Problem.target(rng.standard_normal(nu))
        if m_ub:
            b = b.ub(rng.standard_normal((m_ub, nu)), rng.standard_normal(m_ub))
        if m_eq:
            b = b.eq(rng.standard_normal((m_eq, nu)), rng.standard_normal(m_eq))
        out.append(b.build())
    return out


def test_packing_round_trips(lib):
    pbs = _problems(1, [(3, 2, 7), (0, 4, 5), (6, 0, 9), (1, 1, 1)])
    pk = _pack_problems(pbs)
    assert list(pk.m) == [p.A().shape[0] for p in pbs] and list(pk.n) == [p.A().shape[1] for p in pbs]
    assert pk.A.size == sum(p.A().size for p in pbs) and pk.x.size == pk.c.size == sum(p.c().size for p in pbs)
    for k, p in enumerate(pbs):
        m, n = p.A().shape
        np.testing.assert_array_equal(pk.A[pk.a_off[k]: pk.a_off[k] + m * n].reshape(m, n), p.A())
        np.testing.assert_array_equal(pk.b[pk.b_off[k]: pk.b_off[k] + m], p.b())
        np.testing.assert_array_equal(pk.c[pk.c_off[k]: pk.c_off[k] + n], p.c())
    assert pk.fun.size == pk.it.size == pk.st.size == len(pbs)
    assert pk.it.dtype == np.int64 and pk.st.dtype == np.int32


def test_solve_all_of_nothing():
    assert lp_b200.InteriorPoint.default().solve_all([]) == []
