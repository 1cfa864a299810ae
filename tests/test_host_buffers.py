"""Lifetime of the page-locked host buffers behind Problem.A() / b() / c() and pinned_empty (lp_b200/api.py).

The CPU test swaps liblpb200's allocator for a recording fake, so the pinned code path runs without a GPU: a
view that outlives its Problem must keep the allocation alive, and the allocation must be freed exactly once
when the last view goes away (ADVICE round 1: use-after-free of np.frombuffer views)."""
import ctypes as C
import gc

import numpy as np
import pytest

import lp_b200
from lp_b200 import _ffi, api


class _FakeLib:
    """Stands in for liblpb200 in _HostBuffer: 'pinned' memory is a ctypes array we hold, frees of it are recorded.
    A free of any other address (real pinned memory of an earlier GPU test, collected while the fake is installed)
    goes to the real library."""

    def __init__(self, real):
        self._real = real
        self.live = {}
        self.allocated = set()
        self.freed = []

    def lpb_device_count(self):
        return 1

    def lpb_host_alloc(self, pref, nbytes):
        mem = (C.c_ubyte * max(1, nbytes))()
        addr = C.addressof(mem)
        self.live[addr] = mem
        self.allocated.add(addr)
        C.cast(pref, C.POINTER(C.c_void_p))[0] = addr
        return _ffi.LPB_OK

    def lpb_host_free(self, p):
        addr = p.value if hasattr(p, "value") else int(p)
        if addr not in self.allocated:
            return self._real.lpb_host_free(p)
        self.freed.append(addr)
        mem = self.live.pop(addr)
        C.memset(mem, 0xFF, len(mem))  # poison: a dangling view would read NaN patterns
        return _ffi.LPB_OK

    def __getattr__(self, name):
        return getattr(self._real, name)


@pytest.fixture
def fake_alloc(monkeypatch):
    fake = _FakeLib(_ffi.load())
    monkeypatch.setattr(api._ffi, "load", lambda: fake)
    return fake


def test_views_keep_the_pinned_allocation_alive(fake_alloc):
    def helper():
        pb = (lp_b200.Problem.target([-1.0, 4.0]).ub([[-3.0, 1.0], [1.0, 2.0]], [6.0, 4.0]).eq([[1.0, 1.0]], [1.0])
              .build())
        assert isinstance(pb.A(), api._PinnedArray)
        return pb.A(), pb.A()[1], pb.b().view(np.ndarray), np.asarray(pb.c())[1:]

    A, row, b, c_tail = helper()   # the Problem is gone; only views survive
    gc.collect()
    assert len(fake_alloc.freed) == 0
    np.testing.assert_array_equal(A, [[-3.0, 1.0, 1.0, 0.0], [1.0, 2.0, 0.0, 1.0], [1.0, 1.0, 0.0, 0.0]])
    np.testing.assert_array_equal(row, [1.0, 2.0, 0.0, 1.0])
    np.testing.assert_array_equal(b, [6.0, 4.0, 1.0])
    np.testing.assert_array_equal(c_tail, [4.0, 0.0, 0.0])
    del A
    gc.collect()
    assert len(fake_alloc.freed) == 0   # `row` still views A's allocation
    del row, b, c_tail
    gc.collect()
    assert len(fake_alloc.freed) == 3 and len(set(fake_alloc.freed)) == 3 and not fake_alloc.live


def test_pinned_empty_frees_once(fake_alloc):
    a = lp_b200.pinned_empty((4, 6))
    a[:] = 2.0
    v = a[1:3, ::2]
    del a
    gc.collect()
    assert fake_alloc.freed == [] and float(v.sum()) == 12.0
    del v
    gc.collect()
    assert len(fake_alloc.freed) == 1


@pytest.mark.gpu
def test_real_pinned_views_outlive_their_problem():
    def helper():
        pb = lp_b200.Problem.target(np.arange(5.0)).ub(np.ones((2, 5)), [1.0, 2.0]).build()
        return pb.A()

    A = helper()
    gc.collect()
    junk = [lp_b200.pinned_empty((2, 7)) for _ in range(8)]  # would recycle a freed pinned block
    for j in junk:
        j[:] = -7.0
    assert isinstance(A, api._PinnedArray)
    np.testing.assert_array_equal(A[:, :5], np.ones((2, 5)))
    np.testing.assert_array_equal(A[:, 5:], np.eye(2))
