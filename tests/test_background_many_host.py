"""One query against several stored backgrounds, without a GPU: the C entry points refuse a bad list of backgrounds before
any device work, and engine.run_backgrounds / run_backgrounds_resident refuse with ValueError before any C call."""
import ctypes as C

import numpy as np
import pytest

from frisk_b200 import _lib, engine


def _c_args():
    text = b">a\nACGT\n"
    rows, status, n = np.zeros((4, 5)), np.zeros(4, np.uint32), C.c_uint64(7)
    plane = np.zeros(8, np.uint32)
    off, ln = np.zeros(1, np.uint64), np.full(1, 100, np.uint32)
    return text, rows, status, n, plane, off, ln


def _run_many(L, bgs, n_bg):
    text, rows, status, n, _, _, _ = _c_args()
    qh = C.c_void_p()
    rc = L.frisk_b200_background_run_many(bgs, n_bg, text, len(text), 0, 5000, 2500, 0, 1, 4, C.c_void_p(rows.ctypes.data),
                                          C.c_void_p(status.ctypes.data), C.byref(n), C.byref(qh), None)
    assert not qh.value
    return rc


def _score_many(L, bgs, n_bg):
    _, rows, status, _, plane, off, ln = _c_args()
    pp = C.c_void_p(plane.ctypes.data)
    return L.frisk_b200_background_score_many(bgs, n_bg, pp, pp, None, 128, C.c_void_p(off.ctypes.data),
                                              C.c_void_p(ln.ctypes.data), 1, 100, 1, C.c_void_p(rows.ctypes.data),
                                              C.c_void_p(status.ctypes.data), None)


@pytest.mark.parametrize("call", [_run_many, _score_many])
def test_c_entry_points_refuse_bad_background_lists_before_the_device(call):
    L = _lib.lib()
    nulls = (C.c_void_p * 9)()                         # NULL handles: any dereference would crash, a refusal does not
    assert call(L, None, 1) == _lib.E_INVALID          # NULL list
    for n_bg in (0, -1, 9, _lib.MAX_BACKGROUNDS + 1):  # 1..FRISK_B200_MAX_BACKGROUNDS
        assert call(L, nulls, n_bg) == _lib.E_INVALID
    for n_bg in (1, 2, 8):                             # a NULL entry, first or later
        assert call(L, nulls, n_bg) == _lib.E_INVALID
    assert _lib.MAX_BACKGROUNDS == 8


class _Fake(engine.Background):
    """A Background that was never opened on a device: only its orders and a non-NULL handle value."""

    def __init__(self, kmin, kmax):
        self.kmin, self.kmax, self.device = kmin, kmax, "cuda:0"
        self._h = C.c_void_p(0x1000)

    def close(self):
        self._h = C.c_void_p()


def test_python_refuses_before_any_c_call(monkeypatch):
    def no_lib():
        raise AssertionError("the C library was called")
    monkeypatch.setattr(_lib, "lib", no_lib)
    text = b">a\nACGT\n"
    dq = object()
    for fn, arg in ((engine.run_backgrounds, text), (engine.run_backgrounds_resident, dq)):
        with pytest.raises(ValueError, match="0 backgrounds"):
            fn([], arg)
        with pytest.raises(ValueError, match="9 backgrounds"):
            fn([_Fake(1, 8)] * 9, arg)
        with pytest.raises(ValueError, match="background 1 has orders 1..7, background 0 has 1..8"):
            fn([_Fake(1, 8), _Fake(1, 7)], arg)
        with pytest.raises(ValueError, match="background 2 has orders 2..8"):
            fn([_Fake(1, 8), _Fake(1, 8), _Fake(2, 8)], arg)
        with pytest.raises(ValueError, match="background 1 is not an open engine.Background"):
            fn([_Fake(1, 8), object()], arg)
        closed = _Fake(1, 8)
        closed.close()
        with pytest.raises(ValueError, match="background 0 is not an open"):
            fn([closed], arg)
