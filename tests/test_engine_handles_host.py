"""The one-call background paths' handle protocol, without a GPU: engine.Background.run and engine.run_backgrounds close
the query's frisk_b200_fasta handle exactly once on every path (rows fit, FRISK_E_CAPACITY and the second stage, a C
error, a failing record read), and one background makes the same C calls as a list of one."""
import ctypes as C

import numpy as np
import pytest

from frisk_b200 import _lib, engine

QH = 0x2000
TEXT = b">a\nACGT\n"


class _FakeLib:
    """Records every C call; the query run returns ``rc`` and, when ``handle``, the query handle QH."""

    def __init__(self, rc=_lib.OK, handle=True, records_rc=_lib.OK):
        self.calls, self.rc, self.handle, self.records_rc = [], rc, handle, records_rc

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        fake = getattr(type(self), "_" + name, None)

        def call(*args):
            self.calls.append((name, args))
            return fake(self, *args) if fake else _lib.OK
        return call

    def _frisk_b200_background_run_many(self, hs, nb, buf, n, fmt, w, step, sa, rip, cap, rows, status, n_win, qh, st):
        n_win._obj.value = 0
        if self.handle:
            qh._obj.value = QH
        return self.rc

    def _frisk_b200_background_run(self, bg, *args):                   # the C side's one-background case of the above
        return self._frisk_b200_background_run_many([bg], 1, *args)

    def _frisk_b200_fasta_info(self, h, nrec, padded, stats):
        nrec._obj.value, padded._obj.value = 0, 128
        return _lib.OK

    def _frisk_b200_fasta_records(self, *args):
        return self.records_rc

    def _frisk_b200_fasta_planes(self, h, c, i, lo):
        c._obj.value, i._obj.value = 0x3000, 0x4000
        return _lib.OK

    def names(self):
        return [name for name, _ in self.calls]

    def closed(self):
        return [args[0].value for name, args in self.calls if name == "frisk_b200_fasta_close"]


class _Fake(engine.Background):
    """A Background that was never opened on a device: only its orders and a non-NULL handle value."""

    def __init__(self, i=0):
        self.kmin, self.kmax, self.device = 1, 8, "cuda:0"
        self._h = C.c_void_p(0x1000 + i)
        self.tables, self.meta = np.zeros(0, np.uint64), (0, 0, 0)

    def close(self):
        self._h = C.c_void_p()


@pytest.fixture
def fake(monkeypatch):
    monkeypatch.setattr(engine, "_torch_loaded", lambda: False)

    def install(**kw):
        L = _FakeLib(**kw)
        monkeypatch.setattr(_lib, "lib", lambda: L)
        return L
    return install


CALLS = {"one": lambda assemble: _Fake().run(TEXT, kind="text", assemble_result=assemble),
         "list of 1": lambda assemble: engine.run_backgrounds([_Fake()], TEXT, kind="text", assemble_result=assemble),
         "list of 3": lambda assemble: engine.run_backgrounds([_Fake(i) for i in range(3)], TEXT, kind="text",
                                                              assemble_result=assemble)}


@pytest.mark.parametrize("how", list(CALLS))
@pytest.mark.parametrize("assemble", [True, False])
@pytest.mark.parametrize("rc", [_lib.OK, _lib.E_CAPACITY])
def test_query_handle_closed_once(fake, how, assemble, rc):
    L = fake(rc=rc)
    CALLS[how](assemble)
    assert L.closed() == [QH]
    scored = [args for name, args in L.calls if name.startswith("frisk_b200_background_score")]
    if rc == _lib.E_CAPACITY:               # the second stage scores the handle's planes before the handle is closed
        assert len(scored) == 1 and L.names().index("frisk_b200_fasta_planes") < L.names().index("frisk_b200_fasta_close")
    else:
        assert not scored and "frisk_b200_fasta_planes" not in L.names()


@pytest.mark.parametrize("how", list(CALLS))
@pytest.mark.parametrize("handle", [True, False])
def test_query_handle_closed_once_on_a_c_error(fake, how, handle):
    L = fake(rc=_lib.E_FORMAT, handle=handle)
    with pytest.raises(_lib.FriskError) as e:
        CALLS[how](True)
    assert e.value.code == _lib.E_FORMAT
    assert L.closed() == ([QH] if handle else [])
    assert "frisk_b200_fasta_records" not in L.names()


@pytest.mark.parametrize("how", list(CALLS))
@pytest.mark.parametrize("rc", [_lib.OK, _lib.E_CAPACITY])
def test_query_handle_closed_once_when_reading_the_records_fails(fake, how, rc):
    L = fake(rc=rc, records_rc=_lib.E_INVALID)
    with pytest.raises(_lib.FriskError, match="frisk_b200_fasta_records"):
        CALLS[how](True)
    assert L.closed() == [QH]


@pytest.mark.parametrize("assemble", [True, False])
@pytest.mark.parametrize("rc", [_lib.OK, _lib.E_CAPACITY])
def test_one_background_is_a_list_of_one(fake, assemble, rc):
    L1 = fake(rc=rc)
    CALLS["one"](assemble)
    L2 = fake(rc=rc)
    CALLS["list of 1"](assemble)
    assert L1.names() == L2.names()
    assert "frisk_b200_background_run_many" in L1.names()
