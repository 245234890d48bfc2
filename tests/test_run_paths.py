"""The one-call run paths (frisk_b200_run_host / _sparse / _peers / _run_resident / _run_fasta / _run_fasta_bgzf).

Without a GPU: a fixed table of bad arguments, each refused by one entry point with a fixed code before any device work.
On a GPU: which stage marks of frisk_b200_last_run_timing each path sets (bench.py's e2e.stages reads them)."""
import ctypes as C

import numpy as np
import pytest

from frisk_b200 import _lib

INV, UNS = _lib.E_INVALID, _lib.E_UNSUPPORTED
HUGE = (1 << 37) + 128          # a padded length whose 32-base word indices do not fit 32 bits

# host buffers: 256 bases of planes, one window of 100 bases at 0, its row, status and tables (never read on a refusal)
_bufs = {"codes": np.zeros(16, np.uint32), "inv": np.zeros(8, np.uint32), "idx": np.zeros(1, np.uint32),
         "val": np.zeros(1, np.uint32), "off": np.zeros(1, np.uint64), "len": np.full(1, 100, np.uint32),
         "out": np.zeros(1 << 20, np.uint64), "ptrs": np.zeros(2, np.uint64), "text": np.frombuffer(b">a\nACGT\n", np.uint8)}


def _p(name):
    return C.c_void_p(_bufs[name].ctypes.data)


def _plane_base():
    return dict(hc=_p("codes"), hi=_p("inv"), hl=None, hp=256, qc=_p("codes"), qi=_p("inv"), ql=None, qp=256,
                off=_p("off"), len=_p("len"), n=1, mx=100, kmin=1, kmax=8, rows=_p("out"), stat=_p("out"))


def _call_dense(fn, a):
    return fn(a["hc"], a["hi"], a["hl"], a["hp"], a["qc"], a["qi"], a["ql"], a["qp"], a["off"], a["len"], a["n"], a["mx"],
              a["kmin"], a["kmax"], 0, 1, 100, a["rows"], a["stat"], _p("out"), _p("out"), None)


def run_host(**kw):
    return _call_dense(_lib.lib().frisk_b200_run_host, {**_plane_base(), **kw})


def run_resident(**kw):
    return _call_dense(_lib.lib().frisk_b200_run_resident, {**_plane_base(), **kw})


def run_host_sparse(**kw):
    a = {**_plane_base(), "hidx": _p("idx"), "hval": _p("val"), "hn": 1, "qidx": _p("idx"), "qval": _p("val"), "qn": 1, **kw}
    return _lib.lib().frisk_b200_run_host_sparse(
        a["hc"], a["hidx"], a["hval"], a["hn"], a["hl"], a["hp"], a["qc"], a["qidx"], a["qval"], a["qn"], a["ql"], a["qp"],
        a["off"], a["len"], a["n"], a["mx"], a["kmin"], a["kmax"], 0, 1, 100, a["rows"], a["stat"], _p("out"), _p("out"), None)


def run_host_peers(**kw):
    a = {**_plane_base(), "hidx": _p("idx"), "hval": _p("val"), "hn": 1, "fwd": _p("out"), "peers": _p("ptrs"),
         "flags": _p("ptrs"), "rank": 0, "world": 2, "epoch": 1, **kw}
    return _lib.lib().frisk_b200_run_host_peers(
        a["hc"], a["hidx"], a["hval"], a["hn"], a["hl"], a["hp"], a["off"], a["len"], a["n"], a["mx"], a["kmin"], a["kmax"],
        0, 1, 100, a["fwd"], a["peers"], a["flags"], a["rank"], a["world"], a["epoch"], a["rows"], a["stat"], _p("out"),
        _p("out"), None)


def _run_fasta(fn, kw):
    hh, qh, n = C.c_void_p(), C.c_void_p(), C.c_uint64(0)
    a = {"h": _p("text"), "hn": 8, "q": None, "qn": 0, "w": 5000, "step": 2500, "kmin": 1, "kmax": 8, "cap": 1,
         "rows": _p("out"), "stat": _p("out"), "hout": C.byref(hh), "qout": C.byref(qh), **kw}
    return fn(a["h"], a["hn"], a["q"], a["qn"], a["w"], a["step"], 0, a["kmin"], a["kmax"], 0, 1, a["cap"], a["rows"],
              a["stat"], _p("out"), _p("out"), C.byref(n), a["hout"], a["qout"], None)


def run_fasta(**kw):
    return _run_fasta(_lib.lib().frisk_b200_run_fasta, kw)


def run_fasta_bgzf(**kw):
    return _run_fasta(_lib.lib().frisk_b200_run_fasta_bgzf, kw)


_bufs["outside"] = np.array([200], np.uint64)
_bufs["zero"] = np.zeros(1, np.uint32)
_bufs["long"] = np.full(1, 101, np.uint32)

_PLANE_CASES = [                 # shared by run_host, run_host_sparse and run_resident: (label, overrides, code)
    ("host codes null", dict(hc=None), INV),
    ("query codes null", dict(qc=None), INV),
    ("host padded length not a multiple of 128", dict(hp=200), INV),
    ("query padded length not a multiple of 128", dict(qp=100), INV),
    ("query padded length 0", dict(qp=0), INV),
    ("window offsets null", dict(off=None), INV),
    ("window lengths null", dict(len=None), INV),
    ("rows null", dict(rows=None), INV),
    ("status null", dict(stat=None), INV),
    ("window outside the query planes", dict(off=_p("outside")), INV),
    ("window of length 0", dict(len=_p("zero")), INV),
    ("window longer than max_win_len", dict(len=_p("long")), INV),
    ("kmin > kmax", dict(kmin=3, kmax=2), INV),
    ("kmin 0", dict(kmin=0), INV),
    ("kmax 13", dict(kmax=13), UNS),
    ("codes null before kmax 13", dict(hc=None, kmax=13), INV),
    ("kmax 13 before the window check", dict(kmax=13, off=_p("outside")), UNS),
    ("padded length before the window check", dict(hp=200, off=_p("outside")), INV),
]

CASES = (
    [("run_host", lbl, kw, rc) for lbl, kw, rc in _PLANE_CASES] +
    [("run_host", "host invalid plane null", dict(hi=None), INV),
     ("run_host", "query invalid plane null", dict(qi=None), INV),
     ("run_host", "invalid plane null before kmax 13", dict(qi=None, kmax=13), INV)] +
    [("run_resident", lbl, kw, rc) for lbl, kw, rc in _PLANE_CASES] +
    [("run_resident", "host invalid plane null", dict(hi=None), INV),
     ("run_resident", "query invalid plane null", dict(qi=None), INV)] +
    [("run_host_sparse", lbl, kw, rc) for lbl, kw, rc in _PLANE_CASES] +
    [("run_host_sparse", "host count without indices", dict(hidx=None), INV),
     ("run_host_sparse", "host count without words", dict(hval=None), INV),
     ("run_host_sparse", "query count without indices", dict(qidx=None), INV),
     ("run_host_sparse", "query count without words", dict(qval=None), INV),
     ("run_host_sparse", "no count, no arrays, no codes", dict(hidx=None, hval=None, hn=0, hc=None), INV),
     ("run_host_sparse", "host word index beyond 2^32", dict(hp=HUGE), UNS),
     ("run_host_sparse", "query word index beyond 2^32", dict(qp=HUGE), UNS),
     ("run_host_sparse", "word index beyond 2^32 before null codes", dict(hp=HUGE, hc=None), UNS),
     ("run_host_sparse", "arrays before the word index", dict(hp=HUGE, hidx=None), INV)] +
    [("run_host_peers", "codes null", dict(hc=None), INV),
     ("run_host_peers", "padded length not a multiple of 128", dict(hp=200), INV),
     ("run_host_peers", "count without indices", dict(hidx=None), INV),
     ("run_host_peers", "window offsets null", dict(off=None), INV),
     ("run_host_peers", "rows null", dict(rows=None), INV),
     ("run_host_peers", "window outside the planes", dict(off=_p("outside")), INV),
     ("run_host_peers", "kmin > kmax", dict(kmin=3, kmax=2), INV),
     ("run_host_peers", "epoch 0", dict(epoch=0), INV),
     ("run_host_peers", "world 0", dict(world=0), INV),
     ("run_host_peers", "rank == world", dict(rank=2), INV),
     ("run_host_peers", "rank -1", dict(rank=-1), INV),
     ("run_host_peers", "local counters null", dict(fwd=None), INV),
     ("run_host_peers", "peer counters null", dict(peers=None), INV),
     ("run_host_peers", "peer flags null", dict(flags=None), INV),
     ("run_host_peers", "world 17", dict(world=17), UNS),
     ("run_host_peers", "kmax 9", dict(kmax=9), UNS),
     ("run_host_peers", "kmax 13", dict(kmax=13), UNS),
     ("run_host_peers", "word index beyond 2^32", dict(hp=HUGE), UNS),
     ("run_host_peers", "epoch 0 before kmax 9", dict(epoch=0, kmax=9), INV),
     ("run_host_peers", "world 17 before null codes", dict(world=17, hc=None), UNS)])

_FASTA_CASES = [
    ("no place for the host handle", dict(hout=None), INV),
    ("no place for the query handle", dict(qout=None), INV),
    ("host text null", dict(h=None), INV),
    ("query text null with a length", dict(qn=5), INV),
    ("rows null with a capacity", dict(rows=None), INV),
    ("status null with a capacity", dict(stat=None), INV),
    ("kmin > kmax", dict(kmin=3, kmax=2), INV),
    ("kmin 0", dict(kmin=0), INV),
    ("kmax 13", dict(kmax=13), UNS),
    ("window length 0", dict(w=0), INV),
    ("step 0", dict(step=0), INV),
    ("kmax 13 before the window length", dict(kmax=13, w=0), UNS),
    ("rows before kmax 13", dict(rows=None, kmax=13), INV),
]
CASES += [(fn, lbl, kw, rc) for fn in ("run_fasta", "run_fasta_bgzf") for lbl, kw, rc in _FASTA_CASES]


@pytest.mark.parametrize("fn,label,kw,code", CASES, ids=["%s: %s" % (c[0], c[1]) for c in CASES])
def test_refusal_table(fn, label, kw, code):
    """Checked before anything touches a device: the same code with and without a GPU."""
    assert globals()[fn](**kw) == code


# ---- on the GPU -----------------------------------------------------------------------------------------------------

MARKS = ("uploaded", "counted", "finalised", "scored", "end", "score_start")
ALL = frozenset(MARKS)

# the marks that read >= 0 after each call (None: frisk_b200_last_run_timing refuses -- the call set no end mark)
EXPECTED_MARKS = {
    "run_host": ALL,
    "run_host_sparse": ALL,
    "run_host_pageable": ALL,
    "run_resident": ALL - {"uploaded"},
    "run_fasta_k8": ALL,
    "run_fasta_k6": ALL,
    "run_fasta_k8_too_few_rows": ALL,
    "run_fasta_k6_too_few_rows": None,
    "run_fasta_bgzf": ALL,
}


def _marks():
    ms, n = (C.c_float * 6)(), C.c_int(0)
    if _lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)) != _lib.OK:
        return None
    return frozenset(MARKS[i] for i in range(n.value) if ms[i] >= 0)


@pytest.fixture(scope="module")
def genome():
    from frisk_b200 import engine, synth
    _lib.require_device()
    rng = np.random.Generator(np.random.PCG64(5))
    sc = [("a", synth.iid_bases(rng, 120_000, 0.45)), ("b", synth.iid_bases(rng, 30_000, 0.4))]
    return sc, engine.PackedGenome.from_scaffolds(sc, pinned=True), synth.fasta_bytes(sc)


def _fasta(text, kmax, rows_cap=None, bgzf=False):
    import torch
    from frisk_b200 import engine
    L = _lib.lib()
    buf = np.frombuffer(text, np.uint8)
    out = engine.HostOutputs(rows_cap or 1024, kmax)
    hh, qh, n = C.c_void_p(), C.c_void_p(), C.c_uint64(0)
    fn = L.frisk_b200_run_fasta_bgzf if bgzf else L.frisk_b200_run_fasta
    dev = torch.device("cuda:0")
    with torch.cuda.device(dev):
        st = engine._stream_ptr(dev)
        rc = fn(engine._ptr(buf), buf.shape[0], None, 0, 5000, 2500, 0, 1, kmax, 0, 1, out.rows.shape[0], engine._ptr(out.rows),
                engine._ptr(out.status), engine._ptr(out.tables), engine._ptr(out.valid), C.byref(n), C.byref(hh), C.byref(qh), st)
        for h in (qh, hh):
            if h:
                L.frisk_b200_fasta_close(h, st)
        torch.cuda.synchronize()
    assert rc == (_lib.E_CAPACITY if rows_cap else _lib.OK)


def _run(path, genome):
    from frisk_b200 import engine
    from tests.test_bgzf_host import bgzf
    _, g, text = genome
    if path == "run_host":
        engine.run_host(g, sparse=False)
    elif path == "run_host_sparse":
        engine.run_host(g, sparse=True)
    elif path == "run_host_pageable":
        engine.run_host(g, sparse=False, out=engine.HostOutputs(len(g.windows()), 8, pinned=False))
    elif path == "run_resident":
        engine.run_resident(engine.DeviceGenome(g))
    elif path == "run_fasta_bgzf":
        _fasta(bgzf(text, block=20000), 8, bgzf=True)
    else:
        kmax = int(path.split("_k")[1][0])
        _fasta(text, kmax, rows_cap=8 if path.endswith("too_few_rows") else None)


@pytest.mark.gpu
@pytest.mark.parametrize("path", sorted(EXPECTED_MARKS))
def test_stage_marks_of_each_path(genome, path):
    _run(path, genome)
    assert _marks() == EXPECTED_MARKS[path]
