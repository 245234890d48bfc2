"""One query against several stored backgrounds in one call (frisk_b200_background_run_many / _score_many,
engine.run_backgrounds / run_backgrounds_resident) on the GPU: every background's rows and status are bit for bit those of
its own Background.run, for every window-kernel plan, every query format, 1, 2, 3 and 8 backgrounds; status flags that
belong to one background only; the nibble kernel's hand-over; the capacity hand-over; pinned and pageable rows;
interleaving with other runs; stage marks; and no PyTorch on the path."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from tests.helpers import Golden
from tests.test_bgzf_gpu import _same_result
from tests.test_bgzf_host import bgzf
from tests.test_gpu_parity import _check_against_golden
from tests.test_gzip_host import gz_member

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

QUERY = synth.make("C2", 0.01, seed=31) + synth.make("edge")
LONG = synth.make("C1", 0.1, seed=33)                       # scaffolds long enough for 70 kbp windows
# eight hosts: distinct seeded genomes, C1 and C2 at two scales, the edge genome, and one counted with --maskHost
HOSTS = [
    (synth.make("C2", 0.01, seed=32) + synth.make("edge", seed=9), False),
    (synth.make("C1", 0.1, seed=33), False),
    (synth.make("edge", seed=5), False),
    (synth.make("C2", 0.01, seed=32) + synth.make("edge", seed=9), True),
    (synth.make("C2", 0.005, seed=61), False),
    (synth.make("C1", 0.05, seed=62) + synth.make("edge", seed=63), False),
    (synth.make("C2", 0.003, seed=64), True),
    (synth.make("edge", seed=65) + synth.make("C2", 0.002, seed=66), False),
]
COUNTS = (1, 2, 3, 8)


def _encode(sc, kind):
    text = synth.fasta_bytes(sc)
    return {"text": text, "bgzf": bgzf(text, block=30000), "gzip": gz_member(text), "2bit": synth.twobit_bytes(sc)}[kind]


_OPEN = {}


@pytest.fixture(scope="module", autouse=True)
def _close_backgrounds():
    yield
    for bgs in _OPEN.values():
        for bg in bgs:
            bg.close()
    _OPEN.clear()


def _backgrounds(kmin=1, kmax=8):
    """The eight hosts' backgrounds of orders kmin..kmax (opened once per module)."""
    if (kmin, kmax) not in _OPEN:
        _OPEN[kmin, kmax] = [engine.Background.from_result(engine.run_fasta(synth.fasta_bytes(sc), kmin=kmin, kmax=kmax, mask_host=m))
                             for sc, m in HOSTS]
    return _OPEN[kmin, kmax]


def _check_counts(bgs, query, what, **kw):
    """run_backgrounds over the first B backgrounds, B = 1, 2, 3, 8, against each background's own run."""
    want = [bg.run(query, **kw) for bg in bgs]
    assert len(want[0].rows) > 0, what
    for n in COUNTS:
        got = engine.run_backgrounds(bgs[:n], query, **kw)
        assert len(got) == n
        for b in range(n):
            _same_result(got[b], want[b], "%s, %d backgrounds, background %d" % (what, n, b))
    return want


# ---- 1. every plan, bit for bit -----------------------------------------------------------------------------------------------
PLANS = {
    "k8_nibble": dict(kmax=8), "k7_nibble": dict(kmax=7), "k7_w1000_direct": dict(kmax=7, w=1000, step=500),
    "k4_small": dict(kmax=4), "k6_small": dict(kmax=6), "k10_ext": dict(kmax=10),
    "k8_w10000_dense": dict(kmax=8, w=10000, step=5000), "k8_w70000_general": dict(kmax=8, w=70000, step=35000),
    "kmin2_k8": dict(kmin=2, kmax=8), "scaffolds_all": dict(kmax=8, scaffolds_all=True), "rip_off_k8": dict(kmax=8, rip=False),
}


@pytest.mark.parametrize("name", list(PLANS))
def test_many_equals_one_run_per_background(name):
    kw = dict(PLANS[name])
    bgs = _backgrounds(kw.pop("kmin", 1), kw.pop("kmax"))
    query = synth.fasta_bytes(LONG if "w70000" in name else QUERY)
    want = _check_counts(bgs, query, name, kind="text", **kw)
    # distinct hosts give distinct rows: the call did not score every background against one table
    assert not np.array_equal(want[0].rows, want[1].rows, equal_nan=True)


@pytest.mark.parametrize("kind", ["text", "bgzf", "gzip", "2bit"])
@pytest.mark.parametrize("kmax", [6, 8])
def test_many_query_formats(kind, kmax):
    bgs = _backgrounds(1, kmax)
    _check_counts(bgs, _encode(QUERY, kind), kind, kind=kind)
    got = engine.run_backgrounds(bgs, _encode(QUERY, kind))             # kind by signature
    for b, bg in enumerate(bgs):
        _same_result(got[b], bg.run(_encode(QUERY, kind), kind=kind), "%s by signature, background %d" % (kind, b))


# ---- 2. status flags of one background only; the reference's rows ------------------------------------------------------------
def test_reference_rows_among_other_backgrounds():
    """The golden's host tables (orders 1..8) among other backgrounds: its rows are the reference's."""
    case = "c2_small_query_vs_c1_host"
    g = Golden(case)
    kw = g.kwargs()
    qtext = synth.fasta_bytes(g.scaffolds())
    win = dict(w=kw["w"], step=kw["step"], scaffolds_all=kw["scaffolds_all"], rip=kw["rip"])
    golden = engine.Background(g.tables, kw["kmin"], kw["kmax"], g.genome_meta)
    own = engine.Background.from_result(engine.run_fasta(qtext, kmin=kw["kmin"], kmax=kw["kmax"]))
    try:
        for bgs in ([golden, own], [own, golden, own]):
            got = engine.run_backgrounds(bgs, qtext, kind="text", **win)
            for b, bg in enumerate(bgs):
                _same_result(got[b], bg.run(qtext, kind="text", **win), "background %d" % b)
                if bg is golden:
                    _check_against_golden(got[b], g, case + "[run_backgrounds]")
    finally:
        golden.close()
        own.close()


@pytest.mark.parametrize("kmax", [6, 8])
def test_zero_division_rows_belong_to_their_background(kmax):
    """A genome-IVOM entry is NaN (the reference's ZeroDivisionError) when the host lacks the K-mer's kmin-prefix.  At
    kmin 6 a 1,234-base host lacks most 6-mers: its rows carry FRISK_ROW_KLD_ZERODIV, while the query's own background,
    in the same call, lacks none."""
    qtext = synth.fasta_bytes(QUERY)
    orders = dict(kmin=6, kmax=kmax)
    small = [s for s in synth.make("edge") if s[0] == "edge_small"]
    tiny = engine.Background.from_result(engine.run_fasta(synth.fasta_bytes(small), **orders))
    own = engine.Background.from_result(engine.run_fasta(qtext, **orders))
    other = engine.Background.from_result(engine.run_fasta(synth.fasta_bytes(HOSTS[0][0]), **orders))
    try:
        for bgs in ([tiny, own], [own, tiny, other], [other, own, tiny, tiny]):
            got = engine.run_backgrounds(bgs, qtext, kind="text")
            for b, bg in enumerate(bgs):
                _same_result(got[b], bg.run(qtext, kind="text"), "background %d" % b)
                zd = (got[b].status & _lib.ROW_KLD_ZERODIV) != 0
                if bg is own:
                    assert not zd.any()
                if bg is tiny:
                    assert zd.any() and np.isnan(got[b].rows[zd, 0]).all()
    finally:
        for bg in (tiny, own, other):
            bg.close()


# ---- 3. the nibble kernel's hand-over -----------------------------------------------------------------------------------------
def _hand_over_query(seed):
    """Scaffolds whose windows the nibble kernel hands over: a run of 40 As (AAAAAAAA 33 times: a 4-bit counter wraps), and
    a stretch with an N every 12 bases (two cut words per N: far more than 64 in a window)."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    out = []
    for i in range(3):
        s = acgt[rng.integers(0, 4, 40000)].copy()
        s[9000 + 1000 * i:9040 + 1000 * i] = ord("A")
        s[25000:26800:12] = ord("N")
        out.append(("handover%d" % i, s))
    return out


@pytest.mark.parametrize("kmax", [7, 8])
def test_many_nibble_hand_over(kmax):
    q = _hand_over_query(71)
    n_a = sum(int(np.sum(s[25000:26800] == ord("N"))) for _, s in q)
    assert n_a == 3 * 150
    _check_counts(_backgrounds(1, kmax), synth.fasta_bytes(q + QUERY[:2]), "hand-over k%d" % kmax, kind="text")


# ---- 4. capacity, pinned and pageable rows ------------------------------------------------------------------------------------
def _rows(n, pinned):
    return engine._alloc((n, 5), np.float64, pinned), engine._alloc((n,), np.uint32, pinned)


@pytest.mark.parametrize("pinned", [True, False])
@pytest.mark.parametrize("kmax", [6, 8])
def test_many_rows_cap_capacity_and_score_on_the_query_planes(pinned, kmax):
    """Background b's block starts at b * rows_cap; too few rows give FRISK_E_CAPACITY with a valid query handle, and
    frisk_b200_background_score_many on its planes (blocks b * n_win apart) gives the same rows."""
    bgs = _backgrounds(1, kmax)[:3]
    text = synth.fasta_bytes(QUERY)
    want = [bg.run(text, kind="text") for bg in bgs]
    L = _lib.lib()
    buf = np.frombuffer(text, np.uint8)
    hs = engine._handles(bgs)
    for cap in (want[0].n_candidates + 37, 3):
        rows, status = _rows(3 * cap, pinned)
        n, qh = C.c_uint64(0), C.c_void_p()
        rc = L.frisk_b200_background_run_many(hs, 3, C.c_void_p(buf.ctypes.data), len(buf), 0, 5000, 2500, 0, 1, cap,
                                              C.c_void_p(rows.ctypes.data), C.c_void_p(status.ctypes.data), C.byref(n),
                                              C.byref(qh), None)
        try:
            assert int(n.value) == want[0].n_candidates and qh.value
            query = engine._genome_from_handle(L, qh, buf)
            wins = query.windows()
            nw = len(wins)
            if cap > 3:
                assert rc == _lib.OK
                for b, bg in enumerate(bgs):
                    _same_result(bg._result(query, wins, rows[b * cap:b * cap + nw], status[b * cap:b * cap + nw]), want[b],
                                 "rows_cap %d, background %d" % (cap, b))
                continue
            assert rc == _lib.E_CAPACITY
            rows, status = _rows(3 * nw, pinned)
            c, i, lo = C.c_void_p(), C.c_void_p(), C.c_void_p()
            _lib.check(L.frisk_b200_fasta_planes(qh, C.byref(c), C.byref(i), C.byref(lo)), "frisk_b200_fasta_planes")
            _lib.check(L.frisk_b200_background_score_many(hs, 3, c, i, lo, query.padded_len, C.c_void_p(wins.off.ctypes.data),
                                                          C.c_void_p(wins.length.ctypes.data), nw, wins.max_len, 1,
                                                          C.c_void_p(rows.ctypes.data), C.c_void_p(status.ctypes.data), None),
                       "frisk_b200_background_score_many")
            for b, bg in enumerate(bgs):
                _same_result(bg._result(query, wins, rows[b * nw:(b + 1) * nw], status[b * nw:(b + 1) * nw]), want[b],
                             "capacity, background %d" % b)
        finally:
            L.frisk_b200_fasta_close(qh, None)


@pytest.mark.parametrize("kmax", [6, 8])
def test_many_resident(kmax):
    bgs = _backgrounds(1, kmax)
    dq = engine.DeviceGenome(engine.PackedGenome.from_scaffolds(QUERY))
    got = engine.run_backgrounds_resident(bgs, dq)
    for b, bg in enumerate(bgs):
        _same_result(got[b], bg.run_resident(dq), "resident, background %d" % b)
        _same_result(got[b], bg.run(synth.fasta_bytes(QUERY), kind="text"), "resident vs one-call, background %d" % b)


# ---- 5. interleaving, stage marks, no torch -----------------------------------------------------------------------------------
def test_many_between_ordinary_and_single_runs():
    queries = [synth.fasta_bytes(synth.make("C2", 0.005, seed=s) + synth.make("edge", seed=s)) for s in (41, 42)]
    bgs = _backgrounds(1, 8)[:4]
    first = [engine.run_backgrounds(bgs, q) for q in queries]
    for _ in range(2):
        for qi, q in enumerate(queries):
            assert len(engine.run_fasta(q, kmax=6).rows)           # an ordinary run rewrites the run workspace
            one = bgs[2].run(q)
            again = engine.run_backgrounds(bgs, q)
            _same_result(one, first[qi][2], "single run between")
            for b in range(len(bgs)):
                _same_result(again[b], first[qi][b], "query %d, background %d" % (qi, b))


@pytest.mark.parametrize("kmax", [6, 8])
def test_many_stage_marks(kmax):
    engine.run_backgrounds(_backgrounds(1, kmax)[:4], synth.fasta_bytes(QUERY))
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    assert ms[1] == -1.0 and ms[2] == -1.0                        # nothing counted, nothing finalised
    assert 0.0 < ms[0] <= ms[4]
    assert 0.0 < ms[3] <= ms[4]


def test_many_without_torch(tmp_path):
    paths = []
    for i, (sc, m) in enumerate(HOSTS[:3]):
        res = engine.run_fasta(synth.fasta_bytes(sc), mask_host=m)
        np.save(tmp_path / ("t%d.npy" % i), res.tables)
        paths.append((str(tmp_path / ("t%d.npy" % i)), tuple(res.meta)))
    query = tmp_path / "q.fa"
    query.write_bytes(synth.fasta_bytes(QUERY))
    code = ("import sys, numpy as np\nfrom frisk_b200 import engine\n"
            "bgs = [engine.Background(np.load(p), 1, 8, m) for p, m in %r]\n"
            "r = engine.run_backgrounds(bgs, %r)\n"
            "print(len(r), len(r[0].rows), 'torch' in sys.modules)" % (paths, str(query)))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    n_res, n_rows, torch_loaded = out.stdout.split()[-3:]
    assert n_res == "3" and int(n_rows) > 0
    assert torch_loaded == "False", "torch was imported"
