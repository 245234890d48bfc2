"""Scoring against a resident background (frisk_b200_background_*, engine.Background) on the GPU: pinned to the reference's
goldens, bit-identical to the counted one-call run on every window-kernel class and query format, the capacity hand-over,
reuse of one handle between ordinary runs, the stage marks, the device-only tail, and the CLI reusing its genome pickle
without the host file."""
import ctypes as C
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from tests.helpers import SMALL_CASES, Golden
from tests.test_bgzf_gpu import _same_result
from tests.test_bgzf_host import bgzf
from tests.test_gpu_parity import _check_against_golden
from tests.test_gzip_host import gz_member

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HOST = synth.make("C2", 0.01, seed=32) + synth.make("edge", seed=9)
QUERY = synth.make("C2", 0.01, seed=31) + synth.make("edge")
LONG = synth.make("C1", 0.1, seed=33)                       # scaffolds long enough for 70 kbp windows


def _encode(sc, kind):
    text = synth.fasta_bytes(sc)
    return {"text": text, "bgzf": bgzf(text, block=30000), "gzip": gz_member(text), "2bit": synth.twobit_bytes(sc)}[kind]


def _background(host_text, kmin=1, kmax=8, mask_host=False):
    return engine.Background.from_result(engine.run_fasta(host_text, kmin=kmin, kmax=kmax, mask_host=mask_host))


def _split(kw):
    tab = {k: kw[k] for k in ("kmin", "kmax", "mask_host") if k in kw}
    win = {k: kw[k] for k in ("w", "step", "scaffolds_all", "rip") if k in kw}
    return tab, win


# ---- 1. the reference's own tables and rows ----------------------------------------------------------------------------------
@pytest.mark.parametrize("case", SMALL_CASES + ["c1_full"])
def test_background_matches_reference_golden(case):
    g = Golden(case)
    kw = g.kwargs()
    with engine.Background(g.tables, kw["kmin"], kw["kmax"], g.genome_meta) as bg:
        res = bg.run(synth.fasta_bytes(g.scaffolds()), kind="text", w=kw["w"], step=kw["step"],
                     scaffolds_all=kw["scaffolds_all"], rip=kw["rip"])
    _check_against_golden(res, g, case + "[background]")


# ---- 2. bit-identical to the counted run ----------------------------------------------------------------------------------------
KERNELS = {
    "k4_small": dict(kmax=4), "k6_small": dict(kmax=6),
    "k7_nibble": dict(kmax=7), "k8_nibble": dict(kmax=8),
    "k9_ext": dict(kmax=9), "k12_ext": dict(kmax=12),
    "k8_w10000_dense": dict(kmax=8, w=10000, step=5000), "k8_w70000_general": dict(kmax=8, w=70000, step=35000),
    "scaffolds_all": dict(kmax=8, scaffolds_all=True), "mask_host": dict(kmax=8, mask_host=True),
    "rip_off": dict(kmax=8, rip=False), "rip_off_k6": dict(kmax=6, rip=False), "kmin2": dict(kmin=2, kmax=8),
    "kmin2_k6": dict(kmin=2, kmax=6),
}


@pytest.mark.parametrize("name", list(KERNELS))
def test_background_equals_counted_run(name):
    kw = KERNELS[name]
    tab, win = _split(kw)
    sc = LONG if "w70000" in name else QUERY
    host_text, query_text = synth.fasta_bytes(HOST if sc is QUERY else synth.make("C1", 0.05, seed=34)), synth.fasta_bytes(sc)
    want = engine.run_fasta(query_text, host_text, **kw)
    assert len(want.rows) > 0
    with _background(host_text, **tab) as bg:
        _same_result(bg.run(query_text, kind="text", **win), want, name)


@pytest.mark.parametrize("kind", ["text", "bgzf", "gzip", "2bit"])
@pytest.mark.parametrize("kmax", [6, 8])
def test_background_query_formats(kind, kmax):
    host_text = synth.fasta_bytes(HOST)
    want = engine.run_fasta(synth.fasta_bytes(QUERY), host_text, kmax=kmax)
    with _background(host_text, kmax=kmax) as bg:
        _same_result(bg.run(_encode(QUERY, kind), kind=kind), want, kind)
        _same_result(bg.run(_encode(QUERY, kind)), want, kind + " by signature")


@pytest.mark.parametrize("pinned", [True, False])
@pytest.mark.parametrize("kmax", [6, 8])
def test_background_pinned_and_pageable_rows(pinned, kmax):
    host_text, query_text = synth.fasta_bytes(HOST), synth.fasta_bytes(QUERY)
    want = engine.run_fasta(query_text, host_text, kmax=kmax)
    with _background(host_text, kmax=kmax) as bg:
        out = engine.HostOutputs(len(want.rows) + 100, 0, pinned=pinned)
        _same_result(bg.run(query_text, kind="text", out=out), want, "pinned" if pinned else "pageable")


@pytest.mark.parametrize("kmax", [6, 8])
def test_background_capacity_then_score_on_the_query_planes(kmax):
    """FRISK_E_CAPACITY leaves the query's handle valid; frisk_b200_background_score on its planes gives the same rows."""
    host_text, query_text = synth.fasta_bytes(HOST), synth.fasta_bytes(QUERY)
    want = engine.run_fasta(query_text, host_text, kmax=kmax)
    L = _lib.lib()
    with _background(host_text, kmax=kmax) as bg:
        buf = np.frombuffer(query_text, np.uint8)
        rows, status = np.zeros((3, 5)), np.zeros(3, np.uint32)
        n, qh = C.c_uint64(0), C.c_void_p()
        rc = L.frisk_b200_background_run(bg._h, C.c_void_p(buf.ctypes.data), len(buf), 0, 5000, 2500, 0, 1, 3,
                                         C.c_void_p(rows.ctypes.data), C.c_void_p(status.ctypes.data), C.byref(n), C.byref(qh), None)
        try:
            assert rc == _lib.E_CAPACITY and qh.value
            assert int(n.value) == want.n_candidates
            query = engine._genome_from_handle(L, qh, buf)
            wins = query.windows()
            out = engine.HostOutputs(len(wins), 0, pinned=False)
            c, i, lo = C.c_void_p(), C.c_void_p(), C.c_void_p()
            _lib.check(L.frisk_b200_fasta_planes(qh, C.byref(c), C.byref(i), C.byref(lo)), "frisk_b200_fasta_planes")
            _lib.check(L.frisk_b200_background_score(bg._h, c, i, lo, query.padded_len, C.c_void_p(wins.off.ctypes.data),
                                                     C.c_void_p(wins.length.ctypes.data), len(wins), wins.max_len, 1,
                                                     C.c_void_p(out.rows.ctypes.data), C.c_void_p(out.status.ctypes.data), None),
                       "frisk_b200_background_score")
            _same_result(bg._result(query, wins, out.rows, out.status), want, "capacity")
        finally:
            L.frisk_b200_fasta_close(qh, None)
        # the Python layer takes the same second stage by itself
        _same_result(bg.run(query_text, kind="text", out=engine.HostOutputs(3, 0)), want, "capacity, engine")


# ---- 3. query == host; 4. reuse ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kmax", [6, 8, 9])
def test_background_of_the_query_itself(kmax):
    text = synth.fasta_bytes(HOST)
    want = engine.run_fasta(text, kmax=kmax)
    with engine.Background.from_result(want) as bg:
        _same_result(bg.run(text, kind="text"), want, "query == host")


def test_one_background_many_queries_between_ordinary_runs():
    host_text = synth.fasta_bytes(HOST)
    queries = [synth.fasta_bytes(synth.make("C2", 0.005, seed=s) + synth.make("edge", seed=s)) for s in (41, 42, 43)]
    for kmax, other_kmax in ((8, 6), (6, 8)):                     # device tail, then host tail
        bg = _background(host_text, kmax=kmax)
        for q in queries:
            other = engine.run_fasta(q, kmax=other_kmax)          # an ordinary run rewrites the run workspace, IVOM included
            assert len(other.rows)
            _same_result(bg.run(q, kind="text"), engine.run_fasta(q, host_text, kmax=kmax), "reuse, kmax %d" % kmax)
        bg.close()
        bg.close()                                                # (a second close does nothing)
    with _background(host_text) as again:
        _same_result(again.run(queries[0], kind="text"), engine.run_fasta(queries[0], host_text), "reopened")


# ---- 5. stage marks, the device-only tail, no torch ---------------------------------------------------------------------------
@pytest.mark.parametrize("kmax", [6, 8])
def test_background_stage_marks(kmax):
    with _background(synth.fasta_bytes(HOST), kmax=kmax) as bg:
        bg.run(synth.fasta_bytes(QUERY), kind="text")
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    assert ms[1] == -1.0 and ms[2] == -1.0                        # nothing counted, nothing finalised
    assert 0.0 < ms[0] <= ms[4]
    assert 0.0 < ms[3] <= ms[4]


def test_background_device_only_tail_and_no_torch(tmp_path):
    """kmax 8: windows and window kernel are queued from the query's open (no host-side window step in the trace); kmax 6:
    the host tail.  Background goes through the C ABI alone: torch is never imported."""
    host_text = synth.fasta_bytes(HOST)
    query = tmp_path / "q.fa"
    query.write_bytes(synth.fasta_bytes(QUERY))
    traces = {}
    for kmax in (8, 6):
        res = engine.run_fasta(host_text, kmax=kmax)
        np.save(tmp_path / "t.npy", res.tables)
        code = ("import sys, numpy as np\nfrom frisk_b200 import engine\n"
                "with engine.Background(np.load(%r), 1, %d, %r) as bg:\n    r = bg.run(%r)\n"
                "print(len(r.rows), 'torch' in sys.modules)" % (str(tmp_path / "t.npy"), kmax, tuple(res.meta), str(query)))
        env = dict(os.environ, FRISK_RUN_TRACE="1")
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        assert out.stdout.split()[-1] == "False", "torch was imported"
        lines = [ln for ln in out.stderr.splitlines() if ln.startswith("host trace")]
        assert lines, out.stderr[-2000:]
        traces[kmax] = lines[-1]
    assert "windows" not in traces[8] and "score_queued" not in traces[8] and "done" in traces[8], traces[8]
    assert "windows" in traces[6] and "score_queued" in traces[6] and "finalize_queued" not in traces[6], traces[6]


# ---- 6. the CLI -----------------------------------------------------------------------------------------------------------------
def _cli(args, cwd=ROOT):
    code = ("import sys, frisk\ntry:\n    frisk.main(%r)\nexcept SystemExit as e:\n    assert not e.code, e.code\n"
            "print('torch' in sys.modules)" % (list(args),))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=cwd, timeout=600)
    assert out.returncode == 0, out.stdout[-1000:] + out.stderr[-3000:]
    assert out.stdout.strip().splitlines()[-1] == "False", "torch was imported"
    return out


def test_cli_reuses_the_genome_pickle_without_the_host(tmp_path):
    a, b = tmp_path / "cached", tmp_path / "fresh"
    for d in (a, b):
        d.mkdir()
        (d / "host.fa").write_bytes(synth.fasta_bytes(HOST))
    q1, q2 = tmp_path / "q1.fa", tmp_path / "q2.fa"
    q1.write_bytes(synth.fasta_bytes(synth.make("C2", 0.005, seed=51) + synth.make("edge")))
    q2.write_bytes(synth.fasta_bytes(QUERY))
    flags = ["--quiet", "--RIP"]
    _cli(["-H", str(a / "host.fa"), "-Q", str(q1), "-t", str(a / "temp")] + flags)
    os.remove(a / "host.fa")
    out = _cli(["-H", str(a / "host.fa"), "-Q", str(q2), "-t", str(a / "temp")] + flags)
    assert "against the background tables in" in out.stderr
    _cli(["-H", str(b / "host.fa"), "-Q", str(q2), "-t", str(b / "temp")] + flags)
    for f in ("raw_window_scores.bed", "q2.fa_kmers_1_8_KLD_window_5000_increment_2500.p", "host.fa_kmers_1_8_genome.p"):
        assert (a / "temp" / f).read_bytes() == (b / "temp" / f).read_bytes(), f


def test_cli_scores_against_a_reference_pickle(tmp_path):
    """A genome pickle holding the reference's own tables (a golden's): the TSV rows are the golden's."""
    case = "c2_small_query_vs_c1_host"
    g = Golden(case)
    temp = tmp_path / "temp"
    temp.mkdir()
    with open(temp / "host.fa_kmers_1_8_genome.p", "wb") as fh:
        pickle.dump(engine.genome_kmers(g.tables, 1, 8, g.genome_meta), fh, protocol=2)
    query = tmp_path / "q.fa"
    query.write_bytes(synth.fasta_bytes(g.scaffolds()))
    _cli(["-H", str(tmp_path / "host.fa"), "-Q", str(query), "-t", str(temp), "--quiet", "--RIP"])
    lines = (temp / "raw_window_scores.bed").read_text().splitlines()
    assert lines[0].split("\t") == ["name", "start", "stop", "windowKLD", "GC", "PI", "SI", "CRI"]
    cells = [ln.split("\t") for ln in lines[1:]]
    res = engine.HotPathResult(1, 8, g.tables, tuple(int(x) for x in g.genome_meta), [c[0] for c in cells],
                               np.array([[int(c[1]), int(c[2])] for c in cells], np.int64),
                               np.array([[float(x) for x in c[3:]] for c in cells]), np.zeros(len(cells), np.uint32))
    _check_against_golden(res, g, case + "[CLI]")
