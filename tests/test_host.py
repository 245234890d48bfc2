"""CPU tests of the host side of the product (packing, FASTA scan, window enumeration) and of the
C-ABI surface.  No compute kernels are called (there is no GPU here and no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from oracle import c_oracle
from tests.helpers import Golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "frisk_b200.h")).read()
    declared = set(re.findall(r"\b(frisk_b200_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.PROTOTYPES), "header and ctypes prototypes must list the same entry points"
    L = _lib.lib()
    for name in declared:
        assert hasattr(L, name), name
    assert L.frisk_b200_abi_version() == 2
    assert _lib.table_size(1, 8) == 87380 and _lib.table_size(4, 8) == 87380 - 84


def test_fails_loudly_without_a_gpu():
    """Runs in a child process that sees no CUDA device, so the check holds on machines with a GPU too."""
    code = ("import pytest\n"
            "from frisk_b200 import _lib, engine, synth\n"
            "assert _lib.device_count() == 0\n"
            "g = engine.PackedGenome.from_scaffolds(synth.make('edge'))\n"
            "with pytest.raises(_lib.FriskError) as ei:\n"
            "    engine.run(g)\n"
            "assert ei.value.code == _lib.E_NO_DEVICE\n"
            "with pytest.raises(_lib.FriskError):\n"
            "    engine.run_host(g)\n"
            "print('no device: refused')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert out.returncode == 0 and "no device: refused" in out.stdout, out.stdout[-1000:] + out.stderr[-3000:]


def _unpack(g, s):
    off, ln = int(g.scaf_off[s]), int(g.scaf_len[s])
    pos = off + np.arange(ln)
    code = (g.codes[pos >> 4] >> (30 - 2 * (pos & 15)).astype(np.uint32)) & 3
    inv = (g.inv[pos >> 5] >> (31 - (pos & 31)).astype(np.uint32)) & 1
    low = ((g.low[pos >> 5] >> (31 - (pos & 31)).astype(np.uint32)) & 1) if g.low is not None else np.zeros(ln, np.uint32)
    return code, inv.astype(bool), low.astype(bool)


def test_pack_round_trip_and_stats():
    sc = synth.make("edge")
    g = engine.PackedGenome.from_scaffolds(sc, threads=3)
    letters = np.frombuffer(b"ATGC", dtype=np.uint8)
    for s, (name, seq) in enumerate(sc):
        code, inv, low = _unpack(g, s)
        rebuilt = letters[code]
        rebuilt = np.where(low, rebuilt + 32, rebuilt)
        valid = ~inv
        assert np.array_equal(rebuilt[valid], seq[valid]), name
        is_acgt = np.isin(seq, np.frombuffer(b"ACGTacgt", dtype=np.uint8))
        assert np.array_equal(valid, is_acgt), name
        # >= 1 padding base after the scaffold, flagged invalid
        p = int(g.scaf_off[s]) + len(seq)
        assert (g.inv[p >> 5] >> (31 - (p & 31))) & 1
    assert g.total_len == synth.total_bases(sc)
    upper = sum(int(np.isin(s, np.frombuffer(b"ACGT", dtype=np.uint8)).sum()) for _, s in sc)
    assert g.nn_total == g.total_len - upper              # countN semantics, F:106-118
    assert np.all(g.scaf_off % 128 == 0) and g.padded_len % 128 == 0
    assert g.padded_len - (int(g.scaf_off[-1]) + int(g.scaf_len[-1])) >= 128
    # trailing padding is all-invalid
    assert np.all(g.inv[-4:] == 0xFFFFFFFF)


def test_window_list_outside_the_planes_is_refused():
    """A window that reaches beyond the packed planes (or is longer than the declared maximum) would fault inside the
    score kernel; the one-call entry points check the (host-side) list first and return FRISK_E_INVALID."""
    g = engine.PackedGenome.from_scaffolds(synth.make("edge"))
    wins = g.windows()
    out = engine.HostOutputs(len(wins), 8, pinned=False)
    for mutate in (lambda w: w.off.__setitem__(3, np.uint64(g.padded_len - 100)),      # runs past the end
                   lambda w: w.off.__setitem__(0, np.uint64(2 ** 63)),                  # wrapped offset
                   lambda w: w.length.__setitem__(5, np.uint32(0))):
        bad = engine.WindowList(wins.off.copy(), wins.length.copy(), wins.scaf, wins.start, wins.stop)
        mutate(bad)
        P = engine._ptr
        rc = _lib.lib().frisk_b200_run_host(P(g.codes), P(g.inv), P(g.low), g.padded_len, P(g.codes), P(g.inv), P(g.low), g.padded_len,
                                            P(bad.off), P(bad.length), len(bad), wins.max_len, 1, 8, 0, 1, g.genome_space,
                                            P(out.rows), P(out.status), P(out.tables), P(out.valid), None)
        assert rc == _lib.E_INVALID                      # (checked before any device work: also without a GPU)


def test_whitespace_inside_a_sequence_line_is_refused():
    """F:149 strips a line only at its ends; interior whitespace would be part of the reference's sequence string.
    The scanner refuses it (FRISK_E_FORMAT) rather than dropping it and shifting every later coordinate."""
    for text in (b">a\nAC GT\n", b">a\nACGT\n>b\nAC\tGT\n", b">a\nAC\rGT\n"):
        with pytest.raises(_lib.FriskError) as ei:
            engine.PackedGenome.from_fasta_bytes(text)
        assert ei.value.code == _lib.E_FORMAT
    g = engine.PackedGenome.from_fasta_bytes(b"junk with spaces\n>a\n  ACGT \t \r\n\tGG\r\n   \n>b x y\nAC\n")
    assert g.names == ["a", "b"] and list(g.scaf_len) == [6, 2]


def test_no_lowercase_means_no_low_plane():
    g = engine.PackedGenome.from_scaffolds(synth.make("C1", 0.004))
    assert g.low is None and g.n_lower == 0 and g.nn_total == 0


def test_fasta_scan_matches_reference_rules(tmp_path):
    text = (b"leading junk before any header\n"
            b">>seq1 description words\nACGT\n  \nacgtNN\r\n"
            b">seq2\tother\n\nAC\nGT\n"
            b">empty_record\n"
            b">last\nTTTT")
    g = engine.PackedGenome.from_fasta_bytes(text)
    assert g.names == ["seq1", "seq2", "empty_record", "last"]         # F:156 token rule
    assert list(g.scaf_len) == [10, 4, 0, 4]
    assert g.total_len == 18 and g.nn_total == 6 and g.n_lower == 4
    sc = synth.make("edge")
    p = tmp_path / "edge.fa"
    synth.write_fasta(sc, str(p))
    a = engine.PackedGenome.from_fasta(str(p))
    b = engine.PackedGenome.from_scaffolds(sc)
    assert a.names == b.names
    for f in ("codes", "inv", "low"):
        assert np.array_equal(getattr(a, f), getattr(b, f))
    import gzip
    with gzip.open(str(p) + ".gz", "wb") as fh:
        fh.write(p.read_bytes())
    c = engine.PackedGenome.from_fasta(str(p) + ".gz")
    assert np.array_equal(c.codes, b.codes)


@pytest.mark.parametrize("w,step,sa", [(5000, 2500, False), (5000, 2500, True), (1000, 250, False), (3000, 1000, True),
                                       (4000, 1000, False), (5000, 5000, False), (700, 900, True),
                                       # 0.75 w < step < w: scaffolds SHORTER than the window are windowed (F:231 negative slice)
                                       (5000, 4000, False), (1000, 800, False), (1000, 800, True), (100, 80, False), (1000, 999, True)])
def test_window_enumeration_matches_oracle(w, step, sa):
    """Candidates minus the 30 % rule (applied on the device) == crawlGenome (oracle)."""
    sc = synth.make("edge") + synth.make("C5", 0.00002, seed=3) + synth.make("edge_short")
    rng = np.random.default_rng(w * 7 + step)
    sc += [("near_w_%d" % k, synth.iid_bases(rng, int(n), 0.5)) for k, n in
           enumerate(rng.integers(max(min(int(1.75 * w - step), w) - 3, 1), w + 4, 12))]
    g = engine.PackedGenome.from_scaffolds(sc)
    wins = g.windows(w, step, sa)
    seq, off = c_oracle.concat(sc)
    sidx, woff, wlen, st, sp = c_oracle.crawl(seq, off, w, step, sa)
    # apply the reference's 30 % rule on the host for the comparison
    keep = []
    for i in range(len(wins)):
        s = int(wins.scaf[i]); o = int(wins.off[i] - g.scaf_off[s]); l = int(wins.length[i])
        chunk = sc[s][1][o:o + l]
        bad = l - int(np.isin(chunk, np.frombuffer(b"ACGT", dtype=np.uint8)).sum())
        keep.append(not (bad >= 0.3 * l))
    keep = np.array(keep, bool)
    assert np.array_equal(wins.scaf[keep].astype(np.int64), sidx)
    assert np.array_equal(wins.start[keep], st) and np.array_equal(wins.stop[keep], sp)
    assert np.array_equal(wins.length[keep], wlen)
    rel = wins.off[keep] - g.scaf_off[wins.scaf[keep]]
    assert np.array_equal(rel, woff - off[sidx])
    # ... and == the Python oracle, which keeps the reference's own slicing expression (F:231: a negative
    # start when size < w); the C oracle above restates it with explicit arithmetic
    from oracle import frisk_oracle
    py = list(frisk_oracle.crawl_genome([(n, s.tobytes().decode()) for n, s in sc], w, step, sa))
    assert [(a, b) for _, _, a, b in py] == list(zip(st.tolist(), sp.tolist()))
    assert [len(x[0]) for x in py] == wlen.tolist()
    assert all(x[0] == sc[int(s)][1][int(o - off[s]):int(o - off[s]) + int(l)].tobytes().decode()
               for x, s, o, l in zip(py, sidx, woff, wlen))


def test_window_rows_match_reference_golden_coords():
    g = Golden("edge_default")
    pg = engine.PackedGenome.from_scaffolds(g.scaffolds())
    wins = pg.windows()
    # duplicate tail window when size % step == 0 (SURVEY section 4.1): 15001-20000 then 15000-20000
    a = [(int(s), int(e)) for s, e, c in zip(wins.start, wins.stop, wins.scaf) if c == 0]
    assert a[-2:] == [(15001, 20000), (15000, 20000)]


def test_long_windows_are_enumerated():
    """Windows beyond the shared-memory kernels' 65,535 bases are legal (general kernel)."""
    g = engine.PackedGenome.from_scaffolds([("big", synth.iid_bases(np.random.default_rng(1), 300_000, 0.5))])
    wins = g.windows(70_000, 35_000)
    assert wins.max_len == 70_000 and len(wins) == 8          # j = 0, 35k, ..., 245k (F:228): the last two jump back
    assert _lib.MAX_K == 12 and _lib.MAX_WINDOW == 0x7FFFFFFF


def test_sparse_form_of_the_invalid_plane():
    """frisk_b200_plane_sparse: the non-zero words of a plane, in order; rebuilding the plane from them is exact."""
    for sc in (synth.make("edge"), synth.make("C2", 0.02), [("allN", np.full(1000, ord("N"), np.uint8))]):
        g = engine.PackedGenome.from_scaffolds(sc)
        idx, val = g.inv_sparse()
        nz = np.nonzero(g.inv)[0]
        assert np.array_equal(idx, nz.astype(np.uint32)) and np.array_equal(val, g.inv[nz])
        rebuilt = np.zeros_like(g.inv)
        rebuilt[idx] = val
        assert np.array_equal(rebuilt, g.inv)
    n = C.c_uint64(0)
    rc = _lib.lib().frisk_b200_plane_sparse(engine._ptr(g.inv), g.inv.shape[0], 1, engine._ptr(np.zeros(1, np.uint32)),
                                            engine._ptr(np.zeros(1, np.uint32)), C.byref(n))
    assert rc == _lib.E_CAPACITY and n.value == len(idx)


def test_tsv_formatter_writes_floats_like_python():
    """frisk_b200_format_rows vs "\\t".join(str(v) ...) (what the reference's handle.write does, F:1493)."""
    rng = np.random.default_rng(12)
    n = 20000
    special = np.array([0.0, -0.0, 1.0, 100000.0, 1e15, 1e16, 1e17, 1.5e16, 123456789012345680000.0, 0.0001, 0.00001, 1e-5 * 1.5,
                        5e-324, 1.7976931348623157e308, np.nan, np.inf, -np.inf, 0.1, 1 / 3, 2 / 3, 0.5, 2500 / 5000, 1e22, 1e23,
                        9007199254740993.0, 0.30000000000000004, -2.5e-7, 12345.678, 4.35, 0.000123456789])
    vals = np.concatenate([special, rng.random(n), rng.normal(size=n) * 10.0 ** rng.integers(-12, 12, n),
                           rng.integers(0, 5001, n) / rng.integers(1, 5001, n)])
    vals = np.resize(vals, (len(vals) // 5) * 5).reshape(-1, 5)
    m = len(vals)
    names = ["scaffold_%d" % i for i in range(7)] + ["x"]
    res = engine.HotPathResult(1, 8, np.zeros(0, np.uint64), (0, 0, 0), [], np.stack([np.arange(m) * 2500 + 1, np.arange(m) * 2500 + 5000], 1),
                               vals, np.zeros(m, np.uint32), m, np.arange(m), rng.integers(0, len(names), m), None, scaf_names=names)
    for with_rip in (True, False):
        nv = 5 if with_rip else 2
        want = "".join("\t".join([names[int(s)], str(int(a)), str(int(b))] + [str(float(v)) for v in row[:nv]]) + "\n"
                       for s, (a, b), row in zip(res.row_scaf, res.coords, vals))
        assert res.tsv_body(with_rip).decode() == want
    empty = engine.HotPathResult(1, 8, np.zeros(0, np.uint64), (0, 0, 0), [], np.zeros((0, 2), np.int64), np.zeros((0, 5)),
                                 np.zeros(0, np.uint32), 0, np.zeros(0, np.int64), np.zeros(0, np.int64), None, scaf_names=names)
    assert empty.tsv_body(True) == b""


def test_argument_checks_answer_before_any_device_work():
    """Bad arguments are refused with FRISK_E_INVALID / FRISK_E_UNSUPPORTED by every entry point, without a GPU
    (nothing is dereferenced or launched before the checks)."""
    L = _lib.lib()
    dummy = np.zeros(64, np.uint64)
    p = engine._ptr(dummy)
    null = C.c_void_p(0)
    n = C.c_uint64(0)
    assert L.frisk_b200_background(null, p, null, 0, 64, 8, 0, p, null) == _lib.E_INVALID
    assert L.frisk_b200_background(p, p, null, 16, 64, 8, 0, p, null) == _lib.E_INVALID            # not a multiple of 32
    assert L.frisk_b200_background(p, p, null, 0, 64, 13, 0, p, null) == _lib.E_UNSUPPORTED
    assert L.frisk_b200_background(p, p, null, 64, 64, 8, 0, p, null) == _lib.OK                    # empty range: nothing to do
    assert L.frisk_b200_finalize_tables(null, 8, 1, p, null, null) == _lib.E_INVALID
    assert L.frisk_b200_genome_ivom(p, 3, 2, 1000, p, null) == _lib.E_INVALID                       # kmin > kmax
    assert L.frisk_b200_genome_ivom(p, 1, 13, 1000, p, null) == _lib.E_UNSUPPORTED
    assert L.frisk_b200_score(p, p, null, p, p, 0, 5000, p, 1, 8, 1, p, p, null, null) == _lib.OK   # no windows
    assert L.frisk_b200_score(p, p, null, p, p, 10, 5000, null, 1, 8, 1, p, p, null, null) == _lib.E_INVALID
    assert L.frisk_b200_windows(p, p, 1, 0, 2500, 0, 0, null, null, null, null, null, C.byref(n)) == _lib.E_INVALID
    assert L.frisk_b200_feature_slots(1, 8, null, C.byref(n)) == _lib.E_UNSUPPORTED
    assert L.frisk_b200_feature_slots(3, 2, null, C.byref(n)) == _lib.E_INVALID
    assert L.frisk_b200_format_rows(null, null, null, null, null, null, null, 0, 6, null, 0, C.byref(n), 1) == _lib.E_INVALID
    assert L.frisk_b200_finalize_tables_peers(null, null, 0, 2, 1, 8, 1, p, null, null) == _lib.E_INVALID
    assert L.frisk_b200_run_host(p, null, null, 128, p, p, null, 128, null, null, 0, 0, 1, 8, 0, 1, 100, null, null, null, null,
                                 null) == _lib.E_INVALID
    assert L.frisk_b200_run_resident(p, p, null, 100, p, p, null, 128, null, null, 0, 0, 1, 8, 0, 1, 100, null, null, null, null,
                                     null) == _lib.E_INVALID                                         # padded_len % 128
    assert b"unsupported" in L.frisk_b200_strerror(_lib.E_UNSUPPORTED) and L.frisk_b200_strerror(-99) == b"unknown error"
    assert L.frisk_b200_set_option(b"no_such_option", 1) == _lib.E_INVALID
    assert L.frisk_b200_set_option(None, 1) == _lib.E_INVALID
    # frisk_b200_run_fasta: argument checks come before anything touches a device; without a GPU it says so
    hh, qh = C.c_void_p(), C.c_void_p()
    txt = np.frombuffer(b">a\nACGT\n", dtype=np.uint8)
    tp = C.c_void_p(txt.ctypes.data)
    assert L.frisk_b200_run_fasta(tp, 8, null, 0, 5000, 2500, 0, 1, 8, 0, 1, 0, null, null, null, null, C.byref(n), None,
                                  C.byref(qh), null) == _lib.E_INVALID                               # no place for the handle
    assert L.frisk_b200_run_fasta(null, 8, null, 0, 5000, 2500, 0, 1, 8, 0, 1, 0, null, null, null, null, C.byref(n),
                                  C.byref(hh), C.byref(qh), null) == _lib.E_INVALID                  # text missing
    assert L.frisk_b200_run_fasta(tp, 8, null, 0, 5000, 2500, 0, 1, 8, 0, 1, 4, null, null, null, null, C.byref(n),
                                  C.byref(hh), C.byref(qh), null) == _lib.E_INVALID                  # rows_cap without rows
    assert L.frisk_b200_run_fasta(tp, 8, null, 0, 5000, 2500, 0, 3, 2, 0, 1, 0, null, null, null, null, C.byref(n),
                                  C.byref(hh), C.byref(qh), null) == _lib.E_INVALID                  # kmin > kmax
    assert L.frisk_b200_run_fasta(tp, 8, null, 0, 0, 2500, 0, 1, 8, 0, 1, 0, null, null, null, null, C.byref(n),
                                  C.byref(hh), C.byref(qh), null) == _lib.E_INVALID                  # window length 0
    if L.frisk_b200_device_count() <= 0:
        assert L.frisk_b200_run_fasta(tp, 8, null, 0, 5000, 2500, 0, 1, 8, 0, 1, 0, null, null, null, null, C.byref(n),
                                      C.byref(hh), C.byref(qh), null) == _lib.E_NO_DEVICE
        assert not hh.value and not qh.value
    stats2 = np.zeros(2, np.uint64)
    assert L.frisk_b200_fasta_open_stats(C.c_void_p(stats2.ctypes.data)) == _lib.OK
    assert L.frisk_b200_fasta_open_stats(null) == _lib.E_INVALID
    assert L.frisk_b200_fasta_info(null, None, None, null) == _lib.E_INVALID
    assert L.frisk_b200_fasta_planes(null, None, None, None) == _lib.E_INVALID
    for opt in (b"force_dense_kernel", b"force_general_kernel", b"force_bucket_kernel", b"force_direct_kernel",
                b"force_nibble_kernel", b"ingest_exact_open", b"ingest_chunk_tiles"):
        assert L.frisk_b200_set_option(opt, 1) == 0 and L.frisk_b200_set_option(opt, 0) == 0, opt   # the switches in the header


def test_assemble_copies_or_gathers_the_same_rows():
    """engine.assemble takes plain copies when no window is excluded and gathers otherwise: same fields either way, and the
    result never aliases the (reused, page-locked) buffers it was built from."""
    rng = np.random.default_rng(4)
    sc = [("s%d" % i, np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, int(n))]) for i, n in enumerate((9000, 30000, 700, 12000))]
    g = engine.PackedGenome.from_scaffolds(sc)
    wins = g.windows(1000, 500, True)
    n = len(wins)
    assert n > 50 and wins.max_len == 1000 and wins.max_len == int(wins.length.max())
    rows = rng.random((n, 5))
    tables = np.arange(_lib.table_size(1, 3), dtype=np.uint64)
    for excluded in ([], [0, 7, n - 1]):
        status = np.zeros(n, np.uint32)
        status[excluded] = _lib.ROW_EXCLUDED
        res = engine.assemble(g, g, wins, tables, 123, rows, status, 1, 3)
        keep = np.setdiff1d(np.arange(n), excluded)
        assert np.array_equal(res.rows, rows[keep]) and np.array_equal(res.win_index, keep)
        assert np.array_equal(res.coords[:, 0], wins.start[keep]) and np.array_equal(res.coords[:, 1], wins.stop[keep])
        assert res.names == [g.names[s] for s in wins.scaf[keep]] and np.array_equal(res.row_scaf, wins.scaf[keep])
        assert res.n_candidates == n and not np.shares_memory(res.rows, rows)
        lean = engine.assemble(g, g, wins, tables, 123, rows, status, 1, 3, names=False)
        assert lean.names == [] and np.array_equal(lean.rows, res.rows)
