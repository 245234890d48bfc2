"""The nibble kernel's two other modes against the C oracle: one query against several backgrounds (MANY,
frisk_b200_background_score_many) and the k sweep (frisk_b200_score_sweep, kmax' = 1..8 from one pass).

Part 1 (CPU): a table of MANY cases -- (K, PP band, kmin = 1 / kmin > 1) -- and one of sweep cases -- one per PP band --
that provably reaches every MANY and sweep instantiation, each named by the one-background name with its mode set to 2
(MANY) or 1 (sweep).  Every family sees kmin > 1 (MANY), rip off and the separate CG-free host.

Part 2 (GPU): every MANY case at B = 2, 3 and 8 backgrounds built from oracle tables (the query's own, the CG-free
soft-masked host counted with --maskHost, seeded others, one handle twice at B = 8), and at B = 1, which is the
one-background call (score_many runs the MANY instantiation from two backgrounds on).  Per background: status and rows
against ``c_oracle.score``, no sentinel or hand-over marker left, bit for bit the one-background call, the reversed order
and a second call.  At B = 8 and PP 32 every background takes its own P3 pass; at PP <= 20 two share one, and B = 3 splits
a group.

Part 3 (GPU): the sweep of each PP band, on the query's own tables with rip and on the host's without, every kmax' against
the oracle at kmin 1 / kmax k'.  Windows of 1..9 bases, soft-masked edges (fewer upper-case bases than valid ones, so the
reference's ZeroDivisionError rule n_up == x - 1 can hold while x-mers exist) and words cut by a single N at 6 / 7 bases.

Part 4: windows just over and just under each nibble limit at PP 8 / 20 / 32, for K = 7 and 8: a K-mer seen 16 times vs 15,
the same K-mer in the top nibble of its 64-bit word (the carry out of it is lost), and more than 64 words cut at K-1 / K-2
bases vs 64.  CPU tests restate the rules in numpy; on the GPU every window is held to the oracle, for every background at
B = 3 and 8 and for every kmax' of the sweep, and to the one-background call's own hand-over.

Part 5 (GPU): the first window kernel a MANY or sweep call launches is the table's name.  Part 6 (GPU): FASTA text through
run_backgrounds at PP 8 and PP 32, where the window list is built on the device, equals each background's own run."""
import ctypes as C
import functools
import zlib
from collections import namedtuple

import numpy as np
import pytest

from frisk_b200 import _lib, synth
from tests.helpers import assert_rows_close, max_rel_err
from tests.test_bgzf_gpu import _same_result
from tests.test_kernel_matrix_gpu import (P8, P20, SMEM, UPPER_ACGT, _Builder, _nibble_wrap, _side_list, band, bases_of,
                                          case_windows, concat, kmer_codes, packed, query_scaffolds, side_words, valid_run, window_list)
from tests.test_kernel_matrix_gpu import devices, eng  # noqa: F401  (the matrix's module fixtures, shared here)
from tests.test_score_plan import _window_launches, forced, kernel_name

ROW_SENTINEL = 0x7FF4DEADBEEF0001                 # a NaN payload no kernel writes
STATUS_SENTINEL = 0x5A5A5A5A
SOFT = 75_000                                     # the mix scaffold is soft-masked from here (and upper case before)
SINGLE_N = 60_000                                 # ... and has single Ns at 60,000 + 97 j


# ---- part 1: the case tables ----------------------------------------------------------------------------------------

ManyCase = namedtuple("ManyCase", "opt kmin kmax lengths host rip n")
SweepCase = namedtuple("SweepCase", "kmin kmax lengths n")


def lengths(lo, hi, K):
    """The matrix's band, and every length 1..K+1."""
    return tuple(sorted(set(band(lo, hi, K)) | set(range(1, K + 2)), reverse=True))


def many(opt, kmin, K, lo, hi, host=False, rip=True):
    return ManyCase(opt, kmin, K, lengths(lo, hi, K), host, rip, 48)


MANY_CASES = [
    many(None, 1, 7, 1501, P8), many("force_nibble_kernel", 2, 7, 1, P8, host=True, rip=False),
    many(None, 1, 7, P8 + 1, P20, rip=False), many(None, 3, 7, P8 + 1, P20, host=True),
    many(None, 1, 7, P20 + 1, SMEM), many(None, 2, 7, P20 + 1, SMEM, host=True, rip=False),
    many(None, 1, 8, 1, P8, rip=False), many(None, 2, 8, 1, P8, host=True),
    many(None, 1, 8, P8 + 1, P20), many(None, 3, 8, P8 + 1, P20, host=True, rip=False),
    many(None, 1, 8, P20 + 1, SMEM, rip=False), many(None, 2, 8, P20 + 1, SMEM, host=True),
]
SWEEP_CASES = [SweepCase(1, 8, lengths(lo, hi, 8), 48) for lo, hi in ((1, P8), (P8 + 1, P20), (P20 + 1, SMEM))]

# every instantiation of the two modes in frisk_nibble.cu: MANY for K 7 / 8 x PP 8 / 20 / 32 x kmin 1 / any, the sweep
# for K 8 x PP 8 / 20 / 32
INSTANTIATIONS = ({"score_windows_nibble_kernel<%d, %d, 0, %d, 2>" % (K, pp, allk)
                   for K in (7, 8) for pp in (8, 20, 32) for allk in (0, 1)} |
                  {"score_windows_nibble_kernel<8, %d, 0, 1, 1>" % pp for pp in (8, 20, 32)})


def with_mode(name, mode):
    """The one-background nibble name with its mode argument set."""
    assert name.startswith("score_windows_nibble_kernel<") and name.endswith(", 0>"), name
    return name[:-2] + "%d>" % mode


def many_name(c):
    with forced(c.opt):
        return with_mode(kernel_name(c.kmin, c.kmax, max(c.lengths)), 2)


def sweep_name(c):
    return with_mode(kernel_name(1, 8, max(c.lengths)), 1)


def many_id(c):
    return "%sk%d_%d-w%d%s%s" % ("forced-" if c.opt else "", c.kmin, c.kmax, max(c.lengths), "-host" if c.host else "",
                                  "" if c.rip else "-norip")


def sweep_id(c):
    return "w%d" % max(c.lengths)


def test_case_tables_reach_every_instantiation():
    """kernel_name makes no CUDA call: the tables' reach is checked on any machine."""
    reached = [many_name(c) for c in MANY_CASES] + [sweep_name(c) for c in SWEEP_CASES]
    assert len(set(reached)) == len(reached) and set(reached) == INSTANTIATIONS, sorted(set(reached) ^ INSTANTIATIONS)
    for K in (7, 8):
        cs = [c for c in MANY_CASES if c.kmax == K]
        assert any(c.kmin > 1 for c in cs) and any(not c.rip for c in cs) and any(c.host for c in cs), K
        assert any(c.kmin == 1 and c.rip and not c.host for c in cs), K
        assert all(set(range(1, K + 2)) <= set(c.lengths) for c in cs)
    assert [c for c in MANY_CASES if c.kmax == 7 and max(c.lengths) <= 1500] == []      # the forced case keeps its band
    with forced("force_nibble_kernel"):
        assert kernel_name(2, 7, 1500).startswith("score_windows_nibble_kernel<7, 8,")
    assert kernel_name(2, 7, 1500).startswith("score_windows_direct_kernel")
    assert len({many_id(c) for c in MANY_CASES}) == len(MANY_CASES)


def edge_windows(K):
    """Short windows on the mix scaffold: across the upper / soft-masked edge (n_up below the valid bases: the reference's
    n_up == x - 1 rule can hold while x-mers exist) and around single Ns (words cut at K-2, K-1 and K bases)."""
    out = [(0, SOFT - u, u + extra) for u in range(1, K + 2) for extra in (1, 2, 3)]
    for j in (0, 5, 31):
        p = SINGLE_N + 97 * j
        for v in (K - 2, K - 1, K):
            out += [(0, p - v, v + 1), (0, p - v, v + 12), (0, p + 1, v), (0, p - 11, 12 + v)]
    return out


def test_edge_windows_have_their_features():
    mix = query_scaffolds()[0][1]
    assert np.all(UPPER_ACGT[mix[SOFT - 12:SOFT]]) and np.all(mix[SOFT:SOFT + 12] >= ord("a"))
    for j in (0, 5, 31):
        p = SINGLE_N + 97 * j
        assert mix[p] == ord("N") and np.all(UPPER_ACGT[mix[p - 20:p]]) and np.all(UPPER_ACGT[mix[p + 1:p + 21]])
    for K in (7, 8):
        cut = {int(valid_run(codes_of(mix[s:s + L]))[0]) for _, s, L in edge_windows(K) if mix[s + L - 1] == ord("N")}
        assert {K - 2, K - 1, K} <= cut


# ---- the backgrounds: the query's own, the CG-free host, seeded others ----------------------------------------------
# "query" names the kernel matrix query's own tables.  The hand-over tests of part 4 score another genome, and to them it
# is one more background among the others.

OTHERS = 5
MASKED_OTHER = 2                                  # other2 is counted with --maskHost


@functools.lru_cache(maxsize=None)
def other_scaffolds(i):
    rng = np.random.Generator(np.random.PCG64(7100 + i))
    s = synth.iid_bases(rng, 60_000 + 15_000 * i, 0.33 + 0.06 * i)
    s[5_000:9_000] |= 0x20
    return (("other%d" % i, s),)


@functools.lru_cache(maxsize=None)
def bg_tables(name, kmin, kmax):
    """Oracle tables and meta of a background (orders kmin..kmax)."""
    from oracle import c_oracle
    if name in ("query", "host"):
        seq, off, _ = concat(name == "host")
        return c_oracle.background(seq, off, kmin, kmax, name == "host", threads=8)
    i = int(name[5:])
    seq, off = c_oracle.concat(list(other_scaffolds(i)))
    return c_oracle.background(seq, off, kmin, kmax, i == MASKED_OTHER, threads=8)


def bg_order(host, B):
    """The backgrounds of a B-background call: the host first in a host case; one handle twice at B = 8."""
    order = (["host", "query"] if host else ["query"]) + ["other%d" % i for i in range(OTHERS)] + ([] if host else ["host"])
    return order[:B] if B < 8 else order + [order[0]]


@pytest.fixture(scope="module")
def bgs(eng):
    """name, kmin, kmax -> engine.Background of the oracle's tables (opened once per module)."""
    opened = {}

    def get(name, kmin, kmax):
        if (name, kmin, kmax) not in opened:
            tabs, meta = bg_tables(name, kmin, kmax)
            opened[name, kmin, kmax] = eng.Background(tabs, kmin, kmax, meta)
        return opened[name, kmin, kmax]
    yield get
    for bg in opened.values():
        bg.close()


# ---- oracle and comparison --------------------------------------------------------------------------------------------

def codes_of(s):
    """2-bit codes (A T G C = 0 1 2 3, the kernels' order) of a base array, -1 for anything that is no ACGT."""
    lut = np.full(256, -1, np.int64)
    for i, ch in enumerate(b"ATGC"):
        lut[ch] = lut[ch | 0x20] = i
    return lut[np.asarray(s, np.uint8)]


def oracle_windows(seqinfo, wins, tabs, meta, kmin, kmax, rip):
    """(rows, status, excluded, n_up) of windows (scaffold, start, length) of a concatenated genome."""
    from oracle import c_oracle
    seq, off, non = seqinfo
    coff = np.array([int(off[s]) + r for s, r, _ in wins], np.uint64)
    ln = np.array([w[2] for w in wins], np.uint32)
    rows, status = c_oracle.score(seq, coff, ln, tabs, meta, kmin, kmax, rip, threads=8)
    a = coff.astype(np.int64)
    n_non = non[a + ln] - non[a]
    return rows, status, n_non >= 0.3 * ln, ln.astype(np.int64) - n_non


def check_rows(rows, status, ref, ref_status, excluded, what):
    """One background's (or one kmax''s) rows of every window, excluded ones included, against the oracle."""
    assert not np.any(rows.view(np.uint64) == ROW_SENTINEL), what + ": a row was never written"
    assert not np.any(status == STATUS_SENTINEL), what + ": a status was never written"
    assert not np.any(status & 0x80000000), what + ": internal hand-over marker survived"
    assert np.all(status[excluded] == _lib.ROW_EXCLUDED) and np.isnan(rows[excluded]).all(), what + ": excluded windows"
    keep = ~excluded
    assert np.array_equal(status[keep], ref_status[keep] & 7), what + ": status"
    got, want = rows[keep].copy(), ref[keep].copy()
    bad = ref_status[keep] != 0
    got[bad, 0] = want[bad, 0] = 0.0
    assert_rows_close(got, want, rtol_kld=1e-6, rtol_other=1e-15, what=what)
    assert max_rel_err(rows[keep][~bad, 0], ref[keep][~bad, 0]) < 1e-10, what


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def run_many(eng, g, dq, wl, bl, rip):
    """frisk_b200_background_score_many into sentinel-filled, device-mapped host rows: (rows[B, n, 5], status[B, n]).

    The sentinel shows a row the kernels never wrote only because the rows are page-locked: the run path then has the
    kernels write straight into them (rows_for in frisk_run.cu) instead of copying back a device workspace, whose stale
    rows from an earlier identical call would hide an unwritten one."""
    import torch
    n, nb = len(wl), len(bl)
    rows_t = torch.empty((nb * n, 5), dtype=torch.float64).pin_memory()
    status_t = torch.empty((nb * n,), dtype=torch.int32).pin_memory()
    assert rows_t.is_pinned() and status_t.is_pinned()
    rows, status = rows_t.numpy(), status_t.numpy().view(np.uint32)
    rows.view(np.uint64)[:] = ROW_SENTINEL
    status[:] = STATUS_SENTINEL
    eng._score_many(bl, g, (dq.codes, dq.inv, dq.low), wl, rip, rows, status)
    return rows.reshape(nb, n, 5).copy(), status.reshape(nb, n).copy()


def check_many(eng, g, dq, seqinfo, wins, bgs, names, kmin, kmax, rip, what, again=True, refs=None):
    """One MANY call against the oracle per background, the one-background call, the reversed order and a second call.
    Returns {name: (status, n_up)}.  refs: the oracle's results by background name, kept across calls on these windows."""
    refs = {} if refs is None else refs
    wl = window_list(eng, g, wins)
    bl = [bgs(nm, kmin, kmax) for nm in names]
    B = len(bl)
    rows, status = run_many(eng, g, dq, wl, bl, rip)
    rev_rows, rev_status = run_many(eng, g, dq, wl, bl[::-1], rip)
    if again:
        rows2, status2 = run_many(eng, g, dq, wl, bl, rip)
        assert same_bits(rows2, rows) and np.array_equal(status2, status), what + ": second call"
    out = {}
    for b, nm in enumerate(names):
        w = "%s B=%d background %d (%s)" % (what, B, b, nm)
        if nm not in refs:
            refs[nm] = oracle_windows(seqinfo, wins, *bg_tables(nm, kmin, kmax), kmin, kmax, rip)
        ref, ref_status, excluded, n_up = refs[nm]
        check_rows(rows[b], status[b], ref, ref_status, excluded, w)
        one = bl[b].run_resident(dq, wins=wl, rip=rip, assemble_result=False)
        assert same_bits(rows[b], one.rows[:len(wl)]) and np.array_equal(status[b], one.status[:len(wl)]), w + ": one-background call"
        assert same_bits(rev_rows[B - 1 - b], rows[b]) and np.array_equal(rev_status[B - 1 - b], status[b]), w + ": reversed order"
        out[nm] = (status[b], n_up)
    return out


# ---- part 2: MANY against the oracle ----------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def query_seqinfo():
    return concat(False)


@pytest.mark.gpu
@pytest.mark.parametrize("c", MANY_CASES, ids=many_id)
def test_many_against_c_oracle(devices, bgs, c):
    eng, dq, _ = devices
    g = packed()[0]
    wins = case_windows(c, zlib.crc32(many_id(c).encode())) + edge_windows(c.kmax)
    assert {(int(g.scaf_off[s]) + r) % 32 for s, r, _ in wins} == set(range(32))
    refs = {}
    with forced(c.opt):
        for B in (1, 2, 3, 8):                   # B = 1: the one-background kernel; MANY from B = 2 on
            got = check_many(eng, g, dq, query_seqinfo(), wins, bgs, bg_order(c.host, B), c.kmin, c.kmax, c.rip, many_id(c),
                             refs=refs)
            for nm, (status, n_up) in got.items():
                zd = (status & _lib.ROW_KLD_ZERODIV) != 0
                # the query has every K-mer of its windows: its ZeroDivisionError rows are those of the n_up == x - 1
                # rule, which the short and soft-masked edge windows do reach
                if nm == "query":
                    assert not np.any(zd & ((n_up < c.kmin - 1) | (n_up > c.kmax - 1))), (many_id(c), B)
                if nm == "host" and c.kmin > 1:
                    assert np.any(zd & (n_up > c.kmax)), (many_id(c), B, "the host lacks K-mers of these windows")


# ---- part 3: the sweep against the oracle -----------------------------------------------------------------------------

def run_sweep(eng, dq, wl, tabs, meta, rip):
    """frisk_b200_score_sweep on the eight genome-IVOM tables of `tabs` (orders 1..8) into sentinel-filled device rows:
    ([rows of kmax' 1..8], [status of kmax' 1..8], the device window list and tables for further launches)."""
    import torch
    L = _lib.lib()
    dev = "cuda:0"
    n = len(wl)
    st = eng._stream_ptr(dev)
    d_tab = torch.from_numpy(tabs.view(np.int64).copy()).to(dev)
    space = int(meta[0]) - int(meta[2])
    d_ig = [torch.empty(2 * 4 ** k, dtype=torch.float64, device=dev) for k in range(1, 9)]
    for k in range(1, 9):
        _lib.check(L.frisk_b200_genome_ivom(eng._ptr(d_tab), 1, k, space, eng._ptr(d_ig[k - 1]), st), "frisk_b200_genome_ivom")
    d_rows = [torch.full((n, 5), ROW_SENTINEL, dtype=torch.int64, device=dev) for _ in range(8)]
    d_status = [torch.full((n,), STATUS_SENTINEL, dtype=torch.int32, device=dev) for _ in range(8)]
    d_off = torch.from_numpy(wl.off.view(np.int64)).to(dev)
    d_len = torch.from_numpy(wl.length.view(np.int32)).to(dev)
    ptrs = lambda ts: (C.c_void_p * 8)(*[C.c_void_p(t.data_ptr()) for t in ts])
    _lib.check(L.frisk_b200_score_sweep(eng._ptr(dq.codes), eng._ptr(dq.inv), eng._ptr(dq.low), eng._ptr(d_off), eng._ptr(d_len),
                                        n, wl.max_len, ptrs(d_ig), 8, int(rip), ptrs(d_rows), ptrs(d_status), st),
               "frisk_b200_score_sweep")
    torch.cuda.synchronize()
    rows = [r.cpu().numpy().view(np.float64) for r in d_rows]
    status = [s.cpu().numpy().view(np.uint32) for s in d_status]
    return rows, status, (d_off, d_len, d_ig)


def check_sweep(eng, dq, seqinfo, wins, which, rip, what):
    wl = window_list(eng, dq.host, wins)
    rows, status, dev = run_sweep(eng, dq, wl, *bg_tables(which, 1, 8), rip)
    for k in range(1, 9):
        ref, ref_status, excluded, _ = oracle_windows(seqinfo, wins, *bg_tables(which, 1, k), 1, k, rip)
        check_rows(rows[k - 1], status[k - 1], ref, ref_status, excluded, "%s %s kmax' %d" % (what, which, k))
    return wl, rows, status, dev


@pytest.mark.gpu
@pytest.mark.parametrize("c", SWEEP_CASES, ids=sweep_id)
def test_sweep_against_c_oracle(devices, c):
    eng, dq, _ = devices
    wins = case_windows(c, zlib.crc32(sweep_id(c).encode())) + edge_windows(8)
    for which, rip in (("query", True), ("host", False)):
        _, _, status, _ = check_sweep(eng, dq, query_seqinfo(), wins, which, rip, "sweep " + sweep_id(c))
        zd = [(s & _lib.ROW_KLD_ZERODIV) != 0 for s in status]
        assert np.any(zd[6] != zd[7]), "the n_up == x - 1 rule differs between kmax' 7 and 8 on some window"


# ---- part 4: hand-overs at every PP -----------------------------------------------------------------------------------

def _run_wrap(L, K, base, run, seed):
    """`run` copies of one base between two others: the K-mer base^K seen run - K + 1 times.  No other window position
    makes a K-mer of that base alone: every 8-mer that holds base^7 is the run's."""
    other = 0 if base == 3 else 3
    rep = lambda n: sum(base << (2 * i) for i in range(n))
    forbid = {rep(8)} | {(x << 14) | rep(7) for x in range(4)} | {(rep(7) << 2) | x for x in range(4)}
    b = _Builder(seed, forbid=forbid)
    b.fill(L // 3)
    b.put([other] + [base] * run + [other])
    b.fill(L - len(b.c))
    return b.codes()


def ho_windows(K, L):
    """{name: codes} of one hand-over launch: over and under each limit of the nibble kernel at K."""
    seed = 5000 + 100 * K + L // 1000
    out = {}
    for name, base in (("wrap", 0), ("top", 3)):             # AAA..A: nibble 0 of its word; CCC..C: nibble 15, the top
        for side, run in (("over", K + 15), ("under", K + 14)):
            out["%s_%s" % (name, side)] = (_nibble_wrap(L, run, seed) if K == 8 and base == 0
                                           else _run_wrap(L, K, base, run, seed + base))
    out["side_over"] = _side_list(L, 32, seed)
    out["side_under"] = _side_list(L, 31, seed)
    return out


HO_KEYS = [(K, L) for K in (7, 8) for L in (P8, P20, SMEM)]


def cut_words(c, K):
    """Words cut at K-1 or K-2 bases by an invalid base or the window end: the nibble kernel's side list."""
    v = valid_run(c)
    return int(np.count_nonzero((v == K - 1) | (v == K - 2)))


def kmer_counts(c, K):
    code, ok = kmer_codes(c, K)
    return np.bincount(code[ok], minlength=1 << (2 * K))


@pytest.mark.parametrize("K,L", HO_KEYS)
def test_hand_over_windows_have_their_property(K, L):
    """Each window crosses exactly the limit it is named for, or stays one step short of it and crosses nothing."""
    for name, codes in ho_windows(K, L).items():
        assert len(codes) == L, name
        cnt = kmer_counts(codes, K)
        side = cut_words(codes, K)
        if K == 8:
            assert side == side_words(codes), name
        over = name.endswith("_over")
        if name.startswith("side"):
            assert side == (66 if over else 64) and cnt.max() <= 15, (name, side, cnt.max())
        else:
            top = name.startswith("top")
            kap = (1 << (2 * K)) - 1 if top else 0
            assert cnt[kap] == (16 if over else 15), (name, cnt[kap])
            assert (kap & 15 == 15) == top                  # nibble 15 of its bucket: the top of the 64-bit word
            others = np.delete(cnt, kap)
            assert others.max() <= 15 and side <= 64, (name, others.max(), side)


@functools.lru_cache(maxsize=None)
def ho_scaffolds():
    sc = []
    for K, L in HO_KEYS:
        pad = np.random.Generator(np.random.PCG64(K * 100_000 + L))
        for name, codes in ho_windows(K, L).items():
            lead = 32 + (len(sc) * 13) % 32
            sc.append(("%s_k%d_w%d" % (name, K, L), lead,
                       np.concatenate([synth.iid_bases(pad, lead, 0.5), bases_of(codes), synth.iid_bases(pad, 50, 0.5)])))
    return sc


@functools.lru_cache(maxsize=None)
def ho_seqinfo():
    from oracle import c_oracle
    seq, off = c_oracle.concat([(n, s) for n, _, s in ho_scaffolds()])
    return seq, off, np.concatenate([[0], np.cumsum(~UPPER_ACGT[seq], dtype=np.int64)])


@pytest.fixture(scope="module")
def ho_genome(eng):
    g = eng.PackedGenome.from_scaffolds([(n, s) for n, _, s in ho_scaffolds()])
    return g, eng.DeviceGenome(g)


def ho_launch(K, L):
    """(window list entries, names) of one hand-over launch."""
    sc = ho_scaffolds()
    idx = [i for i, (n, _, _) in enumerate(sc) if n.endswith("_k%d_w%d" % (K, L))]
    return [(i, sc[i][1], L) for i in idx], [sc[i][0].split("_k")[0] for i in idx]


@pytest.mark.gpu
@pytest.mark.parametrize("K,L", HO_KEYS)
def test_many_hand_overs(eng, bgs, ho_genome, K, L):
    g, dq = ho_genome
    wins, names = ho_launch(K, L)
    assert len(wins) == 6 and kernel_name(1, K, L) == "score_windows_nibble_kernel<%d, %d, 0, 1, 0>" % (K, {P8: 8, P20: 20, SMEM: 32}[L])
    refs = {}
    for B in (3, 8):
        got = check_many(eng, g, dq, ho_seqinfo(), wins, bgs, bg_order(False, B), 1, K, True, "hand-over k%d w%d" % (K, L),
                         again=False, refs=refs)
        for status, _ in got.values():
            assert not np.any(status & _lib.ROW_EXCLUDED)


@pytest.mark.gpu
@pytest.mark.parametrize("L", (P8, P20, SMEM))
def test_sweep_hand_overs(eng, ho_genome, L):
    import torch
    g, dq = ho_genome
    wins, names = ho_launch(8, L)
    wl, rows, status, (d_off, d_len, d_ig) = check_sweep(eng, dq, ho_seqinfo(), wins, "query", True, "sweep hand-over w%d" % L)
    # kmax' 8 of a window over a limit: the one-background call's own hand-over, bit for bit
    n = len(wl)
    d_rows = torch.empty((n, 5), dtype=torch.float64, device="cuda:0")
    d_status = torch.empty((n,), dtype=torch.int32, device="cuda:0")
    _lib.check(_lib.lib().frisk_b200_score(eng._ptr(dq.codes), eng._ptr(dq.inv), eng._ptr(dq.low), eng._ptr(d_off), eng._ptr(d_len), n,
                                           wl.max_len, eng._ptr(d_ig[7]), 1, 8, 1, eng._ptr(d_rows), eng._ptr(d_status), None,
                                           eng._stream_ptr("cuda:0")), "frisk_b200_score")
    torch.cuda.synchronize()
    one_rows, one_status = d_rows.cpu().numpy(), d_status.cpu().numpy().view(np.uint32)
    for i, name in enumerate(names):
        if name.endswith("_over"):
            assert same_bits(rows[7][i], one_rows[i]) and status[7][i] == one_status[i], (L, name)


# ---- part 5: the launched kernel is the named one ---------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("c", MANY_CASES, ids=many_id)
def test_many_launches_the_named_kernel(devices, bgs, tmp_path, c):
    eng, dq, _ = devices
    g = packed()[0]
    wl = window_list(eng, g, case_windows(c, 1))
    bl = [bgs(nm, c.kmin, c.kmax) for nm in bg_order(c.host, 2)]
    with forced(c.opt):
        launches, _ = _window_launches(lambda: run_many(eng, g, dq, wl, bl, c.rip), tmp_path)
    assert launches and launches[0] == (many_name(c), 256), launches


@pytest.mark.gpu
@pytest.mark.parametrize("c", SWEEP_CASES, ids=sweep_id)
def test_sweep_launches_the_named_kernel(devices, tmp_path, c):
    eng, dq, _ = devices
    wl = window_list(eng, packed()[0], case_windows(c, 1))
    launches, _ = _window_launches(lambda: run_sweep(eng, dq, wl, *bg_tables("query", 1, 8), True), tmp_path)
    assert launches and launches[0] == (sweep_name(c), 256), launches


# ---- part 6: the device-built window list at PP 8 and 32 --------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("w,step", [(2000, 1000), (8000, 4000)])
@pytest.mark.parametrize("kmax", [7, 8])
@pytest.mark.parametrize("kmin", [1, 3])
def test_run_backgrounds_from_text_at_pp8_and_pp32(eng, bgs, kmin, kmax, w, step):
    assert kernel_name(kmin, kmax, w) == "score_windows_nibble_kernel<%d, %d, 0, %d, 0>" % (kmax, 8 if w <= P8 else 32, kmin == 1)
    text = synth.fasta_bytes(list(query_scaffolds()[:1]))
    bl = [bgs(nm, kmin, kmax) for nm in ("query", "host", "other0")]
    got = eng.run_backgrounds(bl, text, kind="text", w=w, step=step)
    assert len(got) == 3 and len(got[0].rows) > 50
    for b, bg in enumerate(bl):
        _same_result(got[b], bg.run(text, kind="text", w=w, step=step), "w%d k%d_%d background %d" % (w, kmin, kmax, b))
