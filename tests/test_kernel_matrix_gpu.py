"""Every window kernel the planner can pick, and every hand-over of the extension kernel, against the C oracle.

Part 1 (CPU): a table of cases -- (forced kernel, kmin, kmax, window lengths, background, rip) -- that provably reaches
every kernel name of ``test_score_plan.EXPECTED`` (and a few variants that table does not list), with each switch (kmin > 1,
rip off, a separate soft-masked host that lacks the CG dinucleotide) seen by every kernel family.  A variant added to the
planner later fails here until it has a case.

Part 2 (GPU): every case on one launch of hand-picked windows -- every start offset mod 32, the longest length of the
variant's band and the three below it, the shortest, and 1, K-1, K, K+1 -- against ``c_oracle.score``: tables and meta
bit-exact, status bits equal, rows to 1e-10, a second run bit-identical, and (kmax <= 8) every window's tables from the
dump instantiation equal to ``c_oracle.window_tables``.

Part 3: the four reasons the kmax 9..12 extension kernel hands a window to the general kernel -- an 8-mer seen 16 times,
more than 64 words cut at 7 / 6 bases, more than 2,560 hash registrations, a probe chain longer than 64 -- each built just
over and just under its limit.  The CPU tests restate the kernel's rules in numpy and prove each window has the property
it claims; the GPU test checks every window against the oracle and the windows over a limit bit for bit against a forced
general-kernel run (the general kernel's result does not depend on its CTA or grid, so equality shows the hand-over).

Part 4 (GPU): the background counter's 16-bit shared-memory halves wrap at every word size 1..8, on all-valid words and on
words that hold an N, with a pigeonhole check that proves a wrap happened."""
import functools
import zlib
from collections import namedtuple

import numpy as np
import pytest

from frisk_b200 import _lib, synth
from tests.helpers import assert_rows_close, max_rel_err
from tests.test_score_plan import EXPECTED, forced, kernel_name

A, G, C = (ord(ch) for ch in "AGC")
N = ord("N")
UPPER_ACGT = np.zeros(256, bool)
UPPER_ACGT[list(b"ATGC")] = True


@pytest.fixture(scope="module")
def eng():
    from frisk_b200 import engine
    _lib.require_device()          # fail loudly: no CPU fallback exists
    return engine


# ---- numpy restatements of the kernels' rules -----------------------------------------------------------------------

def kmer_codes(c, x):
    """Codes of the x-mers starting at every position of the code array c (first base most significant) and whether
    all x bases are valid."""
    n = len(c) - x + 1
    if n <= 0:
        return np.zeros(0, np.int64), np.zeros(0, bool)
    code = np.zeros(n, np.int64)
    ok = np.ones(n, bool)
    for i in range(x):
        ci = c[i:i + n]
        ok &= ci >= 0
        code = (code << 2) | np.maximum(ci, 0)
    return code, ok


def valid_run(c):
    """Valid bases from each position up to the next invalid base or the window end."""
    n = len(c)
    nxt = np.where(c < 0, np.arange(n), n)
    nxt = np.minimum.accumulate(nxt[::-1])[::-1]
    return nxt - np.arange(n)


def kmer8_counts(c):
    code, ok = kmer_codes(c, 8)
    return np.bincount(code[ok], minlength=1 << 16)


def side_words(c):
    """Words cut at 7 or 6 valid bases (by an invalid base or the window end): the extension kernel's side list."""
    v = valid_run(c)
    return int(np.count_nonzero((v == 6) | (v == 7)))


def ext_tag(x, code):
    return 1 + (((x - 9) << 24) | code)


def ext_slot(tag):
    return ((np.asarray(tag, np.uint64) * np.uint64(2654435761)) & np.uint64(0xffffffff)) >> np.uint64(20)


def ext_registrations(c, K):
    """The extension kernel's P3: per order x = 9..K, the tags registered in the hash, one per position whose
    (x-1)-prefix repeats (order 9: its 8-mer count >= 2; above: it registered at x-1 and that key's count is >= 2)."""
    v = valid_run(c)
    cnt8 = kmer8_counts(c)
    c8, _ = kmer_codes(c, 8)
    out = []
    prev_reg = prev_code = None
    for x in range(9, K + 1):
        code, _ = kmer_codes(c, x)
        n = len(code)
        if x == 9:
            rep = cnt8[c8[:n]] >= 2
        else:
            keys, counts = np.unique(prev_code[prev_reg], return_counts=True)
            seen = np.zeros(n, np.int64)
            if len(keys):
                at = np.minimum(np.searchsorted(keys, prev_code[:n]), len(keys) - 1)
                seen = np.where(keys[at] == prev_code[:n], counts[at], 0)
            rep = prev_reg[:n] & (seen >= 2)
        reg = rep & (v[:n] >= x)
        out.append(ext_tag(x, code[reg]))
        prev_reg, prev_code = reg, code
    return out


def hash_probe_bounds(tags):
    """Linear probing over 4,096 slots leaves the same occupied set whatever the insertion order.  Returns (the most keys
    sharing one home slot, the longest run of occupied slots starting at any key's home).  65+ keys on one home force a
    probe chain longer than 64; no run from a home longer than 64 slots rules one out."""
    keys = np.unique(np.concatenate(tags)) if tags else np.zeros(0, np.int64)
    homes = ext_slot(keys).astype(np.int64)
    occ = np.zeros(4096, bool)
    for h in np.sort(homes):                      # any order gives the same occupied set
        s = int(h)
        while occ[s]:
            s = (s + 1) & 4095
        occ[s] = True
    run = np.zeros(8192, np.int64)                # occupied slots from s on (the table wraps around)
    o2 = np.concatenate([occ, occ])
    for s in range(8191, -1, -1):
        run[s] = run[s + 1] + 1 if s < 8191 and o2[s] else int(o2[s])
    most = int(np.bincount(homes, minlength=4096).max()) if len(homes) else 0
    return most, int(run[homes].max()) if len(homes) else 0


def bases_of(codes):
    return np.where(codes < 0, N, np.frombuffer(b"ATGC", np.uint8)[np.maximum(codes, 0)]).astype(np.uint8)


# ---- genomes --------------------------------------------------------------------------------------------------------

def _cg_free(s):
    """No C followed by G (either case): turning that G into an A cannot make a new CG."""
    up = s & 0xDF
    m = (up[:-1] == C) & (up[1:] == G)
    s[1:][m] = (s[1:][m] & 0x20) | A
    return s


ISLANDS = (4_000, 21_000, 47_000)               # CpG islands of the query (the rest of it has no CG)
NREGION = (100_000, 115_000)                    # 40 % N: windows inside are excluded (>= 30 %, F:238)


def _mix_scaffold():
    rng = np.random.Generator(np.random.PCG64(202610))
    s = _cg_free(synth.iid_bases(rng, 240_000, 0.45))
    for p in ISLANDS:
        isl = synth.iid_bases(rng, 40, 0.6)
        isl[::5], isl[1::5] = C, G
        s[p:p + 40] = isl
    for j in range(64):                          # single Ns at every offset mod 32 (60,000 and 97 = 1 mod 32)
        s[60_000 + 97 * j] = N
    for j in range(48):                          # N runs of 2..5
        p = 68_000 + 173 * j
        s[p:p + 2 + j % 4] = N
    for a, b in ((75_000, 79_000), (150_000, 150_700), (200_000, 200_033)):
        s[a:b] |= 0x20                           # soft-masked
    iupac = np.frombuffer(b"RYKMSWBDHVNnrykmswbdhv", np.uint8)
    for j in range(60):
        s[85_000 + 41 * j] = iupac[j % len(iupac)]
    seg = s[NREGION[0]:NREGION[1]]
    seg[rng.random(len(seg)) < 0.4] = N
    return s


@functools.lru_cache(maxsize=None)
def host_scaffolds():
    """The separate background: soft-masked stretches, an N run, and no CG anywhere, so a K-mer whose kmin-prefix holds a
    CG has a zero genome count there (NaN genome IVOM entry; the reference raises ZeroDivisionError, F:437)."""
    rng = np.random.Generator(np.random.PCG64(41))
    h = synth.iid_bases(rng, 150_000, 0.42)
    h[20_000:26_000] |= 0x20
    h[40_000:40_500] = N
    h[90_001:90_040:3] = ord("Y")
    return (("host", _cg_free(h)),)


@functools.lru_cache(maxsize=None)
def query_scaffolds():
    """The query: the feature scaffold and one scaffold per hand-over construction of part 3."""
    sc = [("mix", _mix_scaffold())]
    for (kmax, L), windows in sorted(HANDOVER_LAUNCHES.items()):
        for name, (codes, _) in windows.items():
            pad = np.random.Generator(np.random.PCG64(L + kmax))
            lead = 32 + (len(sc) * 13) % 32
            sc.append(("%s_k%d_w%d" % (name, kmax, L),
                       np.concatenate([synth.iid_bases(pad, lead, 0.5), bases_of(codes), synth.iid_bases(pad, 50, 0.5)])))
    return tuple(sc)


def construction_start(sc_name):
    """Start of a construction's window inside its scaffold."""
    idx = [n for n, _ in query_scaffolds()].index(sc_name)
    return 32 + (idx * 13) % 32


def test_query_and_host_have_their_features():
    q = dict(query_scaffolds())
    h = host_scaffolds()[0][1]
    up = h & 0xDF
    assert not np.any((up[:-1] == C) & (up[1:] == G)), "the host lacks every K-mer that holds a CG"
    assert np.count_nonzero(h >= ord("a")) > 5000
    mix = q["mix"]
    upm = mix & 0xDF
    cg = np.nonzero((upm[:-1] == C) & (upm[1:] == G))[0]
    assert len(cg) and all(any(p <= i < p + 40 for p in ISLANDS) for i in cg), "CG only inside the islands"
    assert {(60_000 + 97 * j) % 32 for j in range(64) if mix[60_000 + 97 * j] == N} == set(range(32))
    seg = mix[NREGION[0]:NREGION[1]]
    assert 0.36 < np.count_nonzero(seg == N) / len(seg) < 0.44
    assert np.count_nonzero(mix >= ord("a")) > 4000 and np.count_nonzero(np.isin(mix, list(b"RYKMSWBDHV"))) > 20


# ---- part 3: the extension kernel's hand-over constructions ---------------------------------------------------------

class _Builder:
    """A window built left to right; filler bases are chosen so that every 8-mer ending on them is new, so nothing but the
    planted structure repeats."""

    def __init__(self, seed, forbid=()):
        self.rng = np.random.Generator(np.random.PCG64(seed))
        self.c = []
        self.seen = set(forbid)

    def k8(self, c=None):
        tail = (self.c if c is None else c)[-8:]
        if len(tail) < 8 or min(tail) < 0:
            return None
        v = 0
        for b in tail:
            v = (v << 2) | b
        return v

    def fill(self, n):
        for _ in range(n):
            for b in self.rng.permutation(4):
                self.c.append(int(b))
                k = self.k8()
                if k is None or k not in self.seen:
                    break
                self.c.pop()
            else:
                self.c.append(int(self.rng.integers(4)))
            k = self.k8()
            if k is not None:
                self.seen.add(k)

    def put(self, codes):
        for b in codes:
            self.c.append(int(b))
            k = self.k8()
            if k is not None:
                self.seen.add(k)

    def codes(self):
        return np.array(self.c, np.int64)


def _nibble_wrap(L, run, seed):
    """`run` consecutive As between two Cs: AAAAAAAA run - 7 times (16 wraps a 4-bit counter)."""
    b = _Builder(seed, forbid=(0, 3 << 14, 3))     # AAAAAAAA, CAAAAAAA, AAAAAAAC: only the run makes them
    b.fill(L // 3)
    b.put([3] + [0] * run + [3])
    b.fill(L - len(b.c))
    return b.codes()


def _side_list(L, n_ns, seed):
    """Isolated Ns with 11 valid bases before each: each cuts two words (7 and 6 bases), the window end two more."""
    b = _Builder(seed)
    b.fill(12)
    for _ in range(n_ns):
        b.put([-1])
        b.fill(11)
    b.fill(L - len(b.c))
    return b.codes()


def _tandem(L, K, unit, m, seed):
    """A tandem repeat of a `unit`-base unit, m bases in all (<= 15 copies: no 8-mer wraps)."""
    b = _Builder(seed)
    b.fill(40)
    b.fill(unit)
    u = b.c[-unit:]
    b.put([u[i % unit] for i in range(m - unit)])
    b.fill(L - len(b.c))
    return b.codes()


TANDEM_UNIT = {9: 200, 10: 100, 11: 60, 12: 50}


def _hash_pair(L, K, seed):
    """(just over, just under) 2,560 registrations: bisect the tandem's length m on the restated count."""
    unit = TANDEM_UNIT[K]
    regs = lambda m: sum(len(t) for t in ext_registrations(_tandem(L, K, unit, m, seed), K))
    lo, hi = 2 * unit, 15 * unit
    assert regs(lo) <= 2560 < regs(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if regs(mid) > 2560:
            hi = mid
        else:
            lo = mid
    return _tandem(L, K, unit, hi, seed), _tandem(L, K, unit, lo, seed)


@functools.lru_cache(maxsize=None)
def probe_home():
    """The home slot of the most order-9 tags, and its 9-mers (1,421 of the 4,096 slots are home to 65 or more)."""
    codes = np.arange(1 << 18, dtype=np.int64)
    slots = ext_slot(ext_tag(9, codes)).astype(np.int64)
    per = np.bincount(slots, minlength=4096)
    assert int(np.count_nonzero(per >= 65)) == 1421
    h = int(np.argmax(per))
    return h, codes[slots == h]


def _nine(code):
    return [(code >> (2 * (8 - i))) & 3 for i in range(9)]


def _probe(L, K, n_same, seed):
    """n_same distinct 9-mers with one home slot h, each placed twice.  Around every copy, one filler-and-flank attempt
    after another until every 8-mer is new except the copy's own two (the 9-mer's 8-mer prefix and suffix), and the two
    other keys a copy registers (the 9-mer after it, and at kmax >= 10 the 10-mer it starts) have homes at least 65
    slots away from h: the keys on h then fill exactly h .. h + n_same - 1."""
    h, pool = probe_home()
    b = _Builder(seed)
    b.fill(8)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    far = lambda tag: min((int(ext_slot(tag)) - h) % 4096, (h - int(ext_slot(tag))) % 4096) > 64
    placed = []
    for m in pool:
        if len(placed) == n_same:
            break
        M = _nine(int(m))
        for _ in range(200):                      # both copies, each behind 4 filler bases and followed by one flank base
            seg = []
            for _copy in (0, 1):
                seg += [int(v) for v in rng.integers(0, 4, 4)] + M + [int(rng.integers(4))]
            trial, new = b.c[-7:], []
            for j, v in enumerate(seg):
                trial.append(v)
                k = b.k8(trial)
                if k is not None and j not in (14 + 11, 14 + 12):   # the second copy's 8-mer prefix and suffix repeat
                    new.append(k)
            fresh = len(set(new)) == len(new) and not (set(new) & b.seen)
            if fresh and all(far(ext_tag(9, (int(m) << 2 | nb) & ((1 << 18) - 1))) and
                             (K < 10 or far(ext_tag(10, int(m) << 2 | nb))) for nb in (seg[13], seg[27])):
                b.put(seg)
                placed.append(int(m))
                break
    assert len(placed) == n_same
    b.fill(L - len(b.c))
    return b.codes(), placed


def _launch(kmax, L):
    """Windows of one hand-over launch: {name: (codes, what it claims)}."""
    seed = 1000 * kmax + L
    out = {}
    if kmax != 10:
        out["wrap_over"] = (_nibble_wrap(L, 23, seed), "wrap")
        out["wrap_under"] = (_nibble_wrap(L, 22, seed), "wrap")
        out["side_over"] = (_side_list(L, 32, seed), "side")
        out["side_under"] = (_side_list(L, 31, seed), "side")
        out["probe_over"] = (_probe(L, kmax, 65, seed)[0], "probe")
        out["probe_under"] = (_probe(L, kmax, 64, seed)[0], "probe")
    if not (kmax == 9 and L == 2048):             # 2,048 positions cannot make 2,561 registrations at order 9 alone
        over, under = _hash_pair(L, kmax, seed)
        out["hash_over"] = (over, "hash")
        out["hash_under"] = (under, "hash")
    return out


class _Launches(dict):
    """(kmax, window length) -> windows; built on first use."""

    KEYS = [(9, 2048), (9, 5120), (9, 8186), (12, 2048), (12, 5120), (12, 8186), (10, 2048)]

    def items(self):
        return [(k, self[k]) for k in self.KEYS]

    def __missing__(self, key):
        self[key] = v = _launch(*key)
        return v


HANDOVER_LAUNCHES = _Launches()


def handover_facts(codes, K):
    regs = ext_registrations(codes, K)
    most, longest = hash_probe_bounds(regs)
    return dict(max8=int(kmer8_counts(codes).max()), side=side_words(codes), regs=sum(len(r) for r in regs),
                most_on_one_home=most, longest_run_from_a_home=longest)


@pytest.mark.parametrize("kmax,L", _Launches.KEYS)
def test_handover_constructions_have_their_property(kmax, L):
    """Each window crosses exactly the limit it is named for (and none that the kernel checks before it), or stays one
    step short of it and crosses nothing; the numbers come from numpy restatements of the kernel's rules."""
    if (kmax, L) == (9, 2048):                     # order 9 alone registers each position once at most: 2,048 < 2,561
        assert "hash_over" not in HANDOVER_LAUNCHES[(kmax, L)]
    for name, (codes, what) in HANDOVER_LAUNCHES[(kmax, L)].items():
        assert len(codes) == L
        f = handover_facts(codes, kmax)
        over = name.endswith("_over")
        fits = dict(wrap=f["max8"] <= 15, side=f["side"] <= 64, hash=f["regs"] <= 2560,
                    probe=f["longest_run_from_a_home"] <= 64)
        if what == "wrap":
            assert f["max8"] == (16 if over else 15), (name, f)
            assert kmer8_counts(codes)[0] == f["max8"]           # AAAAAAAA
        elif what == "side":
            assert f["side"] == (66 if over else 64), (name, f)
        elif what == "hash":
            assert (f["regs"] > 2560) == over, (name, f)
            assert max(kmer8_counts(codes)) <= 15
        else:
            assert f["most_on_one_home"] == (65 if over else 64), (name, f)
            c9, ok9 = kmer_codes(codes, 9)
            h, pool = probe_home()
            on_h = np.isin(c9[ok9], pool)
            assert len(np.unique(c9[ok9][on_h])) == (65 if over else 64)
            assert np.all(np.bincount(c9[ok9][on_h])[np.unique(c9[ok9][on_h])] == 2)
        checked_before = {"wrap": [], "side": ["wrap"], "hash": ["wrap", "side"], "probe": ["wrap", "side", "hash"]}[what]
        for other in checked_before:
            assert fits[other], (name, other, f)
        if not over:
            assert all(fits.values()), (name, f)


# ---- part 1: the case matrix ----------------------------------------------------------------------------------------

Case = namedtuple("Case", "opt kmin kmax lengths host rip n")


def band(lo, hi, K):
    """The band's longest length and the three below it (every residue mod 4), its shortest, and 1, K-1, K, K+1."""
    ls = [hi, hi - 1, hi - 2, hi - 3, lo, 1, K - 1, K, K + 1]
    return tuple(sorted({x for x in ls if 1 <= x <= hi}, reverse=True))


def case(opt, kmin, kmax, lo, hi, host=False, rip=True, n=40, lengths=None):
    return Case(opt, kmin, kmax, lengths or band(lo, hi, kmax), host, rip, n)


SMEM = 8186
B2, B5 = 2042, 5114                  # bucketed / direct kernel: rounds of 4 positions, 6 bases of look-ahead
P8, P20 = 2048, 5120                 # nibble / extension kernel: positions per thread
LONG = (100_000, 65_536, 65_535, 8_187)

CASES = [
    # small-K kernel: any window up to 65,535 bases
    case(None, 1, 1, 1, 65535), case(None, 2, 2, 1, 65535, host=True, rip=False), case(None, 1, 3, 1, 65535),
    case(None, 3, 4, 1, 65535, host=True, rip=False), case(None, 1, 5, 1, 65535), case(None, 2, 6, 1, 65535, host=True),
    # dense-table kernel: forced, and windows past the shared-memory buffer at kmax 7 / 8
    case("force_dense_kernel", 1, 3, 1, 65535), case("force_dense_kernel", 2, 6, 1, 65535, host=True, rip=False),
    case(None, 1, 7, SMEM + 1, 65535), case(None, 2, 7, SMEM + 1, 65535, host=True, rip=False),
    case(None, 1, 8, SMEM + 1, 65535), case(None, 3, 8, SMEM + 1, 65535, host=True),
    # direct kernel: kmax 7 up to 1,500 bases by default, forced otherwise
    case(None, 1, 7, 1, 1500), case(None, 2, 7, 1, 1500, host=True, rip=False),
    case("force_direct_kernel", 1, 7, B2 + 1, B5), case("force_direct_kernel", 3, 7, B2 + 1, B5, host=True),
    case("force_direct_kernel", 1, 7, B5 + 1, SMEM), case("force_direct_kernel", 2, 7, B5 + 1, SMEM, host=True, rip=False),
    case("force_direct_kernel", 1, 8, 1, B2), case("force_direct_kernel", 2, 8, 1, B2, host=True),
    case("force_direct_kernel", 1, 8, B2 + 1, B5), case("force_direct_kernel", 3, 8, B2 + 1, B5, host=True, rip=False),
    case("force_direct_kernel", 1, 8, B5 + 1, SMEM), case("force_direct_kernel", 2, 8, B5 + 1, SMEM, host=True),
    # nibble kernel: kmax 8, and kmax 7 above 1,500 bases (forced below)
    case(None, 1, 7, 1501, P8), case("force_nibble_kernel", 2, 7, 1, P8, host=True, rip=False),
    case(None, 1, 7, P8 + 1, P20), case(None, 3, 7, P8 + 1, P20, host=True),
    case(None, 1, 7, P20 + 1, SMEM), case(None, 2, 7, P20 + 1, SMEM, host=True, rip=False),
    case(None, 1, 8, 1, P8), case(None, 2, 8, 1, P8, host=True),
    case(None, 1, 8, P8 + 1, P20), case(None, 2, 8, P8 + 1, P20, host=True, rip=False),
    case(None, 1, 8, P20 + 1, SMEM), case(None, 3, 8, P20 + 1, SMEM, host=True),
    # bucketed kernel (forced): kmax 4..8, rounds of 2 / 5 / 8
    case("force_bucket_kernel", 1, 4, B2 + 1, B5), case("force_bucket_kernel", 2, 5, B5 + 1, SMEM, host=True, rip=False),
    case("force_bucket_kernel", 1, 6, 1, B2), case("force_bucket_kernel", 2, 6, 1, B2, host=True),
    case("force_bucket_kernel", 1, 6, B2 + 1, B5), case("force_bucket_kernel", 3, 6, B2 + 1, B5, host=True, rip=False),
    case("force_bucket_kernel", 1, 6, B5 + 1, SMEM), case("force_bucket_kernel", 2, 6, B5 + 1, SMEM, host=True),
    case("force_bucket_kernel", 1, 7, 1, B2), case("force_bucket_kernel", 2, 7, 1, B2, host=True, rip=False),
    case("force_bucket_kernel", 1, 7, B2 + 1, B5), case("force_bucket_kernel", 3, 7, B2 + 1, B5, host=True),
    case("force_bucket_kernel", 1, 7, B5 + 1, SMEM), case("force_bucket_kernel", 2, 7, B5 + 1, SMEM, host=True, rip=False),
    case("force_bucket_kernel", 1, 8, 1, B2), case("force_bucket_kernel", 2, 8, 1, B2, host=True),
    case("force_bucket_kernel", 1, 8, B2 + 1, B5), case("force_bucket_kernel", 2, 8, B2 + 1, B5, host=True, rip=False),
    case("force_bucket_kernel", 1, 8, B5 + 1, SMEM), case("force_bucket_kernel", 3, 8, B5 + 1, SMEM, host=True),
    # extension kernel, kmax 9..12 (kmin 10 and kmin = kmax = 12 on the query's own background: a 150 kbp host lacks
    # nearly every 10-mer)
    case(None, 1, 9, 1, P8), case(None, 1, 10, P8 + 1, P20), case(None, 1, 11, P20 + 1, SMEM),
    case(None, 10, 12, 1, P8, rip=False), case(None, 12, 12, P8 + 1, P20),
    case(None, 2, 12, P20 + 1, SMEM, host=True, rip=False),
    # general kernel: windows over 65,535 bases, kmax 9..12 past the shared-memory buffer, forced with more windows than SMs
    case(None, 1, 8, 0, 0, lengths=LONG + (99_999, 99_998, 99_997, 1, 7, 8, 9)),
    case(None, 1, 9, 0, 0, lengths=LONG + (99_999, 99_998, 99_997, 1, 8, 9, 10)),
    case(None, 2, 12, 0, 0, host=True, rip=False, lengths=LONG + (99_999, 99_998, 99_997, 1, 11, 12, 13)),
    case("force_general_kernel", 2, 5, 1, 65535, host=True),
    case("force_general_kernel", 1, 12, 0, 0, n=400, lengths=(2000, 1999, 1998, 1997, 1900, 1, 11, 12, 13)),
]

# variants the planner reaches that test_score_plan's table does not list
EXTRA_NAMES = {"score_windows_small_kernel<1, 0>", "score_windows_small_kernel<2, 0>", "score_windows_small_kernel<4, 0>",
               "score_windows_small_kernel<5, 0>", "score_windows_bucket_kernel<4, 5, 0, 1>",
               "score_windows_bucket_kernel<5, 8, 0, 0>"}


def case_id(c):
    return "%s-k%d_%d-w%d%s%s" % ((c.opt or "default").replace("force_", "").replace("_kernel", ""), c.kmin, c.kmax,
                                  max(c.lengths), "-host" if c.host else "", "" if c.rip else "-norip")


def family(name):
    return name.split("<")[0]


def test_case_matrix_reaches_every_window_kernel():
    """kernel_name makes no CUDA call: the table's reach is checked on any machine."""
    reached, by = set(), {}
    for c in CASES:
        with forced(c.opt):
            name = kernel_name(c.kmin, c.kmax, max(c.lengths))
        reached.add(name)
        by.setdefault(name, []).append(c)
    planned = {name for rules in EXPECTED.values() for _, name in rules}
    assert reached == planned | EXTRA_NAMES, (sorted(planned - reached), sorted(reached - planned - EXTRA_NAMES))
    ext = [c for n, cs in by.items() if family(n) == "score_windows_nibble_ext_kernel" for c in cs]
    assert {10, 11} <= {c.kmax for c in ext}
    assert {(10, 12), (12, 12)} <= {(c.kmin, c.kmax) for c in ext}
    for fam in {family(n) for n in reached}:
        cs = [c for n, v in by.items() if family(n) == fam for c in v]
        assert any(c.kmin > 1 for c in cs) and any(not c.rip for c in cs) and any(c.host for c in cs), fam
        assert any(c.kmin == 1 and c.rip and not c.host for c in cs), fam
    assert len({case_id(c) for c in CASES}) == len(CASES)


# ---- part 2: every case against the oracle --------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def packed():
    from frisk_b200 import engine
    return engine.PackedGenome.from_scaffolds(list(query_scaffolds())), engine.PackedGenome.from_scaffolds(list(host_scaffolds()))


@functools.lru_cache(maxsize=None)
def concat(host):
    from oracle import c_oracle
    seq, off = c_oracle.concat(list(host_scaffolds() if host else query_scaffolds()))
    non = np.concatenate([[0], np.cumsum(~UPPER_ACGT[seq], dtype=np.int64)])       # countN (F:106-118) prefix sums
    return seq, off, non


@functools.lru_cache(maxsize=4)
def oracle_background(kmin, kmax, host):
    from oracle import c_oracle
    seq, off, _ = concat(host)
    return c_oracle.background(seq, off, kmin, kmax, host, threads=8)   # mask_host together with the separate host


def case_windows(c, seed):
    """(scaffold, start) of every window with its length: anchors at a scaffold start and end, a CpG island and the N-rich
    region, then c.n windows whose lengths cycle through c.lengths and whose starts cycle through every offset mod 32."""
    sc = query_scaffolds()
    lens = np.array([len(s) for _, s in sc])
    rng = np.random.Generator(np.random.PCG64(seed))
    top = max(c.lengths)
    out = [(0, 0, top), (0, lens[0] - top, top)]
    for p in (ISLANDS[0] - 17, NREGION[0] + 5):
        for L in (top, c.lengths[len(c.lengths) // 2]):
            if p + L <= lens[0]:
                out.append((0, p, L))
    for i in range(c.n):
        L = c.lengths[i % len(c.lengths)]
        r = i % 32
        fit = np.nonzero(lens >= L + 32)[0]
        s = int(rng.choice(fit, p=lens[fit] / lens[fit].sum()))
        out.append((s, int(rng.integers(0, (lens[s] - L - r) // 32 + 1)) * 32 + r, L))
    return out


def window_list(eng, g, wins):
    s = np.array([w[0] for w in wins], np.uint32)
    rel = np.array([w[1] for w in wins], np.int64)
    ln = np.array([w[2] for w in wins], np.uint32)
    off = (g.scaf_off[s] + rel.astype(np.uint64)).astype(np.uint64)
    return eng.WindowList(off, ln, s, rel + 1, rel + ln.astype(np.int64))


def oracle_rows(wins, kmin, kmax, host, rip):
    from oracle import c_oracle
    seq, off, non = concat(False)
    coff = np.array([int(off[s]) + r for s, r, _ in wins], np.uint64)
    ln = np.array([w[2] for w in wins], np.uint32)
    tabs, meta = oracle_background(kmin, kmax, host)
    rows, status = c_oracle.score(seq, coff, ln, tabs, meta, kmin, kmax, rip, threads=8)
    excluded = (non[coff.astype(np.int64) + ln] - non[coff.astype(np.int64)]) >= 0.3 * ln     # F:238
    return rows, status, excluded, coff, ln


def check_launch(dev, wins, opt, kmin, kmax, host, rip, what, dump=True):
    """One launch of these windows against the oracle; returns (result, oracle status of its rows, kept windows)."""
    eng, dq, dh = dev
    g = packed()[0]
    wl = window_list(eng, g, wins)
    kw = dict(kmin=kmin, kmax=kmax, mask_host=host, rip=rip, wins=wl)
    with forced(opt):
        res = eng.run(dq, dh if host else None, **kw)
        again = eng.run(dq, dh if host else None, **kw)
    rows, status, excluded, coff, ln = oracle_rows(wins, kmin, kmax, host, rip)
    tabs, meta = oracle_background(kmin, kmax, host)
    assert np.array_equal(res.tables, tabs), what + ": background tables"
    assert list(res.meta) == [int(x) for x in meta], what
    keep = np.nonzero(~excluded)[0]
    assert np.array_equal(res.win_index, keep), what + ": excluded windows"
    assert not np.any(res.status & 0x80000000), what + ": internal hand-over marker survived"
    assert np.array_equal(res.status & 7, status[keep] & 7), what + ": status"
    ref = rows[keep].copy()
    got = res.rows.copy()
    bad = status[keep] != 0
    ref[bad, 0] = 0.0
    got[bad, 0] = 0.0
    assert_rows_close(got, ref, rtol_kld=1e-6, rtol_other=1e-15, what=what)
    ok = ~bad
    assert max_rel_err(res.rows[ok, 0], rows[keep][ok, 0]) < 1e-10, what
    assert np.array_equal(again.rows.view(np.uint64), res.rows.view(np.uint64)), what + ": second run"
    assert np.array_equal(again.status, res.status), what
    if dump and kmax <= 8 and max(w[2] for w in wins) <= 65535:
        from oracle import c_oracle
        seq = concat(False)[0]
        with forced(opt):
            d = eng.run(dq, dh if host else None, dump=True, **kw)
        assert np.array_equal(d.win_index, keep)
        for j, i in enumerate(keep):
            a = int(coff[i])
            _, _, wt, _ = c_oracle.window_tables(seq[a:a + int(ln[i])], tabs, meta, kmin, kmax)
            assert np.array_equal(d.win_tables[j].astype(np.uint64), wt), (what, int(i))
    return res, status[keep], keep


@pytest.fixture(scope="module")
def devices(eng):
    """(engine, query planes, host planes) on the device, shared by the module's launches."""
    q, h = packed()
    return eng, eng.DeviceGenome(q), eng.DeviceGenome(h)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_case_against_c_oracle(devices, c):
    with forced(c.opt):
        name = kernel_name(c.kmin, c.kmax, max(c.lengths))
    wins = case_windows(c, zlib.crc32(case_id(c).encode()))
    offsets = {(int(packed()[0].scaf_off[s]) + r) % 32 for s, r, _ in wins}
    assert offsets == set(range(32))
    _, status, _ = check_launch(devices, wins, c.opt, c.kmin, c.kmax, c.host, c.rip, case_id(c) + " " + name)
    if c.host:
        assert np.any(status & _lib.ROW_KLD_ZERODIV), "the host lacks K-mers of these windows"


# ---- part 3 on the GPU ----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kmax,L", _Launches.KEYS)
def test_extension_kernel_hand_overs(devices, kmax, L):
    eng, dq, _ = devices
    names = [n for n, _ in query_scaffolds()]
    windows = HANDOVER_LAUNCHES[(kmax, L)]
    wins = []
    for name in windows:
        sc = "%s_k%d_w%d" % (name, kmax, L)
        wins.append((names.index(sc), construction_start(sc), L))
    assert kernel_name(1, kmax, L) == "score_windows_nibble_ext_kernel<%d, 1>" % {2048: 8, 5120: 20, 8186: 32}[L]
    what = "hand-over k%d w%d" % (kmax, L)
    res, status, keep = check_launch(devices, wins, None, 1, kmax, False, True, what)
    assert len(keep) == len(wins)
    with forced("force_general_kernel"):
        gen = eng.run(dq, kmin=1, kmax=kmax, wins=window_list(eng, packed()[0], wins))
    for i, name in enumerate(windows):
        if name.endswith("_over"):
            assert np.array_equal(res.rows[i].view(np.uint64), gen.rows[i].view(np.uint64)), (what, name)
            assert res.status[i] == gen.status[i], (what, name)


# ---- part 4: background counter wraps -------------------------------------------------------------------------------

def wrap_scaffolds():
    """polyA and a period-(K+1) A^K T repeat per K (AAA..A and AA..AT share one 32-bit word of counters and wrap
    together), each also as a copy with an N every 31 bases: every 32-base word then holds an N, so every position goes
    through the per-position path."""
    mb = 1_000_000
    base = [("polyA", np.full(8 * mb, A, np.uint8))]
    for K in range(1, 9):
        unit = np.frombuffer(b"A" * K + b"T", np.uint8)
        n = (12 if K >= 7 else 8) * mb
        base.append(("repeat%d" % K, np.tile(unit, 8 * mb // (K + 1) + 1)[:8 * mb]))
        base.append(("repeat%d_N" % K, np.tile(unit, n // (K + 1) + 1)[:n].copy()))
    out = []
    for name, s in base:
        if name.endswith("_N"):
            s[30::31] = N
            out.append((name, s))
        else:
            out.append((name, s))
            if name == "polyA":
                d = s.copy()
                d[30::31] = N
                out.append(("polyA_N", d))
    return out


def a_run_count(s, K):
    """Forward count of A^K (code 0) in a scaffold: the K-words inside its runs of A."""
    isa = np.concatenate([[False], s == A, [False]])
    edges = np.nonzero(np.diff(isa.astype(np.int8)))[0]
    runs = edges[1::2] - edges[0::2]
    return int(np.maximum(runs - K + 1, 0).sum())


def ex_max(lens, invalid, K):
    """K-words that hold a character other than ATGC (F:341-346), from each scaffold's length and invalid positions."""
    total = 0
    for n, q in zip(lens, invalid):
        starts = n - K + 1
        if starts <= 0:
            continue
        bad = np.zeros(starts, bool)
        for d in range(K):
            p = q - d
            bad[p[(p >= 0) & (p < starts)]] = True
        total += int(np.count_nonzero(bad))
    return total


@pytest.mark.gpu
def test_background_16bit_wraps_at_every_word_size(eng):
    import torch
    from oracle import c_oracle
    sc = wrap_scaffolds()
    assert all(np.count_nonzero(s[i:i + 32] == N) for name, s in sc if name.endswith("_N") for i in range(0, 4096, 32))
    g = eng.PackedGenome.from_scaffolds(sc)
    dg = eng.DeviceGenome(g)
    seq, off = c_oracle.concat(sc)
    tabs, meta = c_oracle.background(seq, off, 1, 8, False, threads=16)
    # bg_count_kernel's launch: a grid of min(SMs, words / 2048) CTAs over the words of the padded genome (the last one is
    # look-ahead only), ceil(words / grid) consecutive words each
    words = g.padded_len // 32 - 1
    grid = max(1, min(torch.cuda.get_device_properties(0).multi_processor_count, (words + 2047) // 2048))
    per = -(-words // grid)
    names = [n for n, _ in sc]
    lens = [len(s) for _, s in sc]
    invalid = [np.nonzero(~UPPER_ACGT[s])[0] for _, s in sc]
    for K in range(1, 9):
        for name in ("polyA", "polyA_N", "repeat%d" % K, "repeat%d_N" % K):
            s = names.index(name)
            first, last = int(g.scaf_off[s]) // 32, (int(g.scaf_off[s]) + int(g.scaf_len[s]) - 1) // 32
            ctas = last // per - first // per + 1
            assert a_run_count(sc[s][1], K) > 65535 * ctas, (K, name, "no CTA has to wrap")
        d_tables, d_valid = eng.finalize(eng.background(dg, K), K)
        got = d_tables.cpu().numpy().view(np.uint64)
        assert np.array_equal(got, tabs[:_lib.table_size(1, K)]), K
        assert g.ex_max(K, int(d_valid.item())) == ex_max(lens, invalid, K), K
    assert g.ex_max(8, int(d_valid.item())) == int(meta[1])
