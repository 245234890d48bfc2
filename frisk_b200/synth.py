"""Seeded synthetic genomes for parity tests and benchmarks (SURVEY.md section 8d).

There is no network and the reference ships no example data, so every input is
generated here from ``numpy.random.Generator(PCG64(seed))`` using only ``random`` and
``integers`` (stream-stable across numpy versions).  A scaffold is ``(name, uint8
ASCII array)``.  Configs mirror BASELINE.json ``configs`` C1..C5; ``scale`` shrinks
the total length for tests while keeping the structure.
"""
from __future__ import annotations

import hashlib
from typing import List, Tuple

import numpy as np

Scaffold = Tuple[str, np.ndarray]

_AT = np.frombuffer(b"AT", dtype=np.uint8)
_GC = np.frombuffer(b"GC", dtype=np.uint8)


def iid_bases(rng: np.random.Generator, n: int, gc: float) -> np.ndarray:
    """n iid bases with P(G or C) = gc, A/T and G/C each split evenly."""
    is_gc = rng.random(n) < gc
    second = rng.integers(0, 2, n, dtype=np.uint8)
    return np.where(is_gc, _GC[second], _AT[second]).astype(np.uint8)


def markov_bases(rng: np.random.Generator, n: int, order: int = 3, alpha: float = 0.5) -> np.ndarray:
    """Order-`order` Markov chain; each context row ~ Dirichlet(alpha) (via gammas)."""
    nctx = 4 ** order
    g = -np.log(rng.random((nctx, 4))) ** (1.0 / alpha)  # crude heavy-tailed positive weights
    cum = np.cumsum(g / g.sum(axis=1, keepdims=True), axis=1)
    u = rng.random(n)
    out = np.empty(n, dtype=np.uint8)
    ctx = int(rng.integers(0, nctx))
    letters = b"ATGC"
    mask = nctx - 1
    for j in range(n):
        b = int(np.searchsorted(cum[ctx], u[j]))
        if b > 3:
            b = 3
        out[j] = letters[b]
        ctx = ((ctx << 2) | b) & mask
    return out


def plant_runs(rng, seq: np.ndarray, n_runs: int, lo: int, hi: int, char: bytes = b"N") -> None:
    if len(seq) <= hi + 2:
        return
    for _ in range(n_runs):
        ln = int(rng.integers(lo, hi + 1))
        st = int(rng.integers(0, len(seq) - ln))
        seq[st:st + ln] = char[0]


def config_c1(scale: float = 1.0, seed: int = 1001) -> List[Scaffold]:
    """C1: one 5 Mbp scaffold, iid uniform, 20 GC-skewed islands + 5 Markov islands, no N."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = max(int(5_000_000 * scale), 20_000)
    seq = iid_bases(rng, n, 0.5)
    lo, hi = max(int(20_000 * min(scale * 4, 1.0)), 2_000), max(int(50_000 * min(scale * 4, 1.0)), 5_000)
    for t in range(20):
        ln = int(rng.integers(lo, hi + 1))
        st = int(rng.integers(0, max(n - ln, 1)))
        ln = min(ln, n - st)
        seq[st:st + ln] = iid_bases(rng, ln, 0.25 if t % 2 == 0 else 0.70)
    for t in range(5):
        ln = int(rng.integers(lo, hi + 1))
        st = int(rng.integers(0, max(n - ln, 1)))
        ln = min(ln, n - st)
        seq[st:st + ln] = markov_bases(rng, ln)
    return [("scaffold_1", seq)]


def _lognormal_lengths(rng, count: int, total: int, sigma: float, min_len: int) -> np.ndarray:
    z = np.sqrt(-2.0 * np.log(rng.random(count))) * np.cos(2 * np.pi * rng.random(count))
    raw = np.exp(sigma * z)
    lens = np.maximum((raw / raw.sum() * total).astype(np.int64), min_len)
    return lens


def config_c2(scale: float = 1.0, seed: int = 2002) -> List[Scaffold]:
    """C2: 40 Mbp fungal-style assembly, ~500 scaffolds, AT-rich accessory blocks, N runs."""
    rng = np.random.Generator(np.random.PCG64(seed))
    count = max(int(500 * min(1.0, scale * 10)), 4)
    total = int(40_000_000 * scale)
    lens = _lognormal_lengths(rng, count, total, 1.0, 10_000)
    out = []
    n_runs_total = max(int(200 * scale), 2)
    for s, ln in enumerate(lens):
        ln = int(ln)
        seq = iid_bases(rng, ln, 0.52)
        # ~10 % of bases in AT-rich accessory blocks of 50-200 kbp (clipped to the scaffold)
        budget = int(0.10 * ln)
        while budget > 5_000:
            bl = min(int(rng.integers(50_000, 200_001)), budget, ln)
            st = int(rng.integers(0, ln - bl + 1))
            seq[st:st + bl] = iid_bases(rng, bl, 0.30)
            budget -= bl
        out.append(("scaffold_%d" % (s + 1), seq))
    for _ in range(n_runs_total):
        s = int(rng.integers(0, count))
        plant_runs(rng, out[s][1], 1, 100, 100)
    return out


def config_c3(scale: float = 1.0, seed: int = 3003) -> List[Scaffold]:
    """C3: 120 Mbp plant-style, 12 chromosomes, GC 0.36, 30 % TE-like repeats."""
    rng = np.random.Generator(np.random.PCG64(seed))
    chrom = max(int(10_000_000 * scale), 30_000)
    fams = [iid_bases(rng, int(rng.integers(1_000, 8_001)), 0.42) for _ in range(50)]
    out = []
    for c in range(12):
        seq = iid_bases(rng, chrom, 0.36)
        budget = int(0.30 * chrom)
        while budget > 0:
            fam = fams[int(rng.integers(0, 50))]
            copy = fam.copy()
            mut = rng.random(len(copy)) < 0.10
            copy[mut] = iid_bases(rng, int(mut.sum()), 0.36)
            st = int(rng.integers(0, chrom - len(copy)))
            seq[st:st + len(copy)] = copy
            budget -= len(copy)
        out.append(("chr%d" % (c + 1), seq))
    return out


def config_c4(scale: float = 1.0, seed: int = 4004) -> List[Scaffold]:
    """C4: 3 Gbp human-scale, 24 scaffolds 50-250 Mbp, 300 kbp isochores, one long N run each."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lens = np.linspace(250e6, 50e6, 24)
    lens = (lens / lens.sum() * 3e9 * scale).astype(np.int64)
    out = []
    for c, ln in enumerate(lens):
        ln = int(max(ln, 30_000))
        iso = max(int(300_000 * min(1.0, scale * 100)), 3_000)
        parts = []
        left = ln
        while left > 0:
            bl = min(iso, left)
            z = np.sqrt(-2.0 * np.log(rng.random())) * np.cos(2 * np.pi * rng.random())
            gc = float(np.clip(0.41 + 0.05 * z, 0.25, 0.65))
            parts.append(iid_bases(rng, bl, gc))
            left -= bl
        seq = np.concatenate(parts)
        nl = max(int(3_000_000 * scale), 50)
        st = int(rng.integers(0, ln - nl))
        seq[st:st + nl] = ord("N")
        out.append(("chr%d" % (c + 1), seq))
    return out


def config_c5(scale: float = 1.0, seed: int = 5005) -> List[Scaffold]:
    """C5: 14 Gbp wheat-scale fragmented assembly: 1 M short scaffolds, many N gaps."""
    rng = np.random.Generator(np.random.PCG64(seed))
    count = max(int(1_000_000 * scale), 8)
    total = int(14e9 * scale)
    lens = _lognormal_lengths(rng, count, total, 0.9, 500)
    out = []
    for s, ln in enumerate(lens):
        ln = int(ln)
        seq = iid_bases(rng, ln, 0.46)
        if rng.random() < 0.30:
            plant_runs(rng, seq, int(rng.integers(1, 4)), 10, min(2_000, max(ln // 4, 10)))
        out.append(("scf%07d" % (s + 1), seq))
    return out


def config_edge(seed: int = 7) -> List[Scaffold]:
    """Micro-genome exercising every edge in SURVEY.md section 4: lowercase soft-masking,
    IUPAC codes, '-' gaps, N-rich windows (30 % filter), size % step == 0 (duplicate tail
    window), scaffolds at / below / just above the 6,250 minimum, tiny scaffolds."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    a = iid_bases(rng, 20_000, 0.45)                       # size % step == 0
    a[3_000:3_400] = np.char.lower(a[3_000:3_400].view("S1")).view(np.uint8)  # soft-masked block
    a[7_000:7_010] = np.frombuffer(b"RYKMSWBDHV", dtype=np.uint8)             # IUPAC
    a[9_100:9_103] = ord("-")
    out.append(("edgeA", a))
    b = iid_bases(rng, 17_321, 0.60)                       # ragged tail
    b[5_000:6_600] = ord("N")                              # 1,600 N: >30 % of one window only
    b[12_000:12_900] = ord("n")                            # lowercase n is also invalid
    out.append(("edgeB", b))
    out.append(("edge_at_min", iid_bases(rng, 6_250, 0.5)))    # == minimum -> skipped / rescued
    out.append(("edge_above_min", iid_bases(rng, 6_251, 0.5)))  # smallest windowed scaffold
    out.append(("edge_small", iid_bases(rng, 1_234, 0.35)))
    c = iid_bases(rng, 900, 0.5)
    c[100:500] = ord("N")                                  # >30 % N small scaffold
    out.append(("edge_small_N", c))
    out.append(("edge_tiny", iid_bases(rng, 5, 0.5)))       # shorter than kmax
    d = iid_bases(rng, 9_000, 0.3)
    d[::2] = np.char.lower(d[::2].view("S1")).view(np.uint8)    # 50 % lowercase: windows excluded
    out.append(("edge_half_lower", d))
    e = iid_bases(rng, 8_000, 0.5)
    e[2_000:2_600] = ord("A")                              # homopolymer: heavy bin contention
    e[4_000:4_800] = np.tile(np.frombuffer(b"AT", dtype=np.uint8), 400)  # no 'AC'/'GT' variety
    out.append(("edge_lowcomplex", e))
    return out


def config_edge_short(seed: int = 17) -> List[Scaffold]:
    """Scaffolds around one window length for runs with 0.75 w < step < w (meant for -w 1000 -i 800: minimum
    size 950): a scaffold with 950 < size < w is windowed, its one window overshoots at j = 0, and the
    reference's ``seq[size - w:size]`` (F:231) has a NEGATIVE start -- the last ``w - size`` bases, reported with
    coordinates (size - w, size) (F:243)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for n, gc in [(975, 0.5), (999, 0.4), (951, 0.6), (950, 0.5), (1000, 0.5), (1001, 0.45), (1600, 0.55), (1799, 0.5),
                  (1800, 0.5), (2400, 0.35), (4000, 0.5), (960, 0.3)]:
        out.append(("short_%d" % n, iid_bases(rng, n, gc)))
    a = iid_bases(rng, 970, 0.5)
    a[945:960] = ord("N")                                  # 15 of the last 30 bases unresolved: the short window is excluded
    out.append(("short_970_N", a))
    b = iid_bases(rng, 990, 0.5)
    b[985:988] = ord("n")                                  # 3 of the last 10: exactly 30 % -> excluded (>=, F:238)
    out.append(("short_990_n", b))
    c = iid_bases(rng, 980, 0.5)
    c[962:967] = np.char.lower(c[962:967].view("S1")).view(np.uint8)   # 5 of the last 20 lower case: 25 %, kept
    out.append(("short_980_low", c))
    return out


CONFIGS = {"C1": config_c1, "C2": config_c2, "C3": config_c3, "C4": config_c4, "C5": config_c5}


def make(config: str, scale: float = 1.0, seed: int | None = None) -> List[Scaffold]:
    if config == "edge":
        return config_edge() if seed is None else config_edge(seed)
    if config == "edge_short":
        return config_edge_short() if seed is None else config_edge_short(seed)
    fn = CONFIGS[config]
    return fn(scale) if seed is None else fn(scale, seed)


def total_bases(scaffolds: List[Scaffold]) -> int:
    return int(sum(len(s) for _, s in scaffolds))


def digest(scaffolds: List[Scaffold]) -> str:
    h = hashlib.sha256()
    for name, seq in scaffolds:
        h.update(name.encode())
        h.update(np.ascontiguousarray(seq).tobytes())
    return h.hexdigest()


def fasta_bytes(scaffolds: List[Scaffold], width: int = 60) -> bytes:
    """The scaffolds as FASTA text (the reference's input format), `width` bases per line."""
    parts = []
    for name, seq in scaffolds:
        parts.append(b">" + name.encode() + (" len=%d synthetic\n" % len(seq)).encode())
        n = len(seq)
        full = (n // width) * width
        if full:
            body = np.empty((n // width, width + 1), dtype=np.uint8)
            body[:, :width] = seq[:full].reshape(-1, width)
            body[:, width] = 10
            parts.append(body.tobytes())
        if n > full:
            parts.append(seq[full:].tobytes() + b"\n")
    return b"".join(parts)


_TWOBIT_CODE = np.zeros(256, np.uint8)                   # T=0, C=1, A=2, G=3; anything else (an N) is stored as T
for _c, _v in zip(b"TCAGtcag", (0, 1, 2, 3, 0, 1, 2, 3)):
    _TWOBIT_CODE[_c] = _v


def _runs(flag: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """(starts, sizes) of the runs of True in a boolean array."""
    d = np.diff(np.concatenate([[0], flag.astype(np.int8), [0]]))
    starts = np.nonzero(d == 1)[0]
    return starts.astype(np.uint32), (np.nonzero(d == -1)[0] - starts).astype(np.uint32)


def twobit_bytes(scaffolds: List[Scaffold], big_endian: bool = False, version: int = 0) -> bytes:
    """The scaffolds as a UCSC .2bit file (faToTwoBit's format): N blocks = the runs of characters that are not one of
    ACGTacgt, mask blocks = the runs of lower-case characters, 4 bases per byte with the first in the top two bits.
    ``version`` 1 writes 64-bit index offsets; ``big_endian`` writes every integer byte-swapped."""
    e = ">" if big_endian else "<"
    u32 = np.dtype(e + "u4")
    idx_entry = 4 if version == 0 else 8
    index_len = sum(1 + len(name.encode()) + idx_entry for name, _ in scaffolds)
    records = []
    for _, seq in scaffolds:
        s = np.ascontiguousarray(seq, dtype=np.uint8)
        n = len(s)
        up = s & 0xDF
        n_starts, n_sizes = _runs(~np.isin(up, np.frombuffer(b"ACGT", np.uint8)))
        m_starts, m_sizes = _runs((s >= ord("a")) & (s <= ord("z")))
        codes = np.zeros((n + 3) // 4 * 4, np.uint8)
        codes[:n] = _TWOBIT_CODE[s]
        q = codes.reshape(-1, 4)
        packed = (q[:, 0] << 6) | (q[:, 1] << 4) | (q[:, 2] << 2) | q[:, 3]
        head = np.array([n, len(n_starts)], u32).tobytes() + n_starts.astype(u32).tobytes() + n_sizes.astype(u32).tobytes()
        head += np.array([len(m_starts)], u32).tobytes() + m_starts.astype(u32).tobytes() + m_sizes.astype(u32).tobytes()
        records.append(head + np.array([0], u32).tobytes() + packed.astype(np.uint8).tobytes())
    off = 16 + index_len
    index = []
    for (name, _), rec in zip(scaffolds, records):
        nb = name.encode()
        index.append(bytes([len(nb)]) + nb + np.array([off], np.dtype(e + ("u4" if version == 0 else "u8"))).tobytes())
        off += len(rec)
    header = np.array([0x1A412743, version, len(scaffolds), 0], u32).tobytes()
    return header + b"".join(index) + b"".join(records)


def write_fasta(scaffolds: List[Scaffold], path: str, width: int = 60) -> None:
    with open(path, "wb") as fh:
        fh.write(fasta_bytes(scaffolds, width))
