"""Plain gzip on the host, no GPU: the header parse (frisk_b200_gzip_member) and the chunked speculative inflate run on the
CPU with the decoder, plan, joins and repairs of the device path (frisk_b200_gzip_inflate_host), byte for byte against
zlib; a seeded sweep of corrupted inputs; the refusals; and the share of chunk joins speculation gets right."""
from __future__ import annotations

import ctypes as C
import struct
import zlib

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from tests.test_bgzf_host import malformed_payloads

FTEXT, FHCRC, FEXTRA, FNAME, FCOMMENT = 1, 2, 4, 8, 16


def gz_member(data: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, flush_every: int = 0,
              flush_mode: int = zlib.Z_SYNC_FLUSH, flags: int = 0, extra: bytes = b"", fname: bytes = b"genome.fa",
              comment: bytes = b"a comment") -> bytes:
    """One gzip member as gzip / pigz write it; flush_every: a flush (flush_mode) after every that many input bytes."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    if flush_every:
        payload = b"".join(c.compress(data[i:i + flush_every]) + c.flush(flush_mode) for i in range(0, len(data), flush_every))
    else:
        payload = c.compress(data)
    payload += c.flush()
    head = b"\x1f\x8b\x08" + bytes([flags]) + b"\0\0\0\0\0\x03"
    if flags & FEXTRA:
        head += struct.pack("<H", len(extra)) + extra
    if flags & FNAME:
        head += fname + b"\0"
    if flags & FCOMMENT:
        head += comment + b"\0"
    if flags & FHCRC:
        head += struct.pack("<H", zlib.crc32(head) & 0xffff)
    return head + payload + struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff)


def inflate_host(gz: bytes, cap: int | None = None):
    """(rc, text, stats) of frisk_b200_gzip_inflate_host."""
    buf = np.frombuffer(gz, np.uint8).copy() if gz else np.zeros(1, np.uint8)
    if cap is None:
        cap = 8 * len(gz) + 1024
        for _ in range(2):                              # (the real length comes back with FRISK_E_CAPACITY)
            rc, text, stats = inflate_host(gz, cap)
            if rc != _lib.E_CAPACITY:
                return rc, text, stats
            cap = int(stats[4])
    out = np.zeros(max(cap, 1), np.uint8)
    tl = C.c_uint64(0)
    st = np.zeros(4, np.uint64)
    rc = _lib.lib().frisk_b200_gzip_inflate_host(engine._ptr(buf), len(gz), engine._ptr(out), cap, C.byref(tl), engine._ptr(st), None)
    return rc, out[:min(int(tl.value), cap)].tobytes(), list(map(int, st)) + [int(tl.value)]


def set_chunk(v: int):
    _lib.check(_lib.lib().frisk_b200_set_option(b"gzip_chunk_bytes", v), "set_option")


@pytest.fixture
def chunk_bytes():
    yield set_chunk
    set_chunk(0)


def dna(scale=0.005, seed=3) -> bytes:
    return synth.fasta_bytes(synth.make("C2", scale, seed=seed))


def n_heavy() -> bytes:
    """Long N runs: more than 1000 bytes of text per compressed byte, far beyond the first pass's scratch."""
    return (b">n\n" + b"N" * 1_500_000 + b"\nACGTTGCA\n" + b"n" * 700_000 + b"\n") * 2 + dna(0.002)


def raw_deflate(data: bytes) -> bytes:
    c = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
    return c.compress(data) + c.flush()


def corpus():
    """(name, gzip file, text): the deflate features, flushes, header flags and sizes the inflate must handle."""
    d = dna()
    big_extra = bytes(range(256)) * 255                 # 65,280 bytes of FEXTRA, then a 4 KiB name: a 69 KB header
    rows = [
        ("level0", gz_member(d[:300_000], level=0)),
        ("level1", gz_member(d, level=1)),
        ("level6", gz_member(d, level=6)),
        ("level9", gz_member(d, level=9)),
        ("filtered", gz_member(d, strategy=zlib.Z_FILTERED)),
        ("huffman_only", gz_member(d[:300_000], strategy=zlib.Z_HUFFMAN_ONLY)),
        ("rle", gz_member(d, strategy=zlib.Z_RLE)),
        ("fixed", gz_member(d[:300_000], strategy=zlib.Z_FIXED)),
        ("sync_flush", gz_member(d, flush_every=30_000, flush_mode=zlib.Z_SYNC_FLUSH)),
        ("full_flush", gz_member(d, flush_every=30_000, flush_mode=zlib.Z_FULL_FLUSH)),
        ("ftext", gz_member(d[:100_000], flags=FTEXT)),
        ("fhcrc", gz_member(d[:100_000], flags=FHCRC)),
        ("fextra", gz_member(d[:100_000], flags=FEXTRA, extra=b"AB\x02\0xy")),
        ("fname", gz_member(d[:100_000], flags=FNAME)),
        ("fcomment", gz_member(d[:100_000], flags=FCOMMENT)),
        ("all_flags", gz_member(d[:100_000], flags=31, extra=b"XY\x01\0z")),
        ("header_over_64k", gz_member(d[:100_000], flags=FEXTRA | FNAME | FHCRC, extra=big_extra, fname=b"g" * 4096)),
        ("empty", gz_member(b"")),
        ("n_runs", gz_member(n_heavy())),
        ("random", gz_member(np.random.default_rng(5).integers(0, 256, 200_000, dtype=np.uint8).tobytes())),
        ("stored_deflate", gz_member(raw_deflate(d), level=0)),   # real dynamic headers inside stored blocks: false starts
    ]
    texts = {"level0": d[:300_000], "huffman_only": d[:300_000], "fixed": d[:300_000], "empty": b"", "n_runs": n_heavy(),
             "random": np.random.default_rng(5).integers(0, 256, 200_000, dtype=np.uint8).tobytes(), "stored_deflate": raw_deflate(d)}
    for name in ("ftext", "fhcrc", "fextra", "fname", "fcomment", "all_flags", "header_over_64k"):
        texts[name] = d[:100_000]
    return [(name, gz, texts.get(name, d)) for name, gz in rows]


_CORPUS = None


def corpus_case(name):
    global _CORPUS
    if _CORPUS is None:
        _CORPUS = {n: (gz, t) for n, gz, t in corpus()}
    return _CORPUS[name]


CASES = [n for n, _, _ in corpus()]


@pytest.mark.parametrize("case", CASES)
def test_host_inflate_equals_zlib(case):
    gz, want = corpus_case(case)
    assert zlib.decompress(gz, 31) == want            # the writer is right
    rc, got, st = inflate_host(gz)
    assert rc == _lib.OK and got == want
    assert st[1] <= st[0] - 1 or st[0] == 1
    if case == "n_runs":
        assert st[3] > 0                                # the N runs outgrew the first pass's scratch
    if case == "stored_deflate":
        assert st[2] > 0                                # chunks that started at a false candidate were decoded again


@pytest.mark.parametrize("chunk", [1024, 4096, 65536, 1 << 30])
@pytest.mark.parametrize("case", ["level1", "level6", "level9", "sync_flush", "full_flush", "fixed", "level0", "n_runs",
                                  "stored_deflate"])
def test_forced_chunk_sizes(case, chunk, chunk_bytes):
    """From 1 KiB windows (many false candidates, merges and repairs) to one chunk for the whole stream."""
    gz, want = corpus_case(case)
    chunk_bytes(chunk)
    rc, got, st = inflate_host(gz)
    assert rc == _lib.OK and got == want
    if chunk == 1 << 30:
        assert st[:3] == [1, 0, 0]


def test_no_dynamic_blocks_is_one_chunk():
    for case in ("level0", "fixed"):
        gz, want = corpus_case(case)
        rc, got, st = inflate_host(gz)
        assert rc == _lib.OK and got == want and st[2] == 0


def test_capacity_reports_the_length():
    gz, want = corpus_case("level6")
    rc, _, st = inflate_host(gz, cap=100)
    assert rc == _lib.E_CAPACITY and st[4] == len(want)


def test_member_header():
    L = _lib.lib()
    for flags in (0, FTEXT, FHCRC, FEXTRA, FNAME, FCOMMENT, 31):
        data = b">a\nACGT\n" * 100
        gz = gz_member(data, flags=flags, extra=b"AB\x01\0q")
        payload = raw_deflate(data)
        off, ln = C.c_uint64(0), C.c_uint64(0)
        crc, isize = C.c_uint32(0), C.c_uint32(0)
        buf = np.frombuffer(gz, np.uint8).copy()
        assert L.frisk_b200_gzip_member(engine._ptr(buf), len(gz), C.byref(off), C.byref(ln), C.byref(crc), C.byref(isize)) == _lib.OK
        assert ln.value == len(payload) and off.value + ln.value + 8 == len(gz) and gz[off.value:off.value + ln.value] == payload
        assert crc.value == zlib.crc32(data) and isize.value == len(data)
    for bad in (b"\x1f\x8b\x08\x20" + b"\0" * 30, b"\x1f\x8b\x07\x00" + b"\0" * 30, b"\x1f\x8b\x08\x08abc", b"PK\x03\x04" + b"\0" * 30):
        buf = np.frombuffer(bad, np.uint8).copy()
        assert L.frisk_b200_gzip_member(engine._ptr(buf), len(bad), None, None, None, None) == _lib.E_FORMAT


def test_refusals():
    data = dna(0.002)
    gz = gz_member(data)
    assert inflate_host(gz)[0] == _lib.OK
    assert inflate_host(gz[:len(gz) // 2])[0] == _lib.E_FORMAT                   # truncated
    assert inflate_host(gz[:-8])[0] == _lib.E_FORMAT                             # no trailer
    x = bytearray(gz); x[-8] ^= 1
    assert inflate_host(bytes(x))[0] == _lib.E_FORMAT                           # bad CRC32
    x = bytearray(gz); x[-4] ^= 1
    assert inflate_host(bytes(x))[0] == _lib.E_FORMAT                           # bad ISIZE
    assert inflate_host(gz + b"\0")[0] == _lib.E_FORMAT                          # trailing garbage
    assert inflate_host(gz + b"junk" * 10)[0] == _lib.E_FORMAT
    assert inflate_host(gz + gz_member(b">b\nAC\n"))[0] == _lib.E_UNSUPPORTED    # multi-member
    x = bytearray(gz_member(data, flags=FHCRC)); x[10] ^= 1
    assert inflate_host(bytes(x))[0] == _lib.E_FORMAT                           # header CRC16
    for payload, isize in malformed_payloads():
        m = b"\x1f\x8b\x08\0\0\0\0\0\0\x03" + payload + struct.pack("<II", zlib.crc32(b"x" * isize), isize)
        assert inflate_host(m)[0] == _lib.E_FORMAT


def test_match_before_the_text_is_refused(chunk_bytes):
    """20 KB of text, then a match of distance 32,768: before the first byte, found by chunk 0's decoder (one chunk) or
    when the placeholders are resolved (small chunks)."""
    from tests.test_bgzf_host import BitWriter
    short = dna(0.002)[:20_000]
    c = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
    body = c.compress(short) + c.flush(zlib.Z_SYNC_FLUSH)
    w = BitWriter(); w.put(1, 1); w.put(1, 2)
    w.put_rev(0b0010111, 7); w.put(0, 4)               # length symbol 279: length 99
    w.put_rev(29, 5); w.put(8191, 13)                   # distance symbol 29 + 8,191: distance 32,768
    w.put_rev(0, 7)
    gz = b"\x1f\x8b\x08\0\0\0\0\0\0\x03" + body + w.bytes() + struct.pack("<II", 0, len(short) + 99)
    for chunk in (0, 1024):
        chunk_bytes(chunk)
        assert inflate_host(gz)[0] == _lib.E_FORMAT


def test_speculation_accepts_joins():
    """Scaled C2 at level 6 with the default chunk size: at least 95 % of the joins are right on the first pass (the
    count is deterministic); without this an always-serial inflate would pass every other test."""
    text = synth.fasta_bytes(synth.config_c2(scale=0.25))
    gz = gz_member(text, level=6)
    rc, got, st = inflate_host(gz)
    assert rc == _lib.OK and got == text
    assert st[0] >= 100, st
    assert st[1] >= 0.95 * (st[0] - 1), st


def test_is_gzip_and_raw_reader(tmp_path):
    from tests.test_bgzf_host import bgzf
    text = b">a\nACGT\n" * 1000
    files = {"g.fa.gz": (gz_member(text), "gzip"), "b.fa.gz": (bgzf(text), "bgzf"), "t.fa": (text, "text"),
             "m.fa.gz": (gz_member(text) + gz_member(text), "gzip")}
    for name, (data, kind) in files.items():
        p = tmp_path / name
        p.write_bytes(data)
        buf, k = engine.read_genome_raw(str(p))
        assert k == kind and bytes(buf) == data
    assert engine.is_gzip(gz_member(text)) and not engine.is_gzip(bgzf(text)) and not engine.is_gzip(text)
    assert engine.read_genome_file(str(tmp_path / "g.fa.gz"))[1] is False           # (its contract is unchanged)


# ---- seeded corruption sweep --------------------------------------------------------------------------------------------
def _python_gzip(gz: bytes) -> bytes | None:
    import gzip
    try:
        return gzip.decompress(gz)
    except Exception:
        return None


def test_corruption_sweep(chunk_bytes):
    rng = np.random.default_rng(99)
    data = dna(0.002)[:120_000]
    variants = []
    for lvl, strat, flags in ((6, zlib.Z_DEFAULT_STRATEGY, 0), (1, zlib.Z_DEFAULT_STRATEGY, FNAME), (6, zlib.Z_FIXED, 0), (0, 0, 0),
                              (6, zlib.Z_RLE, FHCRC | FEXTRA)):
        gz = gz_member(data, level=lvl, strategy=strat, flags=flags, extra=b"AB\x01\0q")
        for _ in range(60):                             # bit flips anywhere
            x = bytearray(gz)
            x[int(rng.integers(0, len(gz)))] ^= 1 << int(rng.integers(0, 8))
            variants.append(bytes(x))
        for _ in range(6):                              # truncated, trailer kept
            cut = int(rng.integers(1, len(gz) - 30))
            variants.append(gz[:len(gz) - 8 - cut] + gz[-8:])
    assert len(variants) >= 300
    refused = 0
    for i, v in enumerate(variants):
        chunk_bytes(2048 if i % 2 else 0)               # half of them through many small chunks
        rc, got, _ = inflate_host(v)
        ref = _python_gzip(v)
        if rc == _lib.OK:
            assert ref is not None and got == ref, "accepted a file python's gzip refuses, or inflated it differently"
        else:
            assert rc in (_lib.E_FORMAT, _lib.E_UNSUPPORTED)
            refused += 1
    assert refused > 250
