"""BGZF on the host, no GPU: the block table (frisk_b200_bgzf_blocks) and the decoder the inflate kernel runs, built for
the CPU (frisk_b200_bgzf_inflate_host), byte for byte against zlib, and a seeded sweep of corrupted inputs."""
from __future__ import annotations

import ctypes as C
import struct
import zlib

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_member(data: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, extra_before: bytes = b"",
                sync_every: int = 0) -> bytes:
    """One BGZF block of `data` (<= 64 KiB) as bgzip writes it; `extra_before`: subfields placed before BC;
    `sync_every`: Z_SYNC_FLUSH after every that many bytes (empty stored blocks inside the member)."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    if sync_every:
        body = b"".join(c.compress(data[i:i + sync_every]) + c.flush(zlib.Z_SYNC_FLUSH) for i in range(0, len(data), sync_every))
        body += c.flush()
    else:
        body = c.compress(data) + c.flush()
    xfield = extra_before + b"BC" + struct.pack("<HH", 2, 0)
    size = 12 + len(xfield) + len(body) + 8
    xfield = extra_before + b"BC" + struct.pack("<HH", 2, size - 1)
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", len(xfield)) + xfield + body +
            struct.pack("<II", zlib.crc32(data), len(data)))


def bgzf(data: bytes, block: int = 65280, eof: bool = True, **kw) -> bytes:
    parts = [bgzf_member(data[i:i + block], **kw) for i in range(0, len(data), block)]
    return b"".join(parts) + (EOF_BLOCK if eof else b"")


def block_table(gz: bytes, cap=None):
    L = _lib.lib()
    buf = np.frombuffer(gz, np.uint8)
    nb, tl = C.c_uint64(0), C.c_uint64(0)
    rc = L.frisk_b200_bgzf_blocks(engine._ptr(buf), len(buf), 0, None, None, None, None, C.byref(nb), C.byref(tl))
    if rc:
        return rc, None
    n = int(nb.value) if cap is None else cap
    co, cl, crc, to = np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint64)
    rc = L.frisk_b200_bgzf_blocks(engine._ptr(buf), len(buf), n, engine._ptr(co), engine._ptr(cl), engine._ptr(crc),
                                  engine._ptr(to), C.byref(nb), C.byref(tl))
    return rc, dict(comp_off=co, comp_len=cl, crc=crc, text_off=to, n_blocks=int(nb.value), text_len=int(tl.value))


def inflate_host(gz: bytes):
    """(rc, text, status) of the host build of the decoder."""
    rc, t = block_table(gz)
    if rc:
        return rc, None, None
    buf = np.frombuffer(gz, np.uint8)
    out = np.zeros(max(t["text_len"], 1), np.uint8)
    status = np.zeros(max(t["n_blocks"], 1), np.uint32)
    rc = _lib.lib().frisk_b200_bgzf_inflate_host(engine._ptr(buf), engine._ptr(t["comp_off"]), engine._ptr(t["comp_len"]),
                                                 engine._ptr(t["crc"]), engine._ptr(t["text_off"]), t["n_blocks"], t["text_len"],
                                                 engine._ptr(out), engine._ptr(status), None)
    return rc, out[:t["text_len"]].tobytes(), status[:t["n_blocks"]]


def fasta_like(rng, n: int) -> bytes:
    """FASTA text with lower case, IUPAC codes, N runs and CRLF line ends."""
    alphabet = np.frombuffer(b"ACGTACGTACGTacgtNRYKMSWnBDHV", np.uint8)
    seq = alphabet[rng.integers(0, len(alphabet), n)]
    for a in rng.integers(0, n - 3000, 5):
        seq[a:a + rng.integers(100, 3000)] = ord("N")
    lines = [seq[i:i + 70].tobytes() for i in range(0, n, 70)]
    out = []
    for i, ln in enumerate(lines):
        if i % 400 == 0:
            out.append(b">scaf_%d some description\r\n" % i)
        out.append(ln + b"\r\n")
    return b"".join(out)


def corpus():
    """(name, data, writer kwargs): every deflate feature the decoder must handle."""
    rng = np.random.default_rng(2024)
    dna = synth.fasta_bytes(synth.make("C2", 0.005, seed=3))
    period = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 32768)].tobytes()   # repeats only 32,768 bytes back
    return [
        ("stored", dna[:150_000], dict(level=0)),
        ("fixed", dna[:150_000], dict(strategy=zlib.Z_FIXED)),
        ("level1", dna, dict(level=1)),
        ("level6", dna, dict(level=6)),
        ("level9", dna, dict(level=9)),
        ("huffman_only", dna[:200_000], dict(strategy=zlib.Z_HUFFMAN_ONLY)),
        ("rle_n_runs", (b">n\n" + b"N" * 200_000 + b"\nACGT\n" + b"n" * 70_000 + b"\n") * 2, dict(strategy=zlib.Z_RLE)),
        ("sync_flush", dna[:200_000], dict(sync_every=1000)),
        ("max_distance", period * 6, dict(level=9, block=65536)),
        ("random", rng.integers(0, 256, 300_000, dtype=np.uint8).tobytes(), dict(level=6)),
        ("fasta_crlf_iupac", fasta_like(rng, 300_000), dict(level=6)),
        ("small_blocks", dna[:50_000], dict(level=6, block=1000)),
        ("empty_blocks_inside", None, None),
    ]


def make_gz(name, data, kw):
    if name == "empty_blocks_inside":
        a = bgzf(b"ACGT" * 5000, eof=False)
        return a + EOF_BLOCK + bgzf(b">x\nTTTT\n" * 100, eof=False) + EOF_BLOCK + EOF_BLOCK, b"ACGT" * 5000 + b">x\nTTTT\n" * 100
    kw = dict(kw)
    block = kw.pop("block", 65280)
    return bgzf(data, block=block, **kw), data


# ---- block table ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("block", [1, 1000, 65280, 65536])
def test_block_table_matches_writer(block):
    data = synth.fasta_bytes(synth.make("C2", 0.003, seed=1))[:200_000]
    gz = bgzf(data, block=block)
    rc, t = block_table(gz)
    assert rc == _lib.OK
    pieces = [data[i:i + block] for i in range(0, len(data), block)] + [b""]
    assert t["n_blocks"] == len(pieces) and t["text_len"] == len(data)
    pos, toff = 0, 0
    for b, p in enumerate(pieces):
        m = bgzf_member(p) if p else EOF_BLOCK
        xlen = struct.unpack_from("<H", m, 10)[0]
        assert int(t["comp_off"][b]) == pos + 12 + xlen and int(t["comp_len"][b]) == len(m) - 12 - xlen - 8
        assert int(t["crc"][b]) == zlib.crc32(p) and int(t["text_off"][b]) == toff
        pos += len(m)
        toff += len(p)
    if block == 65536:
        assert (np.diff(t["text_off"][:3]) == 65536).all()


def test_block_table_eof_only_and_extra_subfield_first():
    rc, t = block_table(EOF_BLOCK)
    assert rc == _lib.OK and t["n_blocks"] == 1 and t["text_len"] == 0
    data = b">a\nACGT\n" * 1000
    gz = bgzf(data, extra_before=b"XY" + struct.pack("<H", 5) + b"hello")
    rc, t = block_table(gz)
    assert rc == _lib.OK and t["n_blocks"] == 2 and t["text_len"] == len(data)
    assert inflate_host(gz)[1] == data


def test_block_table_refuses_what_is_not_bgzf():
    import gzip
    data = b">a\nACGT\n" * 5000
    good = bgzf(data, block=10000)
    bad = {
        "single_member_gzip": gzip.compress(data),
        "gzip_with_fname": _gzip_fname(data),
        "truncated_last_block": good[:-10],
        "bsize_past_end": good[:-len(EOF_BLOCK)] + EOF_BLOCK[:16] + struct.pack("<H", 200) + EOF_BLOCK[18:],
        "trailing_garbage": good + b"\0\0",
        "bc_slen_4": good.replace(b"BC\x02\x00", b"BC\x04\x00", 1),
    }
    for name, gz in bad.items():
        rc, _ = block_table(gz)
        assert rc == _lib.E_FORMAT, name


def _gzip_fname(data: bytes) -> bytes:
    import gzip
    import io
    bio = io.BytesIO()
    with gzip.GzipFile(filename="genome.fa", mode="wb", fileobj=bio) as fh:
        fh.write(data)
    return bio.getvalue()


def test_block_table_capacity_and_count_only():
    gz = bgzf(b"ACGT" * 40000, block=10000)           # 16 blocks + EOF
    L = _lib.lib()
    buf = np.frombuffer(gz, np.uint8)
    nb, tl = C.c_uint64(0), C.c_uint64(0)
    assert L.frisk_b200_bgzf_blocks(engine._ptr(buf), len(buf), 0, None, None, None, None, C.byref(nb), C.byref(tl)) == _lib.OK
    assert (int(nb.value), int(tl.value)) == (17, 160000)
    rc, _ = block_table(gz, cap=5)
    assert rc == _lib.E_CAPACITY
    assert engine.bgzf_text_len(gz) == 160000 and engine.is_bgzf(gz) and not engine.is_bgzf(b">a\nACGT\n")


# ---- host build of the decoder vs zlib ------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [c[0] for c in corpus()])
def test_host_inflate_equals_zlib(case):
    name, data, kw = next(c for c in corpus() if c[0] == case)
    gz, want = make_gz(name, data, kw)
    import gzip
    assert gzip.decompress(gz) == want                # the writer is right (python's multi-member gzip reads BGZF)
    rc, got, status = inflate_host(gz)
    assert rc == _lib.OK and (status == 0).all()
    assert got == want


def test_host_inflate_empty_input():
    rc, got, _ = inflate_host(b"")
    assert rc == _lib.OK and got == b""


# ---- seeded corruption sweep --------------------------------------------------------------------------------------------
def _zlib_member_ok(gz: bytes) -> bytes | None:
    """What python's gzip makes of a corrupted file: its output, or None if it refuses it."""
    import gzip
    try:
        return gzip.decompress(gz)
    except Exception:
        return None


def test_corruption_sweep():
    rng = np.random.default_rng(77)
    data = synth.fasta_bytes(synth.make("C2", 0.002, seed=5))[:60_000]
    variants = []
    for lvl, strat in ((6, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED), (0, 0), (6, zlib.Z_RLE)):
        gz = bgzf(data, block=20000, level=lvl, strategy=strat)
        rc, t = block_table(gz)
        assert rc == _lib.OK
        for _ in range(60):                            # bit flips in the deflate payloads
            b = int(rng.integers(0, t["n_blocks"] - 1))
            off, ln = int(t["comp_off"][b]), int(t["comp_len"][b])
            x = bytearray(gz)
            x[off + int(rng.integers(0, ln))] ^= 1 << int(rng.integers(0, 8))
            variants.append(bytes(x))
        for _ in range(8):                             # payload truncated (BSIZE and the trailer kept consistent)
            b = int(rng.integers(0, t["n_blocks"] - 1))
            off, ln = int(t["comp_off"][b]), int(t["comp_len"][b])
            cut = int(rng.integers(1, ln))
            head_start = off - 18
            member = gz[head_start:off + ln + 8]
            short = member[:18 + ln - cut] + member[18 + ln:]
            short = short[:16] + struct.pack("<H", len(short) - 1) + short[18:]
            variants.append(gz[:head_start] + short + gz[off + ln + 8:])
        for b in range(min(3, t["n_blocks"] - 1)):       # wrong CRC, wrong ISIZE (larger and smaller)
            end = int(t["comp_off"][b]) + int(t["comp_len"][b])
            for field, delta in ((0, 1), (4, 1), (4, -1)):
                x = bytearray(gz)
                v = struct.unpack_from("<I", x, end + field)[0]
                struct.pack_into("<I", x, end + field, (v + delta) & 0xffffffff)
                variants.append(bytes(x))
    assert len(variants) >= 300
    refused = 0
    for v in variants:
        rc, got, status = inflate_host(v)
        ref = _zlib_member_ok(v)
        if rc == _lib.OK:
            assert ref is not None and got == ref, "accepted a file zlib refuses, or inflated it differently"
        else:
            assert rc == _lib.E_FORMAT
            refused += 1
    assert refused > 250


def test_malformed_streams_are_refused():
    """Hand-made members: each malformation the kernel must refuse, with the same status words on the host."""
    for payload, isize in malformed_payloads():
        m = raw_member(payload, b"x" * isize)
        rc, _, status = inflate_host(m + EOF_BLOCK)
        assert rc == _lib.E_FORMAT and status[0] != 0 and status[1] == 0


def raw_member(payload: bytes, data: bytes, crc=None, isize=None) -> bytes:
    xfield = b"BC" + struct.pack("<HH", 2, 12 + 6 + len(payload) + 8 - 1)
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", 6) + xfield + payload +
            struct.pack("<II", zlib.crc32(data) if crc is None else crc, len(data) if isize is None else isize))


class BitWriter:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, value: int, bits: int):
        self.v |= (value & ((1 << bits) - 1)) << self.n
        self.n += bits

    def put_rev(self, code: int, bits: int):       # Huffman codes go most significant bit first
        self.put(int(format(code, "0%db" % bits)[::-1], 2), bits)

    def bytes(self) -> bytes:
        return self.v.to_bytes((self.n + 7) // 8, "little")


def malformed_payloads():
    """(deflate payload, isize) pairs, one per malformation."""
    out = []
    # block type 3
    w = BitWriter(); w.put(1, 1); w.put(3, 2); out.append((w.bytes(), 1))
    # stored LEN / NLEN mismatch
    w = BitWriter(); w.put(1, 1); w.put(0, 2); w.put(0, 5); w.put(4, 16); w.put(0, 16)
    out.append((w.bytes() + b"abcd", 4))
    # fixed block: literal 'x' then distance 2 at output position 1 (before the first byte)
    w = BitWriter(); w.put(1, 1); w.put(1, 2)
    w.put_rev(0x30 + ord("x"), 8)                       # literal 0..143: 8-bit codes from 00110000
    w.put_rev(1, 7)                                     # length symbol 257 (length 3): 7-bit code 0000001
    w.put_rev(1, 5)                                     # distance symbol 1 (distance 2)
    w.put_rev(0, 7)                                     # end of block
    out.append((w.bytes(), 4))
    # fixed block: litlen symbol 286
    w = BitWriter(); w.put(1, 1); w.put(1, 2); w.put_rev(0xC0 + 6, 8); w.put_rev(0, 7)
    out.append((w.bytes(), 1))
    # fixed block: distance symbol 30
    w = BitWriter(); w.put(1, 1); w.put(1, 2); w.put_rev(0x30 + ord("x"), 8); w.put_rev(1, 7); w.put_rev(30, 5); w.put_rev(0, 7)
    out.append((w.bytes(), 4))
    # dynamic block: over-subscribed code-length code (all 19 lengths 1)
    w = BitWriter(); w.put(1, 1); w.put(2, 2); w.put(0, 5); w.put(0, 5); w.put(15, 4)
    for _ in range(19):
        w.put(1, 3)
    out.append((w.bytes() + b"\0" * 8, 1))
    # dynamic block: the first code length is a repeat (symbol 16) with no previous length
    w = BitWriter(); w.put(1, 1); w.put(2, 2); w.put(0, 5); w.put(0, 5); w.put(0, 4)
    w.put(1, 3); w.put(1, 3); w.put(0, 3); w.put(0, 3)   # lengths of 16 and 17: 1 bit each (codes 0 and 1)
    w.put_rev(0, 1); w.put(0, 2)                          # symbol 16
    out.append((w.bytes() + b"\0" * 8, 1))
    # output beyond ISIZE: two literals, ISIZE 1
    w = BitWriter(); w.put(1, 1); w.put(1, 2); w.put_rev(0x30 + 1, 8); w.put_rev(0x30 + 2, 8); w.put_rev(0, 7)
    out.append((w.bytes(), 1))
    # truncated: a fixed block without its end-of-block code
    w = BitWriter(); w.put(1, 1); w.put(1, 2); w.put_rev(0x30 + ord("x"), 8)
    out.append((w.bytes(), 1))
    return out
