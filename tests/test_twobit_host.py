"""UCSC .2bit on the host, no GPU: the parser (frisk_b200_2bit_records) and the host decoder (frisk_b200_2bit_unpack_host,
the device path's plan and per-word code run on the CPU) against the FASTA scanner and packer on the same genome, bit for
bit -- a hand-built file, the writer's files over a corpus of edge cases, both byte orders and both versions -- and the
refusals of malformed files."""
from __future__ import annotations

import ctypes as C
import struct

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth

FIXTURE = bytes.fromhex(
    "43 27 41 1a 00 00 00 00 01 00 00 00 00 00 00 00 01 73 16 00 00 00 08 00 00 00 01 00 00 00"
    "04 00 00 00 02 00 00 00 01 00 00 00 06 00 00 00 02 00 00 00 00 00 00 00 1b 09")
FIXTURE_FASTA = b">s\nTCAGNNac\n"


def build(records, big_endian=False, version=0, reverse_layout=False):
    """A .2bit file from raw records, independent of synth.twobit_bytes: records = [(name, dna_size, n_blocks, mask_blocks,
    packed)], blocks as lists of (start, size) written in the given order; reverse_layout puts the records into the file in
    the reverse of index order."""
    e = ">" if big_endian else "<"
    bodies = []
    for name, size, nbl, mbl, packed in records:
        b = struct.pack(e + "II", size, len(nbl)) + b"".join(struct.pack(e + "I", s) for s, _ in nbl)
        b += b"".join(struct.pack(e + "I", z) for _, z in nbl)
        b += struct.pack(e + "I", len(mbl)) + b"".join(struct.pack(e + "I", s) for s, _ in mbl)
        b += b"".join(struct.pack(e + "I", z) for _, z in mbl) + struct.pack(e + "I", 0) + packed
        bodies.append(b)
    idx_len = sum(1 + len(r[0]) + (4 if version == 0 else 8) for r in records)
    order = list(range(len(records)))[::-1] if reverse_layout else list(range(len(records)))
    offs, at = [0] * len(records), 16 + idx_len
    for i in order:
        offs[i] = at
        at += len(bodies[i])
    index = b"".join(bytes([len(r[0])]) + r[0] + struct.pack(e + ("I" if version == 0 else "Q"), o) for r, o in zip(records, offs))
    return struct.pack(e + "IIII", 0x1A412743, version, len(records), 0) + index + b"".join(bodies[i] for i in order)


def fixture(big_endian=False, version=0):
    return build([(b"s", 8, [(4, 2)], [(6, 2)], b"\x1b\x09")], big_endian, version)


def pack_seq(seq: bytes) -> bytes:
    code = {ord(c): v for c, v in zip("TCAGtcag", (0, 1, 2, 3, 0, 1, 2, 3))}
    v = [code.get(c, 0) for c in seq] + [0] * (-len(seq) % 4)
    return bytes((v[i] << 6) | (v[i + 1] << 4) | (v[i + 2] << 2) | v[i + 3] for i in range(0, len(v), 4))


def records(buf):
    a = np.frombuffer(buf, np.uint8)
    n, bases = C.c_uint64(0), C.c_uint64(0)
    rc = _lib.lib().frisk_b200_2bit_records(engine._ptr(a), len(buf), 0, None, None, None, C.byref(n), C.byref(bases))
    return rc, int(n.value), int(bases.value)


def assert_same(a: engine.PackedGenome, b: engine.PackedGenome):
    assert list(a.names) == list(b.names)
    assert np.array_equal(a.scaf_len, b.scaf_len) and np.array_equal(a.scaf_off, b.scaf_off)
    assert a.padded_len == b.padded_len
    assert (a.total_len, a.nn_total, a.n_lower) == (b.total_len, b.nn_total, b.n_lower)
    assert np.array_equal(a.codes, b.codes) and np.array_equal(a.inv, b.inv)
    assert (a.low is None) == (b.low is None)
    if b.low is not None:
        assert np.array_equal(a.low, b.low)


def test_hand_built_fixture_in_every_form():
    assert fixture() == FIXTURE and len(FIXTURE) == 56
    be = fixture(big_endian=True)
    assert be[:4] == bytes.fromhex("1a412743")
    want = engine.PackedGenome.from_fasta_bytes(FIXTURE_FASTA)
    assert (want.total_len, want.nn_total, want.n_lower) == (8, 4, 2)
    for buf in (FIXTURE, be, fixture(version=1), fixture(big_endian=True, version=1)):
        assert records(buf) == (_lib.OK, 1, 8)
        off, ln = engine.twobit_records(buf)[:2]
        assert buf[int(off[0]):int(off[0]) + int(ln[0])] == b"s"
        assert_same(engine.PackedGenome.from_2bit_bytes(buf), want)


def corpus():
    rng = np.random.default_rng(31)

    def bases(n, alphabet=b"ACGT"):
        return np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)].copy()

    a = bases(5000)
    a[100:400] = np.frombuffer(b"acgt", np.uint8)[rng.integers(0, 4, 300)]             # soft-masked
    a[1000:1010] = np.frombuffer(b"RYKMSWBDHV", np.uint8)                              # IUPAC
    a[1500:1505] = np.frombuffer(b"rykms", np.uint8)                                   # lower-case IUPAC: invalid only
    a[2000:2040] = ord("n")                                                            # lower-case n: soft-masked N
    a[3000:3100] = ord("N")
    a[3050:3060] = ord("n")
    a[4000:4003] = ord("-")
    b = bases(300)
    b[:37] = ord("N")                                                                  # N run at the start ...
    b[-45:] = ord("N")                                                                 # ... and at the end
    c = bases(1000)
    c[29:131] = ord("N")                                                               # across several plane words
    c[200:260] = np.char.lower(c[200:260].view("S1")).view(np.uint8)
    c[230:240] = ord("n")
    return [("mixed", a), ("n_ends", b), ("all_N", np.full(333, ord("N"), np.uint8)), ("all_n", np.full(70, ord("n"), np.uint8)),
            ("empty", np.zeros(0, np.uint8)), ("len1", bases(1)), ("len2", bases(2)), ("len3", bases(3)), ("len5", bases(5)),
            ("len127", bases(127)), ("len128", bases(128)), ("len129", bases(129)), ("span", c),
            ("lower_all", bases(77, b"acgt")), ("masked_tail", np.concatenate([bases(64), bases(63, b"acgtn")])),
            ("empty2", np.zeros(0, np.uint8))]


@pytest.mark.parametrize("big_endian,version", [(False, 0), (True, 0), (False, 1), (True, 1)])
def test_writer_round_trip(big_endian, version):
    sc = corpus()
    buf = synth.twobit_bytes(sc, big_endian=big_endian, version=version)
    assert engine.is_2bit(buf)
    assert_same(engine.PackedGenome.from_2bit_bytes(buf), engine.PackedGenome.from_fasta_bytes(synth.fasta_bytes(sc)))


def test_writer_round_trip_fragmented_assembly():
    sc = synth.make("C5", 2e-5, seed=12) + synth.make("edge") + synth.make("edge_short")
    assert len(sc) > 20
    for be in (False, True):
        buf = synth.twobit_bytes(sc, big_endian=be)
        assert_same(engine.PackedGenome.from_2bit_bytes(buf), engine.PackedGenome.from_fasta_bytes(synth.fasta_bytes(sc)))


def _blocks(flag):
    d = np.diff(np.concatenate([[0], flag.astype(np.int8), [0]]))
    s = np.nonzero(d == 1)[0]
    return list(zip(s.tolist(), (np.nonzero(d == -1)[0] - s).tolist()))


def test_shuffled_overlapping_and_zero_size_blocks_out_of_file_order():
    """Blocks in any order, overlapping, split, or of size zero, and records stored in the reverse of index order: OR-ed into
    the planes, they give the same genome."""
    rng = np.random.default_rng(5)
    sc = corpus()
    recs = []
    for name, seq in sc:
        s = bytes(seq)
        up = np.frombuffer(s, np.uint8) & 0xDF
        nb = _blocks(~np.isin(up, np.frombuffer(b"ACGT", np.uint8)))
        mb = _blocks(np.frombuffer(s, np.uint8) >= ord("a"))
        pieces = []
        for st, sz in nb + mb:                                         # every block as two overlapping halves, plus an empty one
            h = sz // 2 + 1
            pieces.append(((st, min(h + 3, sz)), (st + h - 1, sz - h + 1) if sz >= h else (st, 1)))
        nsplit = [p for (st, sz), pr in zip(nb + mb, pieces) if (st, sz) in nb for p in pr] + [(len(s) // 2, 0)]
        msplit = [p for (st, sz), pr in zip(nb + mb, pieces) if (st, sz) not in nb for p in pr] + [(0, 0)]
        rng.shuffle(nsplit)
        rng.shuffle(msplit)
        recs.append((name.encode(), len(s), nsplit, msplit, pack_seq(s)))
    want = engine.PackedGenome.from_fasta_bytes(synth.fasta_bytes(sc))
    for be in (False, True):
        assert_same(engine.PackedGenome.from_2bit_bytes(build(recs, big_endian=be, version=1, reverse_layout=True)), want)


def test_refusals():
    good = synth.twobit_bytes([("a", np.frombuffer(b"ACGTNNacgt" * 5, np.uint8)), ("b", np.frombuffer(b"ACGTACG", np.uint8))])
    assert records(good) == (_lib.OK, 2, 57)
    bad = {
        "signature": b"\0\0\0\0" + good[4:],
        "version_2": good[:4] + struct.pack("<I", 2) + good[8:],
        "empty_name": build([(b"", 4, [], [], b"\x1b")]),
        "offset_past_end": good[:18] + struct.pack("<I", len(good) + 5) + good[22:],
        "block_past_size": build([(b"s", 8, [(4, 5)], [], b"\x1b\x09")]),
        "mask_block_past_size": build([(b"s", 8, [], [(0, 9)], b"\x1b\x09")]),
        "block_start_past_size": build([(b"s", 8, [(9, 0)], [], b"\x1b\x09")]),
        "huge_block_count": build([(b"s", 8, [], [], b"\x1b\x09")])[:26] + struct.pack("<I", 0x40000000) + b"\0" * 30,
    }
    ends = {"header": 10, "index": 20, "record_header": 28, "n_blocks": 34, "mask_blocks": 48, "packed_dna": 55}
    for what, cut in ends.items():                                    # truncated inside each part of FIXTURE
        bad["truncated_" + what] = FIXTURE[:cut]
    bad["truncated_index_of_many"] = struct.pack("<IIII", 0x1A412743, 0, 0xFFFFFFFF, 0) + b"\x01s"
    for name, buf in bad.items():
        assert records(buf)[0] == _lib.E_FORMAT, name
        with pytest.raises(_lib.FriskError) as ei:
            engine.PackedGenome.from_2bit_bytes(buf)
        assert ei.value.code == _lib.E_FORMAT, name
    assert records(FIXTURE[:56])[0] == _lib.OK


def test_capacity_and_count_only():
    sc = corpus()
    buf = np.frombuffer(synth.twobit_bytes(sc), np.uint8)
    L = _lib.lib()
    n, bases = C.c_uint64(0), C.c_uint64(0)
    assert L.frisk_b200_2bit_records(engine._ptr(buf), len(buf), 0, None, None, None, C.byref(n), None) == _lib.OK
    assert n.value == len(sc)
    seq_len = np.zeros(len(sc), np.uint64)
    rc = L.frisk_b200_2bit_records(engine._ptr(buf), len(buf), 3, None, None, engine._ptr(seq_len), C.byref(n), C.byref(bases))
    assert rc == _lib.E_CAPACITY and n.value == len(sc) and bases.value == synth.total_bases(sc)
    name_off = np.zeros(len(sc), np.uint64); name_len = np.zeros(len(sc), np.uint32)
    assert L.frisk_b200_2bit_records(engine._ptr(buf), len(buf), len(sc), engine._ptr(name_off), engine._ptr(name_len),
                                      engine._ptr(seq_len), C.byref(n), C.byref(bases)) == _lib.OK
    assert [bytes(buf[o:o + l]).decode() for o, l in zip(name_off, name_len)] == [nm for nm, _ in sc]
    assert seq_len.tolist() == [len(s) for _, s in sc]
    # the host decoder checks the layout it is given, and refuses lower case without a plane for it
    g = engine.PackedGenome.from_2bit_bytes(buf)
    codes, inv, low = (np.zeros(g.padded_len // d, np.uint32) for d in (16, 32, 32))
    st = np.zeros(3, np.uint64)
    f = L.frisk_b200_2bit_unpack_host
    assert f(engine._ptr(buf), len(buf), g.padded_len + 128, engine._ptr(codes), engine._ptr(inv), engine._ptr(low), engine._ptr(st)) == _lib.E_INVALID
    assert f(engine._ptr(buf), len(buf), g.padded_len, engine._ptr(codes), engine._ptr(inv), None, engine._ptr(st)) == _lib.E_FORMAT
    upper = np.frombuffer(synth.twobit_bytes([("u", np.frombuffer(b"ACGTN" * 9, np.uint8))]), np.uint8)
    gu = engine.PackedGenome.from_2bit_bytes(upper)
    assert gu.low is None and gu.nn_total == 9
    c2, i2 = np.zeros(gu.padded_len // 16, np.uint32), np.zeros(gu.padded_len // 32, np.uint32)
    assert f(engine._ptr(upper), len(upper), gu.padded_len, engine._ptr(c2), engine._ptr(i2), None, engine._ptr(st)) == _lib.OK
    assert np.array_equal(c2, gu.codes) and np.array_equal(i2, gu.inv)


def test_engine_dispatch_by_signature(tmp_path):
    sc = [("x", np.frombuffer(b"ACGTacgtNN", np.uint8))]
    text = synth.fasta_bytes(sc)
    for be in (False, True):
        data = synth.twobit_bytes(sc, big_endian=be)
        for fname in ("g.2bit", "g.fa", "g.fa.gz", "genome"):
            p = tmp_path / (("be_" if be else "le_") + fname)
            p.write_bytes(data)
            buf, kind = engine.read_genome_raw(str(p))
            assert kind == "2bit" and bytes(buf) == data, fname
            assert_same(engine.PackedGenome.from_fasta(str(p)), engine.PackedGenome.from_fasta_bytes(text))
    p = tmp_path / "t.fa"
    p.write_bytes(text)
    assert engine.read_genome_raw(str(p))[1] == "text"
    assert not engine.is_2bit(text) and not engine.is_2bit(FIXTURE[:15])
