"""BGZF on the device: the inflate kernel (frisk_b200_bgzf_inflate) byte for byte against zlib, malformed members refused
without a CUDA error, the BGZF open (frisk_b200_fasta_open_bgzf) against the text open of the inflated text, the one-call
path (frisk_b200_run_fasta_bgzf) against frisk_b200_run_fasta, and the CLI on a BGZF, a gzip and a plain file."""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from tests.helpers import Golden
from tests.test_bgzf_host import EOF_BLOCK, bgzf, block_table, corpus, make_gz, malformed_payloads, raw_member
from tests.test_ingest_gpu import _assert_same, fasta_text, ingest_options

pytestmark = pytest.mark.gpu


def inflate_device(gz: bytes):
    """(rc, text) of frisk_b200_bgzf_inflate; rc is FRISK_E_FORMAT when a status word is set."""
    import torch
    rc, t = block_table(gz)
    assert rc == _lib.OK
    dev = torch.device("cuda:0")
    as_dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).to(dev)
    d_gz = as_dev(np.frombuffer(gz, np.uint8).copy(), np.uint8)
    co, to = as_dev(t["comp_off"], np.int64), as_dev(t["text_off"], np.int64)
    cl, crc = as_dev(t["comp_len"], np.int32), as_dev(t["crc"], np.int32)
    d_text = torch.zeros(t["text_len"] + 1, dtype=torch.uint8, device=dev)
    status = torch.zeros(max(t["n_blocks"], 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().frisk_b200_bgzf_inflate(engine._ptr(d_gz), engine._ptr(co), engine._ptr(cl), engine._ptr(crc),
                                                      engine._ptr(to), t["n_blocks"], t["text_len"], engine._ptr(d_text),
                                                      engine._ptr(status), engine._stream_ptr(dev)), "frisk_b200_bgzf_inflate")
        torch.cuda.synchronize()
    bad = bool((status[:t["n_blocks"]] != 0).any().item())
    return (_lib.E_FORMAT if bad else _lib.OK), d_text[:t["text_len"]].cpu().numpy().tobytes()


@pytest.mark.parametrize("case", [c[0] for c in corpus()])
def test_device_inflate_equals_zlib(case):
    name, data, kw = next(c for c in corpus() if c[0] == case)
    gz, want = make_gz(name, data, kw)
    rc, got = inflate_device(gz)
    assert rc == _lib.OK and got == want


def test_device_inflate_c2_scale():
    text = synth.fasta_bytes(synth.config_c2(scale=0.1))
    gz = bgzf(text, level=1)
    rc, got = inflate_device(gz)
    assert rc == _lib.OK and got == text


def test_device_inflate_refuses_malformed_members():
    """One run each: bad Huffman table, distance too far, bad CRC, wrong ISIZE, truncated payload, block type 3.  Each is
    FRISK_E_FORMAT, leaves no CUDA error behind, and the next valid call succeeds."""
    import torch
    pl = malformed_payloads()
    data = b">a\nACGT\n" * 3000
    good = bgzf(data)
    ok_member = good[:-len(EOF_BLOCK)]
    cases = {
        "bad_huffman_table": raw_member(pl[5][0], b"x" * pl[5][1]),
        "distance_too_far": raw_member(pl[2][0], b"x" * pl[2][1]),
        "bad_crc": raw_member(ok_member[18:-8], data, crc=0x12345678),
        "wrong_isize": raw_member(ok_member[18:-8], data, isize=len(data) - 1),
        "truncated_payload": raw_member(ok_member[18:-40], data),
        "block_type_3": raw_member(pl[0][0], b"x" * pl[0][1]),
    }
    for name, member in cases.items():
        rc, _ = inflate_device(ok_member + member + EOF_BLOCK)
        assert rc == _lib.E_FORMAT, name
        torch.cuda.synchronize()
        rc, got = inflate_device(good)
        assert rc == _lib.OK and got == data, name


# ---- the BGZF open against the text open --------------------------------------------------------------------------------
def _open_inputs():
    rng = np.random.default_rng(11)
    sc = synth.make("C2", 0.01, seed=4)
    text = fasta_text(sc, 60)
    long_header = (b">" + b"h" * 70_000 + b" tail\n" + b"ACGT" * 30_000 + b"\n>second\n" +
                   np.frombuffer(b"ACGTacgtN", np.uint8)[rng.integers(0, 9, 100_000)].tobytes() + b"\n")
    return {
        # blocks of 1000 / 777 bytes: boundaries inside header lines and inside sequence lines
        "c2_blocks_1000": (text, dict(block=1000)),
        "c2_blocks_777": (text, dict(block=777, level=1)),
        "c2_default_blocks": (text, dict()),
        "header_over_64k": (long_header, dict()),
    }


@pytest.mark.parametrize("case", list(_open_inputs()))
def test_fasta_open_bgzf_equals_text_open(case):
    text, kw = _open_inputs()[case]
    gz = bgzf(text, **kw)
    host = engine.PackedGenome.from_fasta_bytes(text)
    for mode in ("default", "chunk1", "chunk3", "exact"):
        with ingest_options(mode):
            dev = engine.DeviceGenome.from_bgzf_bytes(gz)
            ref = engine.DeviceGenome.from_fasta_bytes(text)
        _assert_same(dev.to_host(), host)
        _assert_same(ref.to_host(), host)
        assert list(dev.host.names) == list(ref.host.names)
    nat = engine.DeviceGenome.from_bgzf_bytes_native(gz)
    assert list(nat.host.names) == list(host.names) and np.array_equal(nat.host.scaf_len, host.scaf_len)


def test_fasta_open_bgzf_empty_header_and_empty_file():
    for mode in ("default", "exact"):
        with ingest_options(mode):
            with pytest.raises(_lib.FriskError) as ei:
                engine.DeviceGenome.from_bgzf_bytes(bgzf(b">ok\nACGT\n>\nACGT\n"))
            assert ei.value.code == _lib.E_FORMAT
            for gz in (b"", EOF_BLOCK, bgzf(b"")):
                g = engine.DeviceGenome.from_bgzf_bytes(gz).to_host()
                _assert_same(g, engine.PackedGenome.from_fasta_bytes(b""))
    with pytest.raises(_lib.FriskError) as ei:                     # a corrupt member is never scored
        engine.DeviceGenome.from_bgzf_bytes(bgzf(b">a\nACGT\n" * 1000)[:-len(EOF_BLOCK) - 8] + b"\0" * 8 + EOF_BLOCK)
    assert ei.value.code == _lib.E_FORMAT


# ---- the one-call path ------------------------------------------------------------------------------------------------------
def _same_result(a, b, what):
    assert np.array_equal(a.rows, b.rows, equal_nan=True), what
    assert np.array_equal(a.status, b.status) and np.array_equal(a.tables, b.tables), what
    assert tuple(a.meta) == tuple(b.meta) and list(a.names) == list(b.names), what
    assert np.array_equal(a.coords, b.coords), what


@pytest.mark.parametrize("kw", [dict(kmax=8), dict(kmax=6), dict(kmax=9, w=2000, step=1000), dict(kmax=8, scaffolds_all=True)],
                         ids=["k8_device_tail", "k6_host_tail", "k9_host_tail", "scaffolds_all"])
def test_run_fasta_bgzf_equals_run_fasta(kw):
    sc = synth.make("C2", 0.02, seed=8) + synth.make("edge")
    text = fasta_text(sc, 60)
    gz = bgzf(text, block=30000)
    want = engine.run_fasta(text, **kw)
    for mode in ("default", "chunk1", "exact"):
        with ingest_options(mode):
            got = engine.run_fasta_bgzf(gz, **kw)
        _same_result(got, want, mode)
    small = engine.HostOutputs(1, kw["kmax"])                           # FRISK_E_CAPACITY, second stage on the handles
    _same_result(engine.run_fasta_bgzf(gz, out=small, **kw), want, "capacity")


def test_run_fasta_bgzf_mask_host_and_golden():
    gold = Golden("edge_maskHost")
    host = gold.host()
    qtext, htext = fasta_text(gold.scaffolds()), fasta_text(host) if host is not None else fasta_text(gold.scaffolds()[::-1])
    want = engine.run_fasta(qtext, htext, **gold.kwargs())
    _same_result(engine.run_fasta_bgzf(bgzf(qtext, block=5000), bgzf(htext, block=7000), **gold.kwargs()), want, "maskHost")
    from tests.test_gpu_parity import _check_against_golden
    gold = Golden("edge_scaffoldsAll")
    res = engine.run_fasta_bgzf(bgzf(fasta_text(gold.scaffolds()), block=3000), **gold.kwargs())
    _check_against_golden(res, gold, "edge_scaffoldsAll[run_fasta_bgzf]")


def test_run_fasta_bgzf_timing_mark():
    text = fasta_text(synth.make("C2", 0.02, seed=3), 60)
    engine.run_fasta_bgzf(bgzf(text))
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    assert 0.0 < ms[0] <= ms[4]                                       # compressed bytes uploaded and inflated, then the rest


# ---- CLI ----------------------------------------------------------------------------------------------------------------------
def test_cli_bgzf_gzip_and_text_give_identical_products(tmp_path):
    import subprocess
    import sys
    g = synth.make("C2", 0.01, seed=21) + synth.make("edge")
    text = fasta_text(g, 60)
    files = {"bgzf": (bgzf(text), "genome.fa.gz"), "gzip": (gzip.compress(text), "genome.fa.gz"), "text": (text, "genome.fa")}
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    products = {}
    for kind, (data, fname) in files.items():
        d = tmp_path / kind
        d.mkdir()
        path = d / fname
        path.write_bytes(data)
        tmp = d / "temp"
        code = ("import sys, frisk\ntry:\n    frisk.main(['-H', %r, '-t', %r, '--quiet', '--RIP', '--exitAfter', 'WindowKLD'])\n"
                "except SystemExit:\n    pass\nprint('torch' in sys.modules)" % (str(path), str(tmp)))
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root, timeout=600)
        assert out.returncode == 0, out.stdout[-1000:] + out.stderr[-3000:]
        if kind == "bgzf":
            assert out.stdout.strip().splitlines()[-1] == "False", "torch was imported on the BGZF path"
        products[kind] = {f.replace(fname, "G"): (tmp / f).read_bytes() for f in sorted(os.listdir(tmp))}
    assert len(products["bgzf"]) >= 2
    assert products["bgzf"] == products["text"] and products["gzip"] == products["text"]
