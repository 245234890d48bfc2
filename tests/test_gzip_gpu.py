"""Plain gzip on the device: the chunked speculative inflate (frisk_b200_gzip_inflate) byte for byte against zlib with the
host run's stats, malformed input refused without a CUDA error, the gzip open (frisk_b200_fasta_open_gzip) against the
text open, the one-call path (frisk_b200_run_fasta_gzip) against frisk_b200_run_fasta, and the CLI on a gzip and a
multi-member file."""
import ctypes as C
import os

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from tests.helpers import Golden
from tests.test_bgzf_gpu import _same_result
from tests.test_gzip_host import CASES, chunk_bytes, corpus_case, dna, gz_member, inflate_host, set_chunk  # noqa: F401
from tests.test_ingest_gpu import _assert_same, fasta_text, ingest_options

pytestmark = pytest.mark.gpu


def inflate_device(gz: bytes, cap: int | None = None):
    """(rc, text, stats + [text_len]) of frisk_b200_gzip_inflate."""
    import torch
    dev = torch.device("cuda:0")
    d_gz = torch.from_numpy(np.frombuffer(gz, np.uint8).copy() if gz else np.zeros(1, np.uint8)).to(dev)
    if cap is None:
        cap = inflate_host(gz)[2][4] if gz else 0
    d_text = torch.zeros(max(cap, 1), dtype=torch.uint8, device=dev)
    tl = C.c_uint64(0)
    st = np.zeros(4, np.uint64)
    with torch.cuda.device(dev):
        rc = _lib.lib().frisk_b200_gzip_inflate(engine._ptr(d_gz), len(gz), engine._ptr(d_text), cap, C.byref(tl), engine._ptr(st),
                                                engine._stream_ptr(dev))
        torch.cuda.synchronize()
    n = min(int(tl.value), cap)
    return rc, d_text[:n].cpu().numpy().tobytes(), list(map(int, st)) + [int(tl.value)]


@pytest.mark.parametrize("case", CASES)
def test_device_inflate_equals_zlib_and_host(case):
    gz, want = corpus_case(case)
    for chunk in (0, 1024):
        set_chunk(chunk)
        try:
            rc, got, st = inflate_device(gz)
            hrc, _, hst = inflate_host(gz)
        finally:
            set_chunk(0)
        assert rc == _lib.OK and got == want, chunk
        assert hrc == _lib.OK and st == hst, (chunk, st, hst)


def test_device_inflate_c2_scale():
    text = synth.fasta_bytes(synth.config_c2(scale=0.25))
    for level in (1, 6, 9):
        gz = gz_member(text, level=level)
        rc, got, st = inflate_device(gz)
        assert rc == _lib.OK and got == text
        assert st == inflate_host(gz)[2]
        assert st[1] >= 0.95 * (st[0] - 1)


def test_device_inflate_refuses_malformed_input():
    """Each refusal leaves no CUDA error behind, and the next valid call succeeds."""
    import torch
    data = dna(0.002)
    good = gz_member(data)
    bad_crc = bytearray(good); bad_crc[-8] ^= 1
    bad_isize = bytearray(good); bad_isize[-4] ^= 1
    cases = {
        "truncated": (good[:len(good) // 2], _lib.E_FORMAT),
        "bad_crc": (bytes(bad_crc), _lib.E_FORMAT),
        "bad_isize": (bytes(bad_isize), _lib.E_FORMAT),
        "trailing_garbage": (good + b"junk", _lib.E_FORMAT),
        "multi_member": (good + gz_member(b">b\nAC\n"), _lib.E_UNSUPPORTED),
        "not_gzip": (b"PK\x03\x04" + b"\0" * 40, _lib.E_FORMAT),
    }
    for name, (gz, code) in cases.items():
        rc, _, _ = inflate_device(gz, cap=len(data) + 4096)
        assert rc == code, name
        torch.cuda.synchronize()                                      # (raises if the refusal left a CUDA error)
        rc, got, _ = inflate_device(good)
        assert rc == _lib.OK and got == data, name
    rc, _, st = inflate_device(good, cap=10)
    assert rc == _lib.E_CAPACITY and st[4] == len(data)


# ---- the gzip open against the text open ---------------------------------------------------------------------------------
def _open_inputs():
    rng = np.random.default_rng(11)
    text = fasta_text(synth.make("C2", 0.01, seed=4), 60)
    long_header = (b">" + b"h" * 70_000 + b" tail\n" + b"ACGT" * 30_000 + b"\n>second\n" +
                   np.frombuffer(b"ACGTacgtN", np.uint8)[rng.integers(0, 9, 100_000)].tobytes() + b"\n")
    return {"c2_level6": gz_member(text), "c2_level1_flags": gz_member(text, level=1, flags=31, extra=b"AB\x01\0q"),
            "header_over_64k": gz_member(long_header)}, {"c2_level6": text, "c2_level1_flags": text, "header_over_64k": long_header}


@pytest.mark.parametrize("case", ["c2_level6", "c2_level1_flags", "header_over_64k"])
def test_fasta_open_gzip_equals_text_open(case):
    gzs, texts = _open_inputs()
    gz, text = gzs[case], texts[case]
    host = engine.PackedGenome.from_fasta_bytes(text)
    for mode in ("default", "chunk1", "exact"):
        with ingest_options(mode):
            dev = engine.DeviceGenome.from_gzip_bytes(gz)
            ref = engine.DeviceGenome.from_fasta_bytes(text)
        _assert_same(dev.to_host(), host)
        assert list(dev.host.names) == list(ref.host.names)
    nat = engine.DeviceGenome.from_gzip_bytes_native(gz)
    assert list(nat.host.names) == list(host.names) and np.array_equal(nat.host.scaf_len, host.scaf_len)


def test_fasta_open_gzip_empty_and_refused():
    for mode in ("default", "exact"):
        with ingest_options(mode):
            _assert_same(engine.DeviceGenome.from_gzip_bytes(gz_member(b"")).to_host(), engine.PackedGenome.from_fasta_bytes(b""))
            with pytest.raises(_lib.FriskError) as ei:
                engine.DeviceGenome.from_gzip_bytes(gz_member(b">ok\nACGT\n>\nACGT\n"))
            assert ei.value.code == _lib.E_FORMAT
    good = gz_member(b">a\nACGT\n" * 1000)
    with pytest.raises(_lib.FriskError) as ei:
        engine.DeviceGenome.from_gzip_bytes(good[:-8] + b"\0" * 8)
    assert ei.value.code == _lib.E_FORMAT
    with pytest.raises(_lib.FriskError) as ei:
        engine.DeviceGenome.from_gzip_bytes(good + good)
    assert ei.value.code == _lib.E_UNSUPPORTED


def test_from_fasta_routes_gzip_and_falls_back_for_multi_member(tmp_path):
    text = fasta_text(synth.make("C2", 0.005, seed=6), 60)
    host = engine.PackedGenome.from_fasta_bytes(text)
    half = text.index(b">", len(text) // 2)
    for name, data in (("one.fa.gz", gz_member(text)), ("two.fa.gz", gz_member(text[:half]) + gz_member(text[half:]))):
        p = tmp_path / name
        p.write_bytes(data)
        _assert_same(engine.DeviceGenome.from_fasta(str(p)).to_host(), host)


# ---- the one-call path ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(kmax=8), dict(kmax=6), dict(kmax=9, w=2000, step=1000), dict(kmax=8, scaffolds_all=True)],
                         ids=["k8_device_tail", "k6_host_tail", "k9_host_tail", "scaffolds_all"])
def test_run_fasta_gzip_equals_run_fasta(kw, chunk_bytes):
    text = fasta_text(synth.make("C2", 0.02, seed=8) + synth.make("edge"), 60)
    gz = gz_member(text)
    want = engine.run_fasta(text, **kw)
    for mode in ("default", "chunk1", "exact"):
        with ingest_options(mode):
            _same_result(engine.run_fasta_gzip(gz, **kw), want, mode)
    chunk_bytes(2048)
    _same_result(engine.run_fasta_gzip(gz, **kw), want, "gzip chunks of 2 KiB")
    chunk_bytes(0)
    small = engine.HostOutputs(1, kw["kmax"])                           # FRISK_E_CAPACITY, second stage on the handles
    _same_result(engine.run_fasta_gzip(gz, out=small, **kw), want, "capacity")


def test_run_fasta_gzip_mask_host_and_golden():
    gold = Golden("edge_maskHost")
    host = gold.host()
    qtext, htext = fasta_text(gold.scaffolds()), fasta_text(host) if host is not None else fasta_text(gold.scaffolds()[::-1])
    want = engine.run_fasta(qtext, htext, **gold.kwargs())
    _same_result(engine.run_fasta_gzip(gz_member(qtext), gz_member(htext, level=9), **gold.kwargs()), want, "maskHost")
    from tests.test_gpu_parity import _check_against_golden
    gold = Golden("edge_scaffoldsAll")
    res = engine.run_fasta_gzip(gz_member(fasta_text(gold.scaffolds())), **gold.kwargs())
    _check_against_golden(res, gold, "edge_scaffoldsAll[run_fasta_gzip]")


def test_run_fasta_gzip_timing_mark():
    text = fasta_text(synth.make("C2", 0.02, seed=3), 60)
    engine.run_fasta_gzip(gz_member(text))
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    assert 0.0 < ms[0] <= ms[4]                                       # compressed bytes uploaded and inflated, then the rest


# ---- CLI ----------------------------------------------------------------------------------------------------------------------
def test_cli_gzip_and_multi_member_give_text_products(tmp_path):
    import subprocess
    import sys
    text = fasta_text(synth.make("C2", 0.01, seed=21) + synth.make("edge"), 60)
    half = text.index(b">", len(text) // 2)
    files = {"gzip": (gz_member(text), "genome.fa.gz"), "multi": (gz_member(text[:half]) + gz_member(text[half:]), "genome.fa.gz"),
             "text": (text, "genome.fa")}
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    products = {}
    for kind, (data, fname) in files.items():
        d = tmp_path / kind
        d.mkdir()
        path = d / fname
        path.write_bytes(data)
        tmp = d / "temp"
        code = ("import sys, frisk\nfrom frisk_b200 import engine\ncalls = []\nopen_native = engine.DeviceGenome._open_native\n"
                "def spy(cls, buf, device, kind):\n    calls.append(kind)\n    return open_native.__func__(cls, buf, device, kind)\n"
                "engine.DeviceGenome._open_native = classmethod(spy)\n"
                "try:\n    frisk.main(['-H', %r, '-t', %r, '--quiet', '--RIP', '--exitAfter', 'WindowKLD'])\n"
                "except SystemExit:\n    pass\nprint(calls)\nprint('torch' in sys.modules)" % (str(path), str(tmp)))
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root, timeout=600)
        assert out.returncode == 0, out.stdout[-1000:] + out.stderr[-3000:]
        lines = out.stdout.strip().splitlines()
        assert lines[-1] == "False", "torch was imported on the %s path" % kind
        assert lines[-2] == {"gzip": "['gzip']", "multi": "['gzip', 'text']", "text": "['text']"}[kind], lines[-2]
        products[kind] = {f.replace(fname, "G"): (tmp / f).read_bytes() for f in sorted(os.listdir(tmp))}
    assert len(products["gzip"]) >= 2
    assert products["gzip"] == products["text"] and products["multi"] == products["text"]
