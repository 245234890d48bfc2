"""UCSC .2bit on the device: the open (frisk_b200_fasta_open_2bit) against the text open of the same genome's FASTA, the
one-call path (frisk_b200_run_2bit) against frisk_b200_run_fasta bit for bit, the reference's goldens, mixed formats, the
CLI, the device-only tail, C4-size and > 2^32-base genomes, and malformed files."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from frisk_b200 import _lib, engine, synth
from tests.helpers import SMALL_CASES, Golden
from tests.test_bgzf_gpu import _same_result
from tests.test_ingest_gpu import _assert_same, fasta_text
from tests.test_twobit_host import FIXTURE, corpus

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pinned(data: bytes) -> np.ndarray:
    a = engine._alloc(len(data), np.uint8, True)
    a[:] = np.frombuffer(data, np.uint8)
    return a


# ---- the open against the text open ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["corpus", "corpus_be_v1", "c2_full", "c5_small"])
def test_fasta_open_2bit_equals_text_open(case):
    sc = {"corpus": corpus, "corpus_be_v1": corpus, "c2_full": lambda: synth.make("C2", 1.0),
          "c5_small": lambda: synth.make("C5", 2e-5, seed=3) + synth.make("edge")}[case]()
    buf = synth.twobit_bytes(sc, big_endian=case.endswith("be_v1"), version=1 if case.endswith("v1") else 0)
    text = fasta_text(sc)
    dev = engine.DeviceGenome.from_2bit_bytes(buf)
    ref = engine.DeviceGenome.from_fasta_bytes(text)
    _assert_same(dev.to_host(), ref.to_host())
    _assert_same(dev.to_host(), engine.PackedGenome.from_2bit_bytes(buf))
    nat = engine.DeviceGenome.from_2bit_bytes_native(buf)
    assert list(nat.host.names) == list(ref.host.names) and np.array_equal(nat.host.scaf_len, ref.host.scaf_len)
    assert (nat.host.nn_total, nat.host.n_lower) == (ref.host.nn_total, ref.host.n_lower)


def test_fasta_open_2bit_fixture_and_empty_file():
    _assert_same(engine.DeviceGenome.from_2bit_bytes(FIXTURE).to_host(), engine.PackedGenome.from_fasta_bytes(b">s\nTCAGNNac\n"))
    empty = synth.twobit_bytes([])
    _assert_same(engine.DeviceGenome.from_2bit_bytes(empty).to_host(), engine.PackedGenome.from_fasta_bytes(b""))


# ---- the one-call path -----------------------------------------------------------------------------------------------------
def _genome():
    return synth.make("C2", 0.02, seed=8) + synth.make("edge") + synth.make("edge_short")


@pytest.mark.parametrize("kw", [dict(kmax=8), dict(kmax=7), dict(kmax=6), dict(kmax=4), dict(kmax=9, w=2000, step=1000),
                                dict(kmax=12, w=2000, step=1000), dict(kmax=8, w=1000, step=800),
                                dict(kmax=8, scaffolds_all=True), dict(kmax=8, mask_host=True), dict(kmax=6, rip=False),
                                dict(kmin=2, kmax=8, w=1000, step=800, scaffolds_all=True)],
                         ids=["k8", "k7", "k6", "k4", "k9", "k12", "k8_w1000_i800", "scaffolds_all", "mask_host", "k6_norip",
                              "k2_8_w1000_all"])
def test_run_2bit_equals_run_fasta(kw):
    sc = _genome()
    text, buf = fasta_text(sc), synth.twobit_bytes(sc)
    want = engine.run_fasta(text, **kw)
    _same_result(engine.run_2bit(buf, **kw), want, "pageable")
    _same_result(engine.run_2bit(_pinned(buf), **kw), want, "pinned")
    small = engine.HostOutputs(1, kw["kmax"])                          # FRISK_E_CAPACITY, second stage on the handles
    _same_result(engine.run_2bit(buf, out=small, **kw), want, "capacity")


@pytest.mark.parametrize("kmax", [8, 6])
def test_run_2bit_query_vs_host(kmax):
    q, h = synth.make("C2", 0.01, seed=4) + synth.make("edge"), synth.make("C1", 0.02, seed=9)
    want = engine.run_fasta(fasta_text(q), fasta_text(h), kmax=kmax, mask_host=True)
    got = engine.run_2bit(_pinned(synth.twobit_bytes(q)), synth.twobit_bytes(h, big_endian=True), kmax=kmax, mask_host=True)
    _same_result(got, want, "query != host")


@pytest.mark.parametrize("case", [c for c in SMALL_CASES if c.startswith(("edge_", "short_")) or c == "c2_small"])
def test_run_2bit_against_reference_golden(case):
    from tests.test_gpu_parity import _check_against_golden
    g = Golden(case)
    host = g.host()
    res = engine.run_2bit(synth.twobit_bytes(g.scaffolds()), synth.twobit_bytes(host) if host is not None else None, **g.kwargs())
    _check_against_golden(res, g, case + "[run_2bit]")


def test_run_2bit_timing_mark():
    engine.run_2bit(synth.twobit_bytes(synth.make("C2", 0.02, seed=3)))
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    assert 0.0 < ms[0] <= ms[4]                                       # file uploaded and decoded, then the rest


def _trace(kmax: int) -> str:
    """FRISK_RUN_TRACE's host timeline of one run_2bit call in a process of its own."""
    code = ("from frisk_b200 import engine, synth\nsc = synth.make('C2', 0.01, seed=5)\n"
            "engine.run_2bit(synth.twobit_bytes(sc), kmax=%d)\n" % kmax)
    env = dict(os.environ, FRISK_RUN_TRACE="1")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stderr.splitlines() if ln.startswith("host trace")]
    assert lines, out.stderr[-2000:]
    return lines[-1]


def test_kmax8_takes_the_device_only_tail():
    """With kmax 8 everything behind the decode is queued from inside the open (no host-side tables / window steps in the
    trace); kmax 6 goes through the host tail."""
    t8, t6 = _trace(8), _trace(6)
    assert "open_returned" in t8 and "finalize_queued" not in t8 and "windows" not in t8, t8
    assert "finalize_queued" in t6 and "score_queued" in t6, t6


# ---- mixed formats and the CLI -------------------------------------------------------------------------------------------------
def test_score_genome_mixed_formats(tmp_path):
    import frisk
    from frisk_b200 import api
    q, h = synth.make("C2", 0.01, seed=14) + synth.make("edge"), synth.make("C2", 0.01, seed=15)
    files = {}
    for tag, sc in (("q", q), ("h", h)):
        files[tag + ".fa"] = tmp_path / (tag + ".fa")
        files[tag + ".fa"].write_bytes(fasta_text(sc))
        files[tag + ".2bit"] = tmp_path / (tag + ".2bit")
        files[tag + ".2bit"].write_bytes(synth.twobit_bytes(sc))

    def score(hf, qf):
        return api.score_genome(frisk.mainArgs(["-H", str(files[hf]), "-Q", str(files[qf]), "--RIP"]))

    want = score("h.fa", "q.fa")
    _same_result(score("h.fa", "q.2bit"), want, "host FASTA, query .2bit")
    _same_result(score("h.2bit", "q.fa"), want, "host .2bit, query FASTA")
    _same_result(score("h.2bit", "q.2bit"), want, "both .2bit")


def test_cli_2bit_gives_the_fasta_products(tmp_path):
    sc = synth.make("C2", 0.01, seed=21) + synth.make("edge")
    files = {"2bit": (synth.twobit_bytes(sc), "genome.2bit"), "text": (fasta_text(sc), "genome.fa")}
    products = {}
    for kind, (data, fname) in files.items():
        d = tmp_path / kind
        d.mkdir()
        path = d / fname
        path.write_bytes(data)
        tmp = d / "temp"
        code = ("import sys, frisk\ntry:\n    frisk.main(['-H', %r, '-t', %r, '--quiet', '--RIP', '--exitAfter', 'WindowKLD'])\n"
                "except SystemExit:\n    pass\nprint('torch' in sys.modules)" % (str(path), str(tmp)))
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=600)
        assert out.returncode == 0, out.stdout[-1000:] + out.stderr[-3000:]
        assert out.stdout.strip().splitlines()[-1] == "False", "torch was imported on the %s path" % kind
        products[kind] = {f.replace(fname, "G"): (tmp / f).read_bytes() for f in sorted(os.listdir(tmp))}
    assert len(products["2bit"]) >= 2
    assert products["2bit"] == products["text"]


# ---- full size -----------------------------------------------------------------------------------------------------------------
def planes_to_2bit(dg, runs) -> bytes:
    """A device genome (synth_device) as .2bit bytes, built on the device: the code planes remapped to T,C,A,G = 0..3 and
    byte-reversed into the file's base order, one N block per run."""
    import torch
    g = dg.host
    b = dg.codes.view(torch.uint8).view(-1, 4).flip(1).reshape(-1)
    b = ((~b & 0x55) << 1) | ((b >> 1) & 0x55)
    run_s, run_o, run_l = (np.asarray(x, np.int64) for x in runs)
    R = len(g.names)
    heads = []
    for r in range(R):
        sel = run_s == r
        st, sz = run_o[sel].astype(np.uint32), run_l[sel].astype(np.uint32)
        heads.append(np.array([int(g.scaf_len[r]), len(st)], np.uint32).tobytes() + st.tobytes() + sz.tobytes() +
                     np.array([0, 0], np.uint32).tobytes())
    idx_len = sum(1 + len(nm) + 4 for nm in g.names)
    off, index, parts = 16 + idx_len, [], []
    for r in range(R):
        index.append(bytes([len(g.names[r])]) + g.names[r].encode() + np.array([off], np.uint32).tobytes())
        nbytes = (int(g.scaf_len[r]) + 3) // 4
        off += len(heads[r]) + nbytes
    assert off < 2 ** 32                                               # version 0 covers it
    out = np.empty(off, np.uint8)
    head = np.array([0x1A412743, 0, R, 0], np.uint32).tobytes() + b"".join(index)
    out[:len(head)] = np.frombuffer(head, np.uint8)
    at = len(head)
    for r in range(R):
        out[at:at + len(heads[r])] = np.frombuffer(heads[r], np.uint8)
        at += len(heads[r])
        a, nbytes = int(g.scaf_off[r]) // 4, (int(g.scaf_len[r]) + 3) // 4
        out[at:at + nbytes] = b[a:a + nbytes].cpu().numpy()
        at += nbytes
    return out


def _full_size(lens, runs, seed):
    import torch
    from frisk_b200.synth_device import build_device_genome
    dg = build_device_genome(engine, lens, runs, seed=seed)
    buf = planes_to_2bit(dg, runs)
    opened = engine.DeviceGenome.from_2bit_bytes(buf)
    g, o = dg.host, opened.host
    assert np.array_equal(o.scaf_len, g.scaf_len) and np.array_equal(o.scaf_off, g.scaf_off) and o.padded_len == g.padded_len
    assert (o.total_len, o.nn_total, o.n_lower) == (g.total_len, g.nn_total, 0) and opened.low is None
    assert torch.equal(opened.codes, dg.codes) and torch.equal(opened.inv, dg.inv)
    del opened
    want = engine.run_resident(dg)                                    # rows of the same genome's planes
    got = engine.run_2bit(buf)
    _same_result(got, want, "run_2bit vs the planes")
    del dg
    torch.cuda.empty_cache()
    return g


def test_c4_size_long_n_runs():
    """3 Gbp in 26 scaffolds with one 3 Mbp N run per long scaffold: the runs go through the run expansion (94 K items each)."""
    from frisk_b200.synth_device import c4_spec
    lens, runs = c4_spec()
    g = _full_size(lens, runs, seed=44)
    assert g.total_len > 2.9e9


def test_genome_beyond_2_pow_32_bases():
    """4.4 Gbp: plane offsets pass 2^32 bases (and the file stays below 4 GiB, so version 0 covers it)."""
    lens = np.array([170_000_000] * 26 + [1_000_003, 77], np.int64)
    runs = (list(range(26)) + [26], [int(x) // 2 for x in lens[:26]] + [1000], [3_000_000] * 26 + [5000])
    g = _full_size(lens, runs, seed=45)
    assert g.padded_len > 2 ** 32


# ---- malformed files -------------------------------------------------------------------------------------------------------------
def test_malformed_files_are_refused_and_leave_no_cuda_error():
    import torch
    from tests.test_twobit_host import build
    good = synth.twobit_bytes(synth.make("C2", 0.002, seed=2))
    bad = {"signature": b"\0\0\0\0" + good[4:], "version_2": good[:4] + b"\x02\0\0\0" + good[8:], "truncated": good[:len(good) // 2],
           "empty_name": build([(b"", 4, [], [], b"\x1b")]), "block_past_size": build([(b"s", 8, [(4, 5)], [], b"\x1b\x09")]),
           "offset_past_end": build([(b"s", 8, [], [], b"\x1b\x09")])[:18] + b"\xff\xff\0\0" + b"\0" * 40}
    want = engine.run_fasta(fasta_text(synth.make("C2", 0.002, seed=2)))
    for name, buf in bad.items():
        for call in (lambda: engine.DeviceGenome.from_2bit_bytes(buf), lambda: engine.DeviceGenome.from_2bit_bytes_native(buf),
                     lambda: engine.run_2bit(buf), lambda: engine.run_2bit(good, buf)):
            with pytest.raises(_lib.FriskError) as ei:
                call()
            assert ei.value.code == _lib.E_FORMAT, name
            torch.cuda.synchronize()                                  # (raises if the refusal left a CUDA error)
        _same_result(engine.run_2bit(good), want, name)
