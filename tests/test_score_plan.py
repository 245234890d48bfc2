"""Which window kernel frisk_b200_score runs, pinned from outside the launcher.

frisk_b200_score_kernel_name makes no CUDA call, so the selection for every (kmin, kmax, longest window, forced kernel) on
the boundaries of its rules is checked on any machine against a fixed table: kmax 7 direct / nibble at 1,500 bases,
bucketed and direct rounds at 2,042 and 5,114, nibble and extension PP at 2,048 and 5,120, the shared-memory buffer at
8,186, the general kernel above 65,535.  On a GPU the first window kernel a call launches is the one that name promises,
its block is what frisk_b200_score_occupancy reports, and the one-call FASTA path honours a forced kernel like every
other entry point."""
import contextlib
import ctypes as C
import json
import re

import numpy as np
import pytest

from frisk_b200 import _lib

LENS = (500, 1000, 1500, 1501, 2042, 2043, 2048, 2049, 5000, 5114, 5115, 5120, 5121, 8186, 8187, 65535, 65536)
OPTIONS = (None, "force_dense_kernel", "force_general_kernel", "force_bucket_kernel", "force_direct_kernel",
           "force_nibble_kernel")

# (forced kernel, kmin, kmax): [(longest window up to which, kernel), ...] for the windows of LENS
EXPECTED = {
    (None, 1, 3): [(65535, "score_windows_small_kernel<3, 0>"), (65536, "gen_score_kernel")],
    (None, 1, 6): [(65535, "score_windows_small_kernel<6, 0>"), (65536, "gen_score_kernel")],
    (None, 1, 7): [
        (1500, "score_windows_direct_kernel<7, 256, 2, 0, 1>"), (2048, "score_windows_nibble_kernel<7, 8, 0, 1, 0>"),
        (5120, "score_windows_nibble_kernel<7, 20, 0, 1, 0>"), (8186, "score_windows_nibble_kernel<7, 32, 0, 1, 0>"),
        (65535, "score_windows_kernel<7>"), (65536, "gen_score_kernel")],
    (None, 1, 8): [
        (2048, "score_windows_nibble_kernel<8, 8, 0, 1, 0>"), (5120, "score_windows_nibble_kernel<8, 20, 0, 1, 0>"),
        (8186, "score_windows_nibble_kernel<8, 32, 0, 1, 0>"), (65535, "score_windows_kernel<8>"),
        (65536, "gen_score_kernel")],
    (None, 1, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    (None, 1, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    (None, 3, 3): [(65535, "score_windows_small_kernel<3, 0>"), (65536, "gen_score_kernel")],
    (None, 3, 6): [(65535, "score_windows_small_kernel<6, 0>"), (65536, "gen_score_kernel")],
    (None, 3, 7): [
        (1500, "score_windows_direct_kernel<7, 256, 2, 0, 0>"), (2048, "score_windows_nibble_kernel<7, 8, 0, 0, 0>"),
        (5120, "score_windows_nibble_kernel<7, 20, 0, 0, 0>"), (8186, "score_windows_nibble_kernel<7, 32, 0, 0, 0>"),
        (65535, "score_windows_kernel<7>"), (65536, "gen_score_kernel")],
    (None, 3, 8): [
        (2048, "score_windows_nibble_kernel<8, 8, 0, 0, 0>"), (5120, "score_windows_nibble_kernel<8, 20, 0, 0, 0>"),
        (8186, "score_windows_nibble_kernel<8, 32, 0, 0, 0>"), (65535, "score_windows_kernel<8>"),
        (65536, "gen_score_kernel")],
    (None, 3, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    (None, 3, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 1, 3): [(65535, "score_windows_kernel<3>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 1, 6): [(65535, "score_windows_kernel<6>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 1, 7): [(65535, "score_windows_kernel<7>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 1, 8): [(65535, "score_windows_kernel<8>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 1, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 1, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 3, 3): [(65535, "score_windows_kernel<3>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 3, 6): [(65535, "score_windows_kernel<6>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 3, 7): [(65535, "score_windows_kernel<7>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 3, 8): [(65535, "score_windows_kernel<8>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 3, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_dense_kernel", 3, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_general_kernel", 1, 3): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 1, 6): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 1, 7): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 1, 8): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 1, 9): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 1, 12): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 3, 3): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 3, 6): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 3, 7): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 3, 8): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 3, 9): [(65536, "gen_score_kernel")],
    ("force_general_kernel", 3, 12): [(65536, "gen_score_kernel")],
    ("force_bucket_kernel", 1, 3): [(65535, "score_windows_kernel<3>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 1, 6): [
        (2042, "score_windows_bucket_kernel<6, 2, 0, 1>"), (5114, "score_windows_bucket_kernel<6, 5, 0, 1>"),
        (8186, "score_windows_bucket_kernel<6, 8, 0, 1>"), (65535, "score_windows_kernel<6>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 1, 7): [
        (2042, "score_windows_bucket_kernel<7, 2, 0, 1>"), (5114, "score_windows_bucket_kernel<7, 5, 0, 1>"),
        (8186, "score_windows_bucket_kernel<7, 8, 0, 1>"), (65535, "score_windows_kernel<7>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 1, 8): [
        (2042, "score_windows_bucket_kernel<8, 2, 0, 1>"), (5114, "score_windows_bucket_kernel<8, 5, 0, 1>"),
        (8186, "score_windows_bucket_kernel<8, 8, 0, 1>"), (65535, "score_windows_kernel<8>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 1, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 1, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 3, 3): [(65535, "score_windows_kernel<3>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 3, 6): [
        (2042, "score_windows_bucket_kernel<6, 2, 0, 0>"), (5114, "score_windows_bucket_kernel<6, 5, 0, 0>"),
        (8186, "score_windows_bucket_kernel<6, 8, 0, 0>"), (65535, "score_windows_kernel<6>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 3, 7): [
        (2042, "score_windows_bucket_kernel<7, 2, 0, 0>"), (5114, "score_windows_bucket_kernel<7, 5, 0, 0>"),
        (8186, "score_windows_bucket_kernel<7, 8, 0, 0>"), (65535, "score_windows_kernel<7>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 3, 8): [
        (2042, "score_windows_bucket_kernel<8, 2, 0, 0>"), (5114, "score_windows_bucket_kernel<8, 5, 0, 0>"),
        (8186, "score_windows_bucket_kernel<8, 8, 0, 0>"), (65535, "score_windows_kernel<8>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 3, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_bucket_kernel", 3, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 1, 3): [(65535, "score_windows_small_kernel<3, 0>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 1, 6): [(65535, "score_windows_small_kernel<6, 0>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 1, 7): [
        (2042, "score_windows_direct_kernel<7, 256, 2, 0, 1>"), (5114, "score_windows_direct_kernel<7, 256, 5, 0, 1>"),
        (8186, "score_windows_direct_kernel<7, 256, 8, 0, 1>"), (65535, "score_windows_kernel<7>"),
        (65536, "gen_score_kernel")],
    ("force_direct_kernel", 1, 8): [
        (2042, "score_windows_direct_kernel<8, 256, 2, 0, 1>"), (5114, "score_windows_direct_kernel<8, 256, 5, 0, 1>"),
        (8186, "score_windows_direct_kernel<8, 256, 8, 0, 1>"), (65535, "score_windows_kernel<8>"),
        (65536, "gen_score_kernel")],
    ("force_direct_kernel", 1, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 1, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 3, 3): [(65535, "score_windows_small_kernel<3, 0>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 3, 6): [(65535, "score_windows_small_kernel<6, 0>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 3, 7): [
        (2042, "score_windows_direct_kernel<7, 256, 2, 0, 0>"), (5114, "score_windows_direct_kernel<7, 256, 5, 0, 0>"),
        (8186, "score_windows_direct_kernel<7, 256, 8, 0, 0>"), (65535, "score_windows_kernel<7>"),
        (65536, "gen_score_kernel")],
    ("force_direct_kernel", 3, 8): [
        (2042, "score_windows_direct_kernel<8, 256, 2, 0, 0>"), (5114, "score_windows_direct_kernel<8, 256, 5, 0, 0>"),
        (8186, "score_windows_direct_kernel<8, 256, 8, 0, 0>"), (65535, "score_windows_kernel<8>"),
        (65536, "gen_score_kernel")],
    ("force_direct_kernel", 3, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_direct_kernel", 3, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 1, 3): [(65535, "score_windows_small_kernel<3, 0>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 1, 6): [(65535, "score_windows_small_kernel<6, 0>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 1, 7): [
        (2048, "score_windows_nibble_kernel<7, 8, 0, 1, 0>"), (5120, "score_windows_nibble_kernel<7, 20, 0, 1, 0>"),
        (8186, "score_windows_nibble_kernel<7, 32, 0, 1, 0>"), (65535, "score_windows_kernel<7>"),
        (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 1, 8): [
        (2048, "score_windows_nibble_kernel<8, 8, 0, 1, 0>"), (5120, "score_windows_nibble_kernel<8, 20, 0, 1, 0>"),
        (8186, "score_windows_nibble_kernel<8, 32, 0, 1, 0>"), (65535, "score_windows_kernel<8>"),
        (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 1, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 1, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 1>"), (5120, "score_windows_nibble_ext_kernel<20, 1>"),
        (8186, "score_windows_nibble_ext_kernel<32, 1>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 3, 3): [(65535, "score_windows_small_kernel<3, 0>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 3, 6): [(65535, "score_windows_small_kernel<6, 0>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 3, 7): [
        (2048, "score_windows_nibble_kernel<7, 8, 0, 0, 0>"), (5120, "score_windows_nibble_kernel<7, 20, 0, 0, 0>"),
        (8186, "score_windows_nibble_kernel<7, 32, 0, 0, 0>"), (65535, "score_windows_kernel<7>"),
        (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 3, 8): [
        (2048, "score_windows_nibble_kernel<8, 8, 0, 0, 0>"), (5120, "score_windows_nibble_kernel<8, 20, 0, 0, 0>"),
        (8186, "score_windows_nibble_kernel<8, 32, 0, 0, 0>"), (65535, "score_windows_kernel<8>"),
        (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 3, 9): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
    ("force_nibble_kernel", 3, 12): [
        (2048, "score_windows_nibble_ext_kernel<8, 0>"), (5120, "score_windows_nibble_ext_kernel<20, 0>"),
        (8186, "score_windows_nibble_ext_kernel<32, 0>"), (65536, "gen_score_kernel")],
}


@contextlib.contextmanager
def forced(opt):
    if opt:
        _lib.check(_lib.lib().frisk_b200_set_option(opt.encode(), 1), "set_option")
    try:
        yield
    finally:
        if opt:
            _lib.lib().frisk_b200_set_option(opt.encode(), 0)


def kernel_name(kmin, kmax, max_len):
    buf = C.create_string_buffer(160)
    _lib.check(_lib.lib().frisk_b200_score_kernel_name(kmin, kmax, max_len, buf, 160), "score_kernel_name")
    return buf.value.decode()


def expected(opt, kmin, kmax, max_len):
    return next(name for last, name in EXPECTED[(opt, kmin, kmax)] if max_len <= last)


@pytest.mark.parametrize("opt", OPTIONS)
def test_kernel_name_table(opt):
    keys = [(kmin, kmax, n) for (o, kmin, kmax) in EXPECTED if o == opt for n in LENS]
    assert len(keys) == 2 * 6 * len(LENS)
    with forced(opt):
        got = {k: kernel_name(*k) for k in keys}
    assert got == {k: expected(opt, *k) for k in keys}


# ---- on the GPU -----------------------------------------------------------------------------------------------------

def _norm(name):
    """A kernel name as the profiler prints it, spelled like frisk_b200_score_kernel_name."""
    name = re.sub(r"^void |\(anonymous namespace\)::|<unnamed>::", "", name)
    return name.split("(", 1)[0].replace("true", "1").replace("false", "0")


def _window_launches(fn, tmp_path):
    """(name, block) of every window kernel fn launches, in launch order."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = str(tmp_path / "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = [e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
    ev.sort(key=lambda e: e["ts"])
    names = [(_norm(e["name"]), e["args"]["block"][0]) for e in ev]
    return [(n, b) for n, b in names if n.startswith("score_windows_") or n == "gen_score_kernel"], out


def _occupancy(kmax, max_len):
    ctas, threads = C.c_int(0), C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_score_occupancy(kmax, max_len, C.byref(ctas), C.byref(threads)), "score_occupancy")
    return ctas.value, threads.value


@pytest.fixture(scope="module")
def genome():
    from frisk_b200 import engine, synth
    _lib.require_device()
    rng = np.random.Generator(np.random.PCG64(3))
    return [("s", synth.iid_bases(rng, 200_000, 0.45))], engine


@pytest.mark.gpu
@pytest.mark.parametrize("kmin,kmax,w,opt", [
    (1, 3, 1000, None), (3, 6, 5000, None), (1, 7, 1000, None), (1, 7, 5000, None), (3, 8, 2049, None),
    (1, 8, 8187, None), (1, 9, 5000, None), (3, 12, 2048, None), (1, 8, 65536, None),
    (3, 6, 2043, "force_bucket_kernel"), (1, 8, 5000, "force_bucket_kernel"), (1, 8, 5000, "force_direct_kernel"),
    (1, 7, 1000, "force_nibble_kernel"), (1, 8, 5000, "force_dense_kernel"), (1, 8, 5000, "force_general_kernel")])
def test_launched_kernel_is_the_named_one(genome, tmp_path, kmin, kmax, w, opt):
    sc, engine = genome
    g = engine.PackedGenome.from_scaffolds(sc)
    assert g.windows(w, w).max_len == w
    with forced(opt):
        name = kernel_name(kmin, kmax, w)
        _, threads = _occupancy(kmax, w)
        launches, _ = _window_launches(lambda: engine.run(g, kmin=kmin, kmax=kmax, w=w, step=w), tmp_path)
    assert name == expected(opt, kmin, kmax, w)
    assert launches and launches[0] == (name, threads), launches


@pytest.mark.gpu
def test_occupancy_reports_the_extension_kernel(genome):
    ctas, threads = _occupancy(9, 5000)
    assert threads == 256 and ctas >= 1
    with forced("force_general_kernel"):
        assert _occupancy(8, 5000) == (1, 1024)


@pytest.mark.gpu
def test_run_fasta_honours_a_forced_general_kernel(genome, tmp_path):
    from frisk_b200 import synth
    from tests.helpers import assert_rows_close
    sc, engine = genome
    text = np.frombuffer(synth.fasta_bytes(sc), dtype=np.uint8)
    default = engine.run_fasta(text, kmax=8)
    with forced("force_general_kernel"):
        launches, res = _window_launches(lambda: engine.run_fasta(text, kmax=8), tmp_path)
    assert launches and {n for n, _ in launches} == {"gen_score_kernel"}, launches
    assert np.array_equal(res.status, default.status)
    assert_rows_close(res.rows, default.rows, rtol_kld=1e-12, rtol_other=1e-12, what="run_fasta, general kernel")
