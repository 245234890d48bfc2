"""The nibble kernel's pair gather (frisk_nibble.cu, P3): positions p and p + 1 take their genome-IVOM entries from one
32-byte entry of the (K+1)-mer pair table.  The cases where only one of the two positions holds a full K-word are the
ones this path has to get right: an N at every offset mod 4, runs of N ending at both parities, window lengths of
every residue mod 4 (the last chunk partly past the window end), kmax 7 and 8, kmin 1 and > 1, and NaN genome-IVOM
entries (query k-mers the host lacks).  Checked against the C oracle (tables, status, rows, every window's tables), the
bucketed kernel (which reads the plain genome-IVOM table) and a second run."""
import numpy as np
import pytest

from tests.helpers import assert_rows_close, max_rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from frisk_b200 import _lib, engine
    _lib.require_device()          # fail loudly: no CPU fallback exists
    return engine


def _scaffolds():
    """Single Ns every 379 bases (379 = 3 mod 4: every offset mod 4 in turn) and runs of 2..5 Ns.  At most 54 words cut
    at K-1 / K-2 bases per window, below the nibble kernel's hand-over limit of 64: every window takes the pair path."""
    from frisk_b200 import synth
    rng = np.random.Generator(np.random.PCG64(4711))
    out = []
    for i, n in enumerate((23_001, 17_002, 12_003)):
        a = synth.iid_bases(rng, n, 0.42 + 0.04 * i)
        for p in range(300 + 37 * i, n - 10, 379):
            a[p] = ord("N")
        for j, p in enumerate(range(1_000 + 5 * i, n - 10, 1_733)):
            a[p:p + 2 + j % 4] = ord("N")
        out.append(("pairs%d" % i, a))
    return out


def _host():
    from frisk_b200 import synth
    rng = np.random.Generator(np.random.PCG64(99))
    return [("host", synth.iid_bases(rng, 16_000, 0.5))]      # lacks a few 6-mers: at kmin 6, NaN entries for their 8-mers


def _with_option(opt, fn):
    from frisk_b200 import _lib
    _lib.check(_lib.lib().frisk_b200_set_option(opt, 1), "set_option")
    try:
        return fn()
    finally:
        _lib.lib().frisk_b200_set_option(opt, 0)


@pytest.mark.parametrize("kw", [
    dict(kmax=8),
    dict(kmax=7),
    dict(kmax=8, kmin=3, w=2001, step=1000, scaffolds_all=True),
    dict(kmax=7, kmin=2, w=5003, step=2500, scaffolds_all=True),
    dict(kmax=8, w=8002, step=4001, scaffolds_all=True),
    dict(kmax=7, kmin=6, w=1002, step=500, scaffolds_all=True),
    dict(kmax=8, kmin=6, w=1002, step=500, host=True),
])
def test_nibble_pair_gather_against_c_oracle(eng, kw):
    from oracle import c_oracle
    sc = _scaffolds()
    kw = dict(kw)
    host = _host() if kw.pop("host", False) else None
    full = dict(kmin=1, kmax=8, w=5000, step=2500, mask_host=False, scaffolds_all=False, rip=True)
    full.update(kw)
    ref = c_oracle.run(sc, host=host, threads=8, **full)
    q = eng.PackedGenome.from_scaffolds(sc)
    h = eng.PackedGenome.from_scaffolds(host) if host is not None else None
    run = lambda **k: _with_option(b"force_nibble_kernel", lambda: eng.run(q, h, **k, **full))
    res = run(dump=True)
    assert np.array_equal(res.tables, ref["tables"])
    assert np.array_equal(res.coords, ref["coords"])
    assert np.array_equal(res.status & 7, ref["status"] & 7)
    assert not np.any(res.status & 0x80000000), "internal redo marker must not survive"
    if host is not None:
        assert np.any(res.status & 1) and np.any(res.status == 0), "NaN genome-IVOM entries in some windows, not all"
    ok = ref["status"] == 0
    assert_rows_close(res.rows[ok], ref["rows"][ok], rtol_kld=1e-6, rtol_other=1e-15, what=str(kw))
    assert max_rel_err(res.rows[ok, 0], ref["rows"][ok, 0]) < 1e-10
    seq, _ = c_oracle.concat(sc)
    for i in range(len(ref["rows"])):
        if ref["status"][i] & 8:
            continue
        win = seq[int(ref["win_off"][i]):int(ref["win_off"][i]) + int(ref["win_len"][i])]
        _, _, wt, _ = c_oracle.window_tables(win, ref["tables"], ref["meta"], full["kmin"], full["kmax"])
        assert np.array_equal(res.win_tables[i].astype(np.uint64), wt), (kw, i)
    # the production instantiation (no dump) gives the same rows, bit for bit, twice
    a, b = run(), run()
    assert np.array_equal(a.rows, res.rows, equal_nan=True) and np.array_equal(a.status, res.status)
    assert np.array_equal(a.rows, b.rows, equal_nan=True) and np.array_equal(a.status, b.status)
    # the bucketed kernel reads the plain genome-IVOM table: same integers, another summation order
    other = _with_option(b"force_bucket_kernel", lambda: eng.run(q, h, dump=True, **full))
    assert np.array_equal(other.win_tables, res.win_tables)
    assert np.array_equal(other.status, res.status)
    assert np.array_equal(np.isnan(other.rows), np.isnan(res.rows))
    assert max_rel_err(other.rows[ok, 0], res.rows[ok, 0]) < 1e-12
    assert np.array_equal(other.rows[:, 1:], res.rows[:, 1:], equal_nan=True)
