"""Stored backgrounds without a GPU: the reference's genome pickle <-> tables (engine.genome_kmers /
genome_kmers_tables), every refusal of a malformed pickle, the C entry points' argument refusals (made before any
device is touched), and the CLI refusing a pickle whose orders are not -m..-k before it does any device work."""
import ctypes as C
import os
import pickle
import random

import numpy as np
import pytest

from frisk_b200 import _lib, api, engine
from tests.helpers import Golden

RANGES = ["edge_default", "edge_k2_5_w1000_i250", "edge_k9_10_w2500_i2500"]      # orders 1..8, 2..5, 9..10


def _maps(case):
    g = Golden(case)
    kw = g.kwargs()
    return g, kw["kmin"], kw["kmax"], engine.genome_kmers(g.tables, kw["kmin"], kw["kmax"], g.genome_meta)


@pytest.mark.parametrize("case", RANGES)
def test_pickle_round_trip(case):
    g, kmin, kmax, maps = _maps(case)
    assert len(maps) == kmax - kmin + 4
    assert [len(d) for d in maps[:-3]] == [4 ** k for k in range(kmin, kmax + 1)]
    assert maps[-3:] == [{"totalLen": int(g.genome_meta[0])}, {"exMax": int(g.genome_meta[1])}, {"nnTotal": int(g.genome_meta[2])}]
    # the object api.genome_kmers_from_result pickles (F:363), through the pickle itself
    res = engine.HotPathResult(kmin, kmax, g.tables, tuple(int(x) for x in g.genome_meta), [], np.zeros((0, 2), np.int64),
                               np.zeros((0, 5)), np.zeros(0, np.uint32))
    assert api.genome_kmers_from_result(res) == maps
    back = pickle.loads(pickle.dumps(maps, protocol=2))
    tables, a, b, meta = engine.genome_kmers_tables(back)
    assert (a, b) == (kmin, kmax) and meta == tuple(int(x) for x in g.genome_meta)
    assert tables.dtype == np.uint64 and np.array_equal(tables, g.tables)
    assert np.array_equal(engine.genome_kmers_tables(back, kmin, kmax)[0], g.tables)


@pytest.mark.parametrize("case", RANGES)
def test_shuffled_key_order_gives_the_same_tables(case):
    """A pickle written by the reference's Python 2 frisk holds its dicts in py2 hash order: words are looked up by key."""
    g, kmin, kmax, maps = _maps(case)
    rng = random.Random(5)
    shuffled = []
    for d in maps[:-3]:
        items = list(d.items())
        rng.shuffle(items)
        shuffled.append(dict(items))
    shuffled = shuffled[::-1] + maps[-3:][::-1]          # orders and meta dicts out of place too
    assert list(shuffled[-1]) != list(maps[0])
    assert np.array_equal(engine.genome_kmers_tables(shuffled)[0], g.tables)


def _refused(maps, match, kmin=None, kmax=None):
    with pytest.raises(ValueError, match=match):
        engine.genome_kmers_tables(maps, kmin, kmax)


def test_malformed_pickles_are_refused():
    _, kmin, kmax, maps = _maps("edge_k2_5_w1000_i250")
    orders, meta = maps[:-3], maps[-3:]
    _refused(orders[:1] + orders[2:] + meta, "order 3 is missing")
    _refused(maps, "order 2 is extra", kmin=3, kmax=5)
    _refused(maps, "order 6 is missing", kmin=2, kmax=6)
    _refused(maps, "order 1 is missing", kmin=1, kmax=5)
    _refused(orders + [dict(orders[1])] + meta, "order 3 appears twice")
    short = dict(orders[2])
    short.pop(next(iter(short)))
    _refused(orders[:2] + [short] + orders[3:] + meta, "order 4 holds 255 words, not 4\\^4 = 256")
    long_ = dict(orders[0], NN=1)
    _refused([long_] + orders[1:] + meta, "order 2 holds 17 words")
    wrong = dict(orders[0])
    wrong.pop("AA")
    wrong["AN"] = 0
    _refused([wrong] + orders[1:] + meta, "order 2 lacks the word AA")
    for i, key in enumerate(("totalLen", "exMax", "nnTotal")):
        _refused(orders + meta[:i] + meta[i + 1:], "meta dict \\{'%s'\\} is missing" % key)
    _refused(meta, "no k-mer table")
    _refused([{}] + orders + meta, "empty")
    _refused({"a": 1}, "expected a list")
    _refused(orders + [("totalLen", 1)] + meta, "not a dict")


def test_python_background_refuses_before_the_device():
    g = Golden("edge_k2_5_w1000_i250")
    with pytest.raises(ValueError, match="orders 2..6 need"):
        engine.Background(g.tables, 2, 6, g.genome_meta)
    with pytest.raises(ValueError, match="orders 3..2"):
        engine.Background(g.tables, 3, 2, g.genome_meta)
    with pytest.raises(_lib.FriskError) as e:
        engine.Background(np.zeros(_lib.table_size(1, 13), np.uint64), 1, 13, (10, 0, 0))
    assert e.value.code == _lib.E_UNSUPPORTED


def test_c_entry_points_refuse_bad_arguments_before_the_device():
    L = _lib.lib()
    tables = np.zeros(_lib.table_size(1, 8), np.uint64)
    tp = C.c_void_p(tables.ctypes.data)
    h = C.c_void_p()
    assert L.frisk_b200_background_open(None, 1, 8, 1000, None, C.byref(h)) == _lib.E_INVALID
    assert L.frisk_b200_background_open(tp, 1, 8, 1000, None, None) == _lib.E_INVALID
    for space in (0, -1, -(2 ** 62)):                   # totalLen - nnTotal <= 0: where F:379-437 divides by zero
        assert L.frisk_b200_background_open(tp, 1, 8, space, None, C.byref(h)) == _lib.E_INVALID
    assert L.frisk_b200_background_open(tp, 0, 8, 1000, None, C.byref(h)) == _lib.E_INVALID
    assert L.frisk_b200_background_open(tp, 5, 4, 1000, None, C.byref(h)) == _lib.E_INVALID
    assert L.frisk_b200_background_open(tp, 1, 13, 1000, None, C.byref(h)) == _lib.E_UNSUPPORTED
    assert not h.value
    text = b">a\nACGT\n"
    rows, status, n = np.zeros((4, 5)), np.zeros(4, np.uint32), C.c_uint64(7)
    qh = C.c_void_p()
    assert L.frisk_b200_background_run(None, text, len(text), 0, 5000, 2500, 0, 1, 4, C.c_void_p(rows.ctypes.data),
                                       C.c_void_p(status.ctypes.data), C.byref(n), C.byref(qh), None) == _lib.E_INVALID
    plane = np.zeros(8, np.uint32)
    pp = C.c_void_p(plane.ctypes.data)
    off, ln = np.zeros(1, np.uint64), np.full(1, 100, np.uint32)
    assert L.frisk_b200_background_score(None, pp, pp, None, 128, C.c_void_p(off.ctypes.data), C.c_void_p(ln.ctypes.data), 1,
                                         100, 1, C.c_void_p(rows.ctypes.data), C.c_void_p(status.ctypes.data), None) == _lib.E_INVALID
    assert L.frisk_b200_background_close(None, None) == _lib.OK


def test_cli_refuses_a_pickle_of_other_orders(tmp_path, caplog):
    """The reference's cache key is the host's basename and -m / -k: a pickle that does not hold exactly those orders is an
    error naming the file, raised before the query is read or any device work is done; no TSV is written."""
    g = Golden("edge_k2_5_w1000_i250")
    temp = tmp_path / "temp"
    temp.mkdir()
    query = tmp_path / "q.fa"
    query.write_bytes(b">q\nACGT\n")
    pickle_path = temp / "host.fa_kmers_2_6_genome.p"
    with open(pickle_path, "wb") as fh:
        pickle.dump(engine.genome_kmers(g.tables, 2, 5, g.genome_meta), fh, protocol=2)
    with pytest.raises(SystemExit) as e:
        api.main(["-H", str(tmp_path / "host.fa"), "-Q", str(query), "-t", str(temp), "-m", "2", "-k", "6", "--quiet"])
    assert e.value.code == 1
    assert str(pickle_path) in caplog.text and "order 6 is missing" in caplog.text
    assert sorted(os.listdir(temp)) == [pickle_path.name]
