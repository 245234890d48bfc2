"""A query scored against a stored background against the same query scored with the host counted, on one GPU, seeded
inputs generated in the run:

  host     the C4 stand-in of synth_device (3 Gbp), as 60-column FASTA text and as .2bit, page-locked
  queries  synth.config_c2() (40 Mbp) and synth.config_c1(), in the host's format
  arms     engine.run_fasta(query, host) (engine.run_2bit for .2bit) against engine.Background.run(query), the background
           opened once from the counted run's tables, outside the timed calls; median of --reps calls each, alternating,
           every path warmed up first, rows compared bit for bit, stage marks (frisk_b200_last_run_timing) of both
  cli      wall clock of `python -m frisk -H c4.fa -Q c2.fa` in a fresh process, without the genome pickle (the host is
           read and counted, the pickle written) and with it (the host file is not opened), --cli-reps runs each,
           alternating; the products of the two compared byte for byte

The card's name and power limit come from the same run.  Writes one JSON file (--out).

    python tools/background_timing.py --out profiles/r07_background_timing.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from frisk_b200 import _lib, engine, synth  # noqa: E402
from bgzf_timing import device_info, pinned  # noqa: E402

LEGEND = ["query uploaded", "host counted (-1: background)", "tables + IVOM (-1: background)", "window kernel done",
          "rows on the host", "window kernel could start"]


def marks() -> list:
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    return list(ms)[:n.value]


def same(a, b) -> bool:
    return bool(np.array_equal(a.rows, b.rows, equal_nan=True) and np.array_equal(a.status, b.status) and
                np.array_equal(a.tables, b.tables) and list(a.names) == list(b.names) and np.array_equal(a.coords, b.coords) and
                tuple(a.meta) == tuple(b.meta))


def pair(kind: str, host: np.ndarray, query: np.ndarray, reps: int) -> dict:
    counted = engine.run_2bit if kind == "2bit" else engine.run_fasta
    want = counted(query, host)
    bg = engine.Background.from_result(want)
    res = {"windows": int(want.n_candidates), "rows_identical": same(bg.run(query, kind=kind), want)}
    out_c, out_b = engine.HostOutputs(want.n_candidates + 64, 8), engine.HostOutputs(want.n_candidates + 64, 0)
    paths = {"counted": lambda: counted(query, host, out=out_c, assemble_result=False),
             "background": lambda: bg.run(query, kind=kind, out=out_b, assemble_result=False)}
    for _ in range(2):
        for f in paths.values():
            f()
    times = {k: [] for k in paths}
    mk = {k: [] for k in paths}
    for _ in range(reps):
        for k, f in paths.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
            mk[k].append(marks())
    n = want.n_candidates
    res["raw_rows_identical"] = bool(np.array_equal(out_c.rows[:n], out_b.rows[:n], equal_nan=True) and
                                     np.array_equal(out_c.status[:n], out_b.status[:n]))
    bg.close()
    res["call_ms"] = {k: {"median": float(np.median(v)), "min": float(min(v)), "all": v} for k, v in times.items()}
    res["stage_marks_ms"] = {"legend": LEGEND, **{k: [float(np.median([m[j] for m in v])) for j in range(len(v[0]))]
                                                  for k, v in mk.items()}}
    res["counted_over_background"] = res["call_ms"]["counted"]["median"] / res["call_ms"]["background"]["median"]
    return res


def cli(host_path: str, query_path: str, reps: int, work: str) -> dict:
    """`python -m frisk -H host -Q query` without and with the genome pickle, each in a process of its own."""
    def run(temp):
        t0 = time.perf_counter()
        r = subprocess.run([sys.executable, "-m", "frisk", "-H", host_path, "-Q", query_path, "-t", temp, "--quiet", "--RIP"],
                           capture_output=True, text=True, cwd=ROOT)
        dt = time.perf_counter() - t0
        if r.returncode != 0:
            raise RuntimeError(r.stderr[-3000:])
        return dt
    cached = os.path.join(work, "cached")
    run(cached)                                                  # writes the genome pickle (and warms the file cache)
    windows = [f for f in os.listdir(cached) if "_KLD_window_" in f]
    times = {"without_pickle": [], "with_pickle": []}
    products = {}
    for i in range(reps):
        fresh = os.path.join(work, "fresh%d" % i)
        times["without_pickle"].append(run(fresh))
        for f in windows:
            os.remove(os.path.join(cached, f))                   # the windows are computed again, against the pickle
        times["with_pickle"].append(run(cached))
        products = {f: open(os.path.join(fresh, f), "rb").read() == open(os.path.join(cached, f), "rb").read()
                    for f in sorted(os.listdir(fresh))}
        shutil.rmtree(fresh)
    return {"wall_s": {k: {"median": float(np.median(v)), "all": v} for k, v in times.items()},
            "products_identical": products}


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--cli-reps", type=int, default=3)
    ap.add_argument("--skip-cli", action="store_true")
    a = ap.parse_args(argv)
    import torch
    from frisk_b200.synth_device import build_device_genome, c4_spec
    from test_twobit_gpu import planes_to_2bit
    from twobit_timing import device_fasta
    _lib.require_device()
    res = {"info": device_info()}
    lens, runs = c4_spec()
    dg = build_device_genome(engine, lens, runs, seed=44, at_rich_block=300_000 // 16)
    host = {"2bit": planes_to_2bit(dg, runs), "text": device_fasta(dg)}
    del dg
    torch.cuda.empty_cache()
    res["host"] = {"genome": "C4 stand-in", "bases": int(np.sum(lens)), "bytes": {k: int(v.shape[0]) for k, v in host.items()}}
    host = {k: pinned(v.tobytes()) for k, v in host.items()}
    queries = {"c2": synth.config_c2(), "c1": synth.config_c1()}
    for qname, sc in queries.items():
        q = {"text": pinned(synth.fasta_bytes(sc)), "2bit": pinned(synth.twobit_bytes(sc))}
        for kind in ("text", "2bit"):
            key = "%s_%s" % (qname, kind)
            res[key] = {"query_bytes": int(q[kind].shape[0]), **pair(kind, host[kind], q[kind], a.reps)}
            r = res[key]
            print(key, "rows identical:", r["rows_identical"], r["raw_rows_identical"], "median ms:",
                  {p: round(v["median"], 3) for p, v in r["call_ms"].items()}, "marks:", r["stage_marks_ms"], flush=True)
    if not a.skip_cli:
        work = tempfile.mkdtemp(prefix="frisk_bg_")
        try:
            hp, qp = os.path.join(work, "c4.fa"), os.path.join(work, "c2.fa")
            host["text"].tofile(hp)
            synth.write_fasta(queries["c2"], qp)
            del host
            res["cli"] = {"host": "C4 stand-in FASTA", "query": "C2 FASTA", **cli(hp, qp, a.cli_reps, work)}
            print("cli", res["cli"], flush=True)
        finally:
            shutil.rmtree(work, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(res["info"])


if __name__ == "__main__":
    main()
