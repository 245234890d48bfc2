"""UCSC .2bit ingest on one GPU against FASTA text of the same genome, seeded inputs generated in the run:

  c2   synth.config_c2() (40 Mbp, 40.8 MB of FASTA, 10 MB of .2bit): engine.run_2bit against engine.run_fasta, median of
       --reps calls each, alternating, page-locked inputs and outputs, every path warmed up first; the stage marks of both
       (frisk_b200_last_run_timing) and their rows compared bit for bit
  c4   the C4 stand-in of synth_device (3 Gbp, a 3 Mbp N run per long scaffold), written as .2bit and as 60-column FASTA on
       the device: the same pair (--c4-reps calls each), and the decode kernels alone (torch.profiler, CUDA activities, in a
       pass of its own over frisk_b200_fasta_open_2bit calls)

The card's name and power limit come from the same run.  Writes one JSON file (--out).

    python tools/twobit_timing.py --out profiles/r06_2bit_timing.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from frisk_b200 import _lib, engine, synth  # noqa: E402
from bgzf_timing import device_info, pinned  # noqa: E402

KERNELS = ("twobit_runs_kernel", "twobit_decode_kernel")
LEGEND = ["file uploaded (and decoded, .2bit)", "packed + counted", "tables + IVOM", "window kernel done", "rows on the host",
          "window kernel could start"]


def marks() -> list:
    ms = (C.c_float * 6)()
    n = C.c_int(0)
    _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)), "last_run_timing")
    return list(ms)[:n.value]


def same(a, b) -> bool:
    return bool(np.array_equal(a.rows, b.rows, equal_nan=True) and np.array_equal(a.status, b.status) and
                np.array_equal(a.tables, b.tables) and list(a.names) == list(b.names) and np.array_equal(a.coords, b.coords) and
                tuple(a.meta) == tuple(b.meta))


def pair(text: np.ndarray, tb: np.ndarray, reps: int, n_rows: int) -> dict:
    """run_fasta on the text against run_2bit on the .2bit file: rows, then alternating timed calls with their marks."""
    out = engine.HostOutputs(n_rows, 8)
    res = {"rows_identical": same(engine.run_2bit(tb), engine.run_fasta(text))}
    paths = {"fasta": lambda: engine.run_fasta(text, out=out, assemble_result=False),
             "2bit": lambda: engine.run_2bit(tb, out=out, assemble_result=False)}
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
    res["windows"] = int(out.n_win)
    res["call_ms"] = {k: {"median": float(np.median(v)), "min": float(min(v)), "all": v} for k, v in times.items()}
    res["stage_marks_ms"] = {"legend": LEGEND, **{k: [float(np.median([m[j] for m in v])) for j in range(len(v[0]))]
                                                  for k, v in mk.items()}}
    res["fasta_over_2bit"] = res["call_ms"]["fasta"]["median"] / res["call_ms"]["2bit"]["median"]
    return res


def decode_kernel_ms(tb: np.ndarray, reps: int) -> dict:
    """Device time of the decode kernels per open (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    engine.DeviceGenome.from_2bit_bytes(tb)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            engine.DeviceGenome.from_2bit_bytes(tb)
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                out[k] = {"ms_per_open": t / 1e3 / reps, "launches_per_open": e.count / reps}
    return out


def device_fasta(dg, width: int = 60) -> np.ndarray:
    """The planes of a device genome as FASTA text (ASCII decoded on the device, 'N' under the invalid plane)."""
    import torch
    g = dg.host
    lut = torch.tensor(list(b"ATGC"), dtype=torch.uint8, device=dg.codes.device)
    shifts = torch.arange(30, -1, -2, dtype=torch.int32, device=dg.codes.device)
    parts = []
    for r, name in enumerate(g.names):
        a, n = int(g.scaf_off[r]), int(g.scaf_len[r])
        parts.append(np.frombuffer((">%s\n" % name).encode(), np.uint8))
        for c0 in range(0, n, 1 << 28):                        # 256 Mbases at a time
            c1 = min(n, c0 + (1 << 28))
            w0, w1 = (a + c0) >> 4, (a + c1 + 15) >> 4
            codes = (dg.codes[w0:w1].unsqueeze(1) >> shifts) & 3
            seq = lut[codes.reshape(-1).long()][(a + c0) - (w0 << 4):(a + c1) - (w0 << 4)]
            m0 = (a + c0) >> 5
            inv = dg.inv[m0:((a + c1 + 31) >> 5)]
            bits = (inv.unsqueeze(1) >> torch.arange(31, -1, -1, dtype=torch.int32, device=inv.device)) & 1
            bad = bits.reshape(-1)[(a + c0) - (m0 << 5):(a + c1) - (m0 << 5)].bool()
            seq = torch.where(bad, torch.full_like(seq, ord("N")), seq).cpu().numpy()
            parts.append(seq)
        # (lines of `width` bases: the text path's tokeniser does not care where the chunk seams fall)
    flat = []
    for p in parts:
        if p.shape[0] and p[0] == ord(">"):
            flat.append(p)
            continue
        full = (p.shape[0] // width) * width
        body = np.empty((p.shape[0] // width, width + 1), np.uint8)
        body[:, :width] = p[:full].reshape(-1, width)
        body[:, width] = 10
        flat.append(body.reshape(-1))
        if p.shape[0] > full:
            flat.append(np.concatenate([p[full:], [10]]).astype(np.uint8))
    return np.concatenate(flat)


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--c4-reps", type=int, default=5)
    ap.add_argument("--skip-c4", action="store_true")
    a = ap.parse_args(argv)
    import torch
    _lib.require_device()
    res = {"info": device_info()}
    sc = synth.config_c2()
    text, tb = synth.fasta_bytes(sc), synth.twobit_bytes(sc)
    res["c2"] = {"sizes": {"fasta": len(text), "2bit": len(tb), "bases": synth.total_bases(sc)}}
    res["c2"].update(pair(pinned(text), pinned(tb), a.reps, len(text) // 2500 + len(text) // 4096 + 64))
    res["c2"]["decode_kernels"] = decode_kernel_ms(pinned(tb), 10)
    del sc, text, tb
    if not a.skip_c4:
        from frisk_b200.synth_device import build_device_genome, c4_spec
        from test_twobit_gpu import planes_to_2bit
        lens, runs = c4_spec()
        dg = build_device_genome(engine, lens, runs, seed=44, at_rich_block=300_000 // 16)
        tb = planes_to_2bit(dg, runs)
        text = device_fasta(dg)
        del dg
        torch.cuda.empty_cache()
        res["c4"] = {"sizes": {"fasta": int(text.shape[0]), "2bit": int(tb.shape[0]), "bases": int(np.sum(lens))}}
        pt, pb = pinned(text.tobytes()), pinned(tb.tobytes())
        del text, tb
        res["c4"].update(pair(pt, pb, a.c4_reps, int(np.sum(lens)) // 2500 + 4096))
        res["c4"]["decode_kernels"] = decode_kernel_ms(pb, 3)
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    for k in ("c2", "c4"):
        if k in res:
            r = res[k]
            print(k, r["sizes"], "rows identical:", r["rows_identical"], "median ms:",
                  {p: round(v["median"], 3) for p, v in r["call_ms"].items()}, "marks:", r["stage_marks_ms"],
                  "decode kernels:", r["decode_kernels"])
    print(res["info"])


if __name__ == "__main__":
    main()
