"""Plain gzip ingest on one GPU, seeded inputs generated in the run: C2 (synth.config_c2(), 40.8 MB of FASTA text) as one
gzip member at levels 1, 6 and 9, each through four paths with their rows compared bit for bit --

  gzip       engine.run_fasta_gzip (frisk_b200_run_fasta_gzip: the member goes up and is inflated on the device)
  host_gzip  the route a .gz took before: gzip.decompress on the host + run_fasta
  text       engine.run_fasta on the plain text
  bgzf       engine.run_fasta_bgzf on the same text as BGZF level 6

-- the stage marks of every gzip call (frisk_b200_last_run_timing), the stats of every inflate, the inflate alone
(frisk_b200_gzip_inflate from device memory: host clock around the synchronising call), its kernels (torch.profiler, in a
pass of its own: boundary search, speculative decode, the serial context step, translation + CRC), and the inflate of
>= 1 GB of text (copies of C2 level 6 joined by full flushes, as pigz writes them: one valid gzip member).
Page-locked inputs and outputs; every path warmed up first; the paths alternate within each repetition.  Writes one
JSON file (--out).

    python tools/gzip_timing.py --out profiles/r04_gzip_timing.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import gzip
import json
import os
import struct
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from frisk_b200 import _lib, engine, synth  # noqa: E402
from bgzf_timing import bgzf, device_info, pinned  # noqa: E402

KERNELS = ("gzip_search_kernel", "gzip_decode_kernel", "gzip_literal_kernel", "gzip_context_kernel", "gzip_translate_kernel")


def gz_member(data: bytes, level: int) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8)
    return (b"\x1f\x8b\x08\0\0\0\0\0\0\x03" + c.compress(data) + c.flush() +
            struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff))


class DeviceInflate:
    """frisk_b200_gzip_inflate on a member already in device memory."""

    def __init__(self, gz: bytes, text_len: int):
        import torch
        self.dev = torch.device("cuda:0")
        self.d_gz = torch.from_numpy(np.frombuffer(gz, np.uint8).copy()).to(self.dev)
        self.d_text = torch.empty(text_len, dtype=torch.uint8, device=self.dev)
        self.n, self.cap = len(gz), text_len

    def __call__(self):
        tl = C.c_uint64(0)
        st = np.zeros(4, np.uint64)
        _lib.check(_lib.lib().frisk_b200_gzip_inflate(engine._ptr(self.d_gz), self.n, engine._ptr(self.d_text), self.cap, C.byref(tl),
                                                      engine._ptr(st), engine._stream_ptr(self.dev)), "frisk_b200_gzip_inflate")
        assert int(tl.value) == self.cap
        return [int(x) for x in st]

    def timed(self, reps: int) -> dict:
        self()
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            self()
            times.append((time.perf_counter() - t0) * 1e3)
        med = float(np.median(times))
        return {"ms_median": med, "ms_min": float(min(times)), "ms_all": times, "text_GB_per_s": self.cap / (med * 1e-3) / 1e9}

    def matches(self, text: bytes) -> bool:
        import torch
        ref = torch.from_numpy(np.frombuffer(text, np.uint8).copy()).to(self.dev)
        k = len(text)
        return all(torch.equal(self.d_text[i:i + k], ref) for i in range(0, self.cap, k))


def kernel_ms(inf: DeviceInflate, reps: int) -> dict:
    """Device time of each inflate kernel per call (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    inf()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            inf()
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                out[k] = {"ms_per_call": t / 1e3 / reps, "launches_per_call": e.count / reps}
    return out


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--big-gb", type=float, default=1.0, help="text of the large inflate run, GB (>= 1)")
    a = ap.parse_args(argv)
    import torch
    _lib.require_device()
    res = {"info": device_info()}
    text = synth.fasta_bytes(synth.config_c2())
    levels = (1, 6, 9)
    gzs = {lv: gz_member(text, lv) for lv in levels}
    gz_b = bgzf(text, 6)
    res["sizes"] = {"text": len(text), "bgzf6": len(gz_b), **{"gzip%d" % lv: len(g) for lv, g in gzs.items()}}
    p_text, p_b = pinned(text), pinned(gz_b)
    p_gz = {lv: pinned(g) for lv, g in gzs.items()}
    out = engine.HostOutputs(len(text) // 2500 + len(text) // 4096 + 64, 8)

    def host_route(blob):
        return engine.run_fasta(np.frombuffer(gzip.decompress(blob), np.uint8), out=out, assemble_result=False)
    paths = {"text": lambda: engine.run_fasta(p_text, out=out, assemble_result=False),
             "bgzf": lambda: engine.run_fasta_bgzf(p_b, out=out, assemble_result=False)}
    for lv in levels:
        paths["gzip%d" % lv] = (lambda g: lambda: engine.run_fasta_gzip(g, out=out, assemble_result=False))(p_gz[lv])
        paths["host_gzip%d" % lv] = (lambda g: lambda: host_route(g))(gzs[lv])
    # rows of every path, bit for bit
    full = {"text": engine.run_fasta(p_text), "bgzf": engine.run_fasta_bgzf(p_b)}
    for lv in levels:
        full["gzip%d" % lv] = engine.run_fasta_gzip(p_gz[lv])
        full["host_gzip%d" % lv] = engine.run_fasta(np.frombuffer(gzip.decompress(gzs[lv]), np.uint8))
    ref = full["text"]
    res["rows_identical"] = {k: bool(np.array_equal(v.rows, ref.rows, equal_nan=True) and np.array_equal(v.status, ref.status) and
                                     np.array_equal(v.tables, ref.tables) and list(v.names) == list(ref.names) and
                                     np.array_equal(v.coords, ref.coords) and tuple(v.meta) == tuple(ref.meta))
                             for k, v in full.items()}
    res["windows"] = int(len(ref.rows))
    del full
    for _ in range(2):
        for f in paths.values():
            f()
    times = {k: [] for k in paths}
    marks = {lv: [] for lv in levels}
    host_inflate = {lv: [] for lv in levels}
    for _ in range(a.reps):
        for k, f in paths.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
            if k.startswith("gzip"):
                ms = (C.c_float * 6)()
                nm = C.c_int(0)
                _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(nm)), "last_run_timing")
                marks[int(k[4:])].append(list(ms)[:nm.value])
        for lv in levels:
            t0 = time.perf_counter()
            gzip.decompress(gzs[lv])
            host_inflate[lv].append((time.perf_counter() - t0) * 1e3)
    res["c2_call_ms"] = {k: {"median": float(np.median(v)), "min": float(min(v)), "all": v} for k, v in times.items()}
    res["c2_host_gunzip_ms"] = {"gzip%d" % lv: float(np.median(v)) for lv, v in host_inflate.items()}
    res["gzip_stage_marks_ms"] = {
        "legend": ["compressed bytes uploaded and inflated", "tokenised + packed + counted", "tables + IVOM",
                   "window kernel done", "rows on the host", "window kernel could start"],
        **{"gzip%d" % lv: [float(np.median([m[j] for m in ms])) for j in range(len(ms[0]))] for lv, ms in marks.items()}}
    med = {k: v["median"] for k, v in res["c2_call_ms"].items()}
    res["ratios"] = {**{"host_gzip%d_over_gzip%d" % (lv, lv): med["host_gzip%d" % lv] / med["gzip%d" % lv] for lv in levels},
                     **{"gzip%d_over_text" % lv: med["gzip%d" % lv] / med["text"] for lv in levels},
                     **{"gzip%d_over_bgzf" % lv: med["gzip%d" % lv] / med["bgzf"] for lv in levels}}
    # the inflate alone, its stats and its kernels
    res["inflate_c2"] = {}
    for lv in levels:
        inf = DeviceInflate(gzs[lv], len(text))
        st = inf()
        r = inf.timed(a.reps)
        r["stats"] = dict(zip(["chunks", "joins_accepted_first_pass", "chunks_repaired", "chunks_rerun_overflow"], st))
        r["output_correct"] = inf.matches(text)
        r["kernels"] = kernel_ms(inf, 5)
        res["inflate_c2"]["gzip%d" % lv] = r
        del inf
    # >= 1 GB of text: copies of C2 level 6, each ended by a full flush, then an empty final block
    c = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
    piece = c.compress(text) + c.flush(zlib.Z_FULL_FLUSH)
    copies = max(1, int(np.ceil(a.big_gb * 1e9 / len(text))))
    crc = 0
    for _ in range(copies):
        crc = zlib.crc32(text, crc)
    big = (b"\x1f\x8b\x08\0\0\0\0\0\0\x03" + piece * copies + b"\x03\x00" +
           struct.pack("<II", crc, (len(text) * copies) & 0xffffffff))
    inf = DeviceInflate(big, len(text) * copies)
    st = inf()
    r = inf.timed(3)
    r.update({"copies_of_c2": copies, "text_bytes": len(text) * copies, "compressed_bytes": len(big),
              "stats": dict(zip(["chunks", "joins_accepted_first_pass", "chunks_repaired", "chunks_rerun_overflow"], st)),
              "output_correct": inf.matches(text), "kernels": kernel_ms(inf, 2)})
    res["inflate_big"] = r
    del inf, big
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("info", "sizes", "rows_identical", "ratios", "gzip_stage_marks_ms")}, indent=1))
    print("c2 call ms (median):", {k: round(v, 3) for k, v in med.items()})
    for k, v in res["inflate_c2"].items():
        print("inflate %s: %.3f ms, stats %s, kernels %s" % (k, v["ms_median"], v["stats"],
              {n: round(x["ms_per_call"], 3) for n, x in v["kernels"].items()}))
    print("inflate big: %.3f ms = %.2f GB/s of text, stats %s" % (r["ms_median"], r["text_GB_per_s"], r["stats"]))


if __name__ == "__main__":
    main()
