"""BGZF ingest on one GPU, seeded inputs generated in the run: C2 (synth.config_c2(), 40.8 MB of FASTA text) through
four paths with their rows compared bit for bit --

  text       plain text -> engine.run_fasta (frisk_b200_run_fasta)
  bgzf       BGZF level 6 -> engine.run_fasta_bgzf (frisk_b200_run_fasta_bgzf: compressed bytes up, inflated on the device)
  host_bgzf  today's route for a .gz: gzip.decompress of the BGZF file on the host + run_fasta
  host_gzip  the same for a single-member gzip -6 file

-- the stage marks of the BGZF call (frisk_b200_last_run_timing), and the inflate kernel alone (frisk_b200_bgzf_inflate,
CUDA events) on C2's blocks and on >= 1 GB of text (copies of the C2 BGZF file back to back: a valid BGZF file).
Host clocks around calls that end in a synchronisation; page-locked inputs and outputs; every path warmed up first; the
paths alternate within each repetition.  Writes one JSON file (--out).

    python tools/bgzf_timing.py --out profiles/r03_bgzf_timing.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import gzip
import json
import os
import struct
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from frisk_b200 import _lib, engine, synth  # noqa: E402

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf(data: bytes, level: int = 6, block: int = 65280, eof: bool = True) -> bytes:
    """BGZF as bgzip writes it: one gzip member per 65,280 bytes, the BC subfield giving its size, the EOF block last."""
    out = []
    for i in range(0, len(data), block):
        piece = data[i:i + block]
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8)
        body = c.compress(piece) + c.flush()
        out.append(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\x00BC\x02\x00" + struct.pack("<H", 18 + len(body) + 8 - 1) + body +
                   struct.pack("<II", zlib.crc32(piece), len(piece)))
    return b"".join(out) + (EOF_BLOCK if eof else b"")


def pinned(data: bytes) -> np.ndarray:
    a = engine._alloc(len(data), np.uint8, True)
    a[:] = np.frombuffer(data, np.uint8)
    return a


def device_info() -> dict:
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "not available"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not available"
    return info


def inflate_kernel_ms(gz: bytes, reps: int, check_text: bytes | None = None) -> dict:
    """The inflate kernel alone: everything on the device first, then CUDA events around each launch."""
    import torch
    L = _lib.lib()
    buf = np.frombuffer(gz, np.uint8)
    nb, tl = C.c_uint64(0), C.c_uint64(0)
    _lib.check(L.frisk_b200_bgzf_blocks(engine._ptr(buf), len(buf), 0, None, None, None, None, C.byref(nb), C.byref(tl)), "blocks")
    n, t_len = int(nb.value), int(tl.value)
    co, cl, crc, to = np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint64)
    _lib.check(L.frisk_b200_bgzf_blocks(engine._ptr(buf), len(buf), n, engine._ptr(co), engine._ptr(cl), engine._ptr(crc),
                                        engine._ptr(to), C.byref(nb), C.byref(tl)), "blocks")
    dev = torch.device("cuda:0")
    as_dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).to(dev)
    d_gz, d_co, d_to = as_dev(buf.copy(), np.uint8), as_dev(co, np.int64), as_dev(to, np.int64)
    d_cl, d_crc = as_dev(cl, np.int32), as_dev(crc, np.int32)
    d_text = torch.empty(t_len, dtype=torch.uint8, device=dev)
    status = torch.zeros(n, dtype=torch.int32, device=dev)
    st = engine._stream_ptr(dev)

    def launch():
        _lib.check(L.frisk_b200_bgzf_inflate(engine._ptr(d_gz), engine._ptr(d_co), engine._ptr(d_cl), engine._ptr(d_crc),
                                             engine._ptr(d_to), n, t_len, engine._ptr(d_text), engine._ptr(status), st), "inflate")
    for _ in range(2):
        launch()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        launch()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    ok = int((status != 0).sum().item()) == 0
    if check_text is not None:                    # the output is the text, every copy of it
        ref = torch.from_numpy(np.frombuffer(check_text, np.uint8).copy()).to(dev)
        k = len(check_text)
        ok = ok and all(torch.equal(d_text[i:i + k], ref) for i in range(0, t_len, k))
    med = float(np.median(times))
    return {"blocks": n, "text_bytes": t_len, "compressed_bytes": len(gz), "ms_median": med, "ms_min": float(min(times)),
            "ms_all": times, "text_GB_per_s": t_len / (med * 1e-3) / 1e9, "output_correct": bool(ok)}



def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--big-gb", type=float, default=1.0, help="text of the large inflate-kernel run, GB (>= 1)")
    a = ap.parse_args(argv)
    import torch
    _lib.require_device()
    res = {"info": device_info()}
    text = synth.fasta_bytes(synth.config_c2())
    t0 = time.perf_counter(); gz6 = bgzf(text, 6); res["bgzf_compress_s"] = time.perf_counter() - t0
    gzs = gzip.compress(text, 6)
    res["sizes"] = {"text": len(text), "bgzf6": len(gz6), "gzip6": len(gzs)}
    p_text, p_gz = pinned(text), pinned(gz6)
    out = engine.HostOutputs(len(text) // 2500 + len(text) // 4096 + 64, 8)

    def host_route(blob):                         # gzip.decompress reads single- and multi-member files alike
        t = gzip.decompress(blob)
        return engine.run_fasta(np.frombuffer(t, np.uint8), out=out, assemble_result=False)
    paths = {
        "text": lambda: engine.run_fasta(p_text, out=out, assemble_result=False),
        "bgzf": lambda: engine.run_fasta_bgzf(p_gz, out=out, assemble_result=False),
        "host_bgzf": lambda: host_route(gz6),
        "host_gzip": lambda: host_route(gzs),
    }
    # (a) rows of all four paths, bit for bit
    full = {"text": engine.run_fasta(p_text), "bgzf": engine.run_fasta_bgzf(p_gz),
            "host_bgzf": engine.run_fasta(np.frombuffer(gzip.decompress(gz6), np.uint8)),
            "host_gzip": engine.run_fasta(np.frombuffer(gzip.decompress(gzs), np.uint8))}
    ref = full["text"]
    res["rows_identical"] = {k: bool(np.array_equal(v.rows, ref.rows, equal_nan=True) and np.array_equal(v.status, ref.status) and
                                     np.array_equal(v.tables, ref.tables) and list(v.names) == list(ref.names) and
                                     np.array_equal(v.coords, ref.coords)) for k, v in full.items()}
    res["windows"] = int(len(ref.rows))
    for _ in range(3):
        for f in paths.values():
            f()
    times = {k: [] for k in paths}
    host_inflate = {"host_bgzf": [], "host_gzip": []}
    marks = []
    for _ in range(a.reps):
        for k, f in paths.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
            if k == "bgzf":
                ms = (C.c_float * 6)()
                nm = C.c_int(0)
                _lib.check(_lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(nm)), "last_run_timing")
                marks.append(list(ms)[:nm.value])
        for k, blob in (("host_bgzf", gz6), ("host_gzip", gzs)):
            t0 = time.perf_counter()
            gzip.decompress(blob)
            host_inflate[k].append((time.perf_counter() - t0) * 1e3)
    res["c2_call_ms"] = {k: {"median": float(np.median(v)), "min": float(min(v)), "all": v} for k, v in times.items()}
    res["c2_host_inflate_ms"] = {k: {"median": float(np.median(v)), "min": float(min(v))} for k, v in host_inflate.items()}
    res["bgzf_stage_marks_ms"] = {
        "legend": ["compressed bytes uploaded and inflated", "tokenised + packed + counted", "tables + IVOM",
                   "window kernel done", "rows on the host", "window kernel could start"],
        "median": [float(np.median([m[j] for m in marks])) for j in range(len(marks[0]))]}
    med = {k: v["median"] for k, v in res["c2_call_ms"].items()}
    res["ratios"] = {"host_bgzf_over_bgzf": med["host_bgzf"] / med["bgzf"], "host_gzip_over_bgzf": med["host_gzip"] / med["bgzf"],
                     "bgzf_over_text": med["bgzf"] / med["text"]}
    # (c) the inflate kernel alone
    res["inflate_kernel_c2"] = inflate_kernel_ms(gz6, a.reps, text)
    copies = max(1, int(np.ceil(a.big_gb * 1e9 / len(text))))
    big = gz6[:-len(EOF_BLOCK)] * copies + EOF_BLOCK
    res["inflate_kernel_big"] = inflate_kernel_ms(big, 5, text)
    res["inflate_kernel_big"]["copies_of_c2"] = copies
    del big
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("info", "sizes", "rows_identical", "ratios", "bgzf_stage_marks_ms")}, indent=1))
    print("c2 call ms (median):", {k: round(v, 3) for k, v in med.items()})
    print("inflate kernel: c2 %.3f ms, big %.3f ms = %.1f GB/s of text" % (res["inflate_kernel_c2"]["ms_median"],
          res["inflate_kernel_big"]["ms_median"], res["inflate_kernel_big"]["text_GB_per_s"]))


if __name__ == "__main__":
    main()
