#!/usr/bin/env python
"""Benchmark of the frisk hot path (BASELINE.json metric: Gbp/s of scaffold scored =
background k-mer count + per-window IVOM/KLD score).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the CPU arm (oracle port)

Headline workload: BASELINE config C2 -- synthetic 40 Mbp fungal-style assembly, ~500 scaffolds, default
k = 1..8, window 5000 / step 2500, RIP on.  At N > 1 (torchrun, one rank per GPU) every rank holds its own
40 Mbp shard (seed 2002 + rank) of a 40*N Mbp assembly -- weak scaling -- and the only exchange on the data
path is the sum of the 87,380 forward k-mer counters (fused into the finalise kernel over NVLink peer memory;
--nccl: one NCCL all-reduce).

A step = one full pass: zero counters, background count, [exchange], finalise tables, genome IVOM table,
score every window.  `value` has the packed planes + window list resident in HBM; `e2e` goes through ONE
C-ABI call from pinned HOST buffers (H2D of planes and window list, D2H of rows/status/tables inside the
timed region).  L2 (126 MB) is flushed between timed steps by writing a 512 MiB buffer.

Further blocks of the same JSON line (each measured in this run):
  roofline   the dominant kernel against the bound that binds it (shared-memory atomic updates, SURVEY 8d), the
             HBM view, and live micro-benchmarks of the other two candidate bounds (L2 gathers, fp64)
  parity     N > 1: the globally finalised tables against the C oracle on all shards, fused vs NCCL exchange,
             and sampled rows of every rank against the oracle
  strong     BASELINE config C4 (3 Gbp, 1.2 M windows): the same genome on N GPUs, equal slices of the base range
             and of the window list per rank (strong scaling), with N-independent checksums
  c5         N > 1: BASELINE config C5 at 1.75 Gbp / 125,000 scaffolds per GPU (14 Gbp on 8) from FASTA TEXT, each rank
             ingesting its own byte range on its own GPU: ingest-inclusive and kernel-only time, imbalance
  c3_sweep   BASELINE config C3 (120 Mbp, kmax' = 1..8 from one counting pass)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "C2: synthetic 40 Mbp fungal-style assembly, ~500 scaffolds, k=1..8, w=5000, step=2500, RIP"
METRIC = "Gbp/s scaffold scored (k-mer count+window score)"
PARAMS = dict(kmin=1, kmax=8, w=5000, step=2500, mask_host=False, scaffolds_all=False, rip=True)
# the same dict in both arms (the driver compares them); arm-specific detail goes to `run`
CONFIG = {"workload": WORKLOAD, "kmin": 1, "kmax": 8, "window": 5000, "step": 2500, "rip": True,
          "bases_per_gpu": "40.09 Mbp (seed 2002 + rank)", "l2": "flushed between timed steps (512 MiB write)"}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ----------------------------------------------------------------------------- live micro-benchmarks
def _best(fn, n=3):
    best = 0.0
    for _ in range(n):
        best = max(best, fn())
    return best


def measure_smem_atomic_rate():
    """Shared-memory atomic updates/s of this GPU on uniformly random bins (the realistic-conflict case)."""
    from frisk_b200 import _lib

    def once():
        ms = C.c_float(0)
        blocks, iters = 148 * 2, 4096
        _lib.check(_lib.lib().frisk_b200_bench_smem_atomics(blocks, iters, 1, C.byref(ms), None), "bench_smem_atomics")
        return blocks * 1024 * iters / (ms.value * 1e-3)
    try:
        return _best(once)
    except Exception:
        return None


def measure_l2_gather_rate(mode=0):
    """Random 16-byte gathers/s from an L2-resident 1 MiB table (= the genome IVOM table of kmax 8); mode 1: a warp's
    lanes read increasing addresses (the pattern of an epilogue that walks the K-mers in sorted order)."""
    from frisk_b200 import _lib

    def once():
        ms = C.c_float(0)
        blocks, iters = 148 * 4, 2048
        _lib.check(_lib.lib().frisk_b200_bench_l2_gather(blocks, iters, 1 << 20, mode, C.byref(ms), None), "bench_l2_gather")
        return blocks * 256 * iters / (ms.value * 1e-3)
    try:
        return _best(once)
    except Exception:
        return None


def measure_smem_load_rate(nbytes):
    from frisk_b200 import _lib

    def once():
        ms = C.c_float(0)
        blocks, iters = 148 * 4, 8192
        _lib.check(_lib.lib().frisk_b200_bench_smem_loads(blocks, iters, nbytes, C.byref(ms), None), "bench_smem_loads")
        return blocks * 256 * iters / (ms.value * 1e-3)
    try:
        return _best(once)
    except Exception:
        return None


def score_kernel_name(kmin, kmax, max_len):
    from frisk_b200 import _lib
    buf = C.create_string_buffer(160)
    _lib.check(_lib.lib().frisk_b200_score_kernel_name(kmin, kmax, max_len, buf, 160), "score_kernel_name")
    return buf.value.decode()


def committed_capture(kernel):
    """The committed `ncu --set full` capture of the dominant kernel (profiles/r02_ncu_score_kernel.json, written by
    tools/ncu_capture.py from the same command; a run under ncu is never timed).  The capture must be OF THE KERNEL
    THE LAUNCHER SELECTS TODAY: a stale capture is reported as such, loudly, instead of being quoted."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_score_kernel.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
    except Exception as e:
        return {"error": "no committed capture (%s)" % e}
    want = kernel.replace(" ", "")
    got = str(d.get("kernel", "")).replace(" ", "")
    if want not in got:
        msg = "STALE ncu capture: profiles/r02_ncu_score_kernel.json is of '%s' but the launcher runs '%s'" % (d.get("kernel"), kernel)
        print("bench.py: " + msg, file=sys.stderr)
        return {"error": msg}
    d["source"] = "profiles/r02_ncu_score_kernel.json (ncu --set full of this bench command, not timed)"
    return d


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append((time.time(), [x.strip() for x in line.split(",")]))
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def finish(self, t0, t1):
        self.stop_flag.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        rows = [r for t, r in self.samples if t0 - 0.05 <= t <= t1 + 0.15 and len(r) >= 7] or \
               [r for _, r in self.samples if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


# ----------------------------------------------------------------------------- CPU arms
def cpu_port_sample(scaffolds, target_seconds: float, threads: int):
    """Time the C oracle (a port of the reference's algorithm, oracle/frisk_oracle.c) on a bounded
    sample: the first scaffolds of the workload, background pass + every window of the sample,
    scored against the sample's own background.  Cost is linear in bases and windows, so Gbp/s
    of the sample is the CPU path's Gbp/s on the workload."""
    probe = []
    tot = 0
    for s in scaffolds:
        probe.append(s)
        tot += len(s[1])
        if tot >= 400_000:
            break
    t0 = time.perf_counter()
    _one_cpu_pass(probe, threads)
    rate = tot / (time.perf_counter() - t0)
    want = max(int(rate * target_seconds), 200_000)
    sample, tot = [], 0
    for s in scaffolds:
        sample.append(s)
        tot += len(s[1])
        if tot >= want:
            break
    return sample, tot


def _one_cpu_pass(sample, threads):
    from oracle import c_oracle
    seq, off = c_oracle.concat(sample)
    tabs, meta = c_oracle.background(seq, off, PARAMS["kmin"], PARAMS["kmax"], False, threads)
    _, woff, wlen, _, _ = c_oracle.crawl(seq, off, PARAMS["w"], PARAMS["step"], False)
    rows, status = c_oracle.score(seq, woff, wlen, tabs, meta, PARAMS["kmin"], PARAMS["kmax"], True, threads)
    return len(woff)


def python_port_rate(scaffolds, bases: int = 30_000):
    """The Python restatement (same data structures as the reference: dicts of k-mer strings) on a
    tiny sample, 1 core -- how fast the reference itself runs."""
    from oracle import frisk_oracle
    name, seq = scaffolds[0]
    sub = [(name, seq[:bases].tobytes().decode())]
    t0 = time.perf_counter()
    frisk_oracle.score_windows(sub, PARAMS["kmin"], PARAMS["kmax"], PARAMS["w"], PARAMS["step"])
    return bases / (time.perf_counter() - t0) / 1e9


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The
    reference is Python-2-only pure Python and cannot be installed or run on the GPU box (see
    DESIGN.md), so the arm times the oracle PORT (C restatement, all host threads): a far faster
    stand-in than the reference's own dict loops, whose speed is reported beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from frisk_b200 import synth
    threads = os.cpu_count() or 1
    scaffolds = synth.make("C2", 1.0)
    sample, tot = cpu_port_sample(scaffolds, 2.0, threads)
    for _ in range(args.warmup):
        _one_cpu_pass(sample, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        nwin = _one_cpu_pass(sample, threads)
    dt = time.perf_counter() - t0
    value = tot * args.steps / dt / 1e9
    sample_desc = "first %d scaffolds of C2 = %d bp, %d windows per step (background + all windows of the sample)" % (
        len(sample), tot, nwin)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64 counts + f64 scores", "data": "synthetic",
        "config": dict(CONFIG),
        "run": {"sample": sample_desc, "cores": threads},
        "cpu_baseline": {"value": value, "unit": "Gbp/s", "cores": threads, "kind": "port", "sample": sample_desc,
                         "python_port_1core_gbps": python_port_rate(scaffolds)},
        "e2e": {"value": value, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm: the extra blocks
def parity_block(rank, world, dev, scaffolds, genome, pipe, allreduce, space):
    """N > 1, after the timed region: (1) the tables every rank finalised from the fused peer sum == the tables of a
    second pass through the NCCL all-reduce == the C oracle's background of ALL shards (rank 0 regenerates them);
    (2) 32 sampled windows per rank, scored by the oracle against those tables."""
    import torch
    import torch.distributed as dist
    from frisk_b200 import engine, synth
    torch.cuda.synchronize(dev)
    tables_main = pipe.d_tables.clone()
    exchange_main = "fused" if pipe.peers is not None else "nccl"
    other = engine.Pipeline(pipe.dq, device=dev, allreduce=allreduce, genome_space=space, wins=pipe.wins, **PARAMS)   # NCCL exchange
    other.enqueue()
    torch.cuda.synchronize(dev)
    same = torch.tensor([int(torch.equal(other.d_tables, tables_main)), int(torch.equal(other.d_rows.nan_to_num(-1.0), pipe.d_rows.nan_to_num(-1.0)))],
                        device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    # sampled rows of this rank
    status = pipe.d_status.cpu().numpy().view(np.uint32)
    rows = pipe.d_rows.cpu().numpy()
    ok = np.nonzero((status & 8) == 0)[0]
    rng = np.random.Generator(np.random.PCG64(77 + rank))
    pick = np.sort(rng.choice(ok, min(32, len(ok)), replace=False))
    w = pipe.wins
    payload = (w.scaf[pick].astype(np.int64), (w.off[pick] - genome.scaf_off[w.scaf[pick]]).astype(np.int64),
               w.length[pick].astype(np.int64), rows[pick], status[pick])
    out = [None] * world if rank == 0 else None
    dist.gather_object(payload, out, dst=0)
    if rank != 0:
        return None
    from oracle import c_oracle
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    shards = [scaffolds] + [synth.make("C2", 1.0, seed=2002 + r) for r in range(1, world)]
    seq, off = c_oracle.concat([s for sh in shards for s in sh])
    tabs, meta = c_oracle.background(seq, off, PARAMS["kmin"], PARAMS["kmax"], False, threads)
    tables_exact = bool(np.array_equal(tables_main.cpu().numpy().view(np.uint64), tabs))
    base = np.cumsum([0] + [len(sh) for sh in shards])                 # first scaffold of every shard in the concatenation
    woff, wlen, got, gst = [], [], [], []
    for r, (sc, rel, ln, rw, st) in enumerate(out):
        woff.append(off[base[r] + sc].astype(np.int64) + rel)
        wlen.append(ln); got.append(rw); gst.append(st)
    woff = np.concatenate(woff).astype(np.uint64); wlen = np.concatenate(wlen).astype(np.uint32)
    got = np.concatenate(got); gst = np.concatenate(gst)
    ref_rows, ref_st = c_oracle.score(seq, woff, wlen, tabs, meta, PARAMS["kmin"], PARAMS["kmax"], True, threads)
    good = ref_st == 0
    rel_err = np.abs(got[good, 0] - ref_rows[good, 0]) / np.maximum(np.abs(ref_rows[good, 0]), 1e-300)
    others_exact = bool(np.array_equal(got[good, 1:], ref_rows[good, 1:], equal_nan=True)) and bool(np.array_equal(gst & 7, ref_st & 7))
    return {"tables": "exact" if tables_exact else "MISMATCH", "tables_exchange": exchange_main,
            "tables_fused_vs_nccl": "exact" if int(same[0]) else "MISMATCH", "rows_fused_vs_nccl": "identical" if int(same[1]) else "MISMATCH",
            "rows_checked": int(good.sum()), "rows_max_rel": float(rel_err.max()) if rel_err.size else None,
            "gc_pi_si_cri": "exact" if others_exact else "MISMATCH",
            "oracle": "C port of the reference (oracle/frisk_oracle.c): background of all %d shards (%d bp) + %d sampled windows, %d threads, %.1f s"
                      % (world, int(off[-1]), len(woff), threads, time.perf_counter() - t0)}


def strong_block(rank, world, dev, peers_ok, steps=3):
    """BASELINE config C4 (3 Gbp, 26 scaffolds of up to 250 Mbp, 3 Mbp N runs, 1.2 M windows), STRONG scaling: every rank
    holds the planes (drawn on its own GPU from the same seed: frisk_b200/synth_device.py), counts an equal slice of the
    base range and scores an equal slice of the window list (dist.score_balanced's scheme); one exchange of the counters."""
    import torch
    import torch.distributed as dist
    from frisk_b200 import engine, synth_device
    from frisk_b200 import dist as fdist
    dg = synth_device.c4_device_genome(engine, device=dev)
    g = dg.host
    wins_all = g.windows(PARAMS["w"], PARAMS["step"], False)
    a, b = fdist.split_windows(wins_all.length, world)[rank]
    kw = {}
    peers = None
    if world > 1:
        if peers_ok:
            peers = fdist.PeerExchange(PARAMS["kmax"], dev)
        kw = dict(allreduce=fdist.make_allreduce(), bg_range=fdist.split_base_range(g.padded_len, world)[rank], peers=peers)
    pipe = engine.Pipeline(dg, wins=wins_all.slice(a, b), device=dev, **kw, **PARAMS)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    pipe.enqueue()
    barrier()
    ms = []
    for _ in range(steps):
        barrier()
        marks = []
        pipe.enqueue(marks)
        torch.cuda.synchronize(dev)
        ms.append([marks[i].elapsed_time(marks[i + 1]) for i in range(3)])
    ms = np.array(ms)
    step = torch.tensor([float(ms.sum(1).mean())] + [float(x) for x in ms.mean(0)], dtype=torch.float64, device=dev)
    st = pipe.d_status.view(torch.int32)
    ok = st == 0
    kld = pipe.d_rows[:, 0]
    chk = torch.stack([torch.where(ok, kld, torch.zeros_like(kld)).sum(), ok.sum().to(torch.float64),
                       ((st & 8) != 0).sum().to(torch.float64)])
    if world > 1:
        dist.all_reduce(step, op=dist.ReduceOp.MAX)
        dist.all_reduce(chk, op=dist.ReduceOp.SUM)
    out = None
    if rank == 0:
        t = float(step[0])
        out = {"workload": "C4: 3 Gbp human-scale stand-in, 26 scaffolds, w=5000 step=2500 k=1..8 (device-drawn: synth_device.c4_spec)",
               "scaling": "strong", "bases": int(g.total_len), "windows": len(wins_all), "ms_per_step": t,
               "value": g.total_len / t / 1e6, "unit": "Gbp/s", "steps": steps,
               "stage_ms_max": {"background": float(step[1]), "tables+ivom+exchange": float(step[2]), "score": float(step[3])},
               "exchange": "fused peer sum" if pipe.peers is not None else ("NCCL all-reduce" if world > 1 else "none"),
               "checksums": {"kld_sum": repr(float(chk[0])), "rows_ok": int(chk[1]), "rows_excluded": int(chk[2]),
                             "tables_sum": int(pipe.d_tables.sum().item())},
               "note": "checksums do not depend on N (kld_sum up to the order of the final sum over ranks, ~1e-16 relative)"}
    del pipe, dg
    torch.cuda.empty_cache()
    return out


def c5_text_on_device(rank, dev, n_scaf, total_bases):
    """This rank's share of the C5 stand-in as FASTA TEXT, built on the GPU and copied to pinned host memory: lognormal
    scaffold lengths (median ~9 kbp, min 480, rounded to whole 60-base lines), 30 % of the scaffolds with 1-3 N runs of
    10-2,000 bp, 61-byte lines (headers padded to the line width, so the text is one [rows, 61] byte matrix)."""
    import torch
    from frisk_b200 import engine, synth_device
    lens, (run_s, run_o, run_l) = synth_device.c5_spec(n_scaf, total_bases, seed=5005 + rank)
    lines = np.maximum(lens // 60, 8)                                   # whole lines per scaffold
    lens = lines * 60
    first_row = np.cumsum(lines + 1) - (lines + 1)                       # header row of every scaffold
    n_rows = int((lines + 1).sum())
    gen = torch.Generator(device=dev)
    gen.manual_seed(5055 + rank)
    lut = torch.tensor(list(b"ATGC"), dtype=torch.uint8, device=dev)
    text = torch.empty((n_rows, 61), dtype=torch.uint8, device=dev)
    step_rows = 1 << 22
    for r0 in range(0, n_rows, step_rows):                               # bases: uniform ACGT, GC 0.5 (chunked: bounded temporaries)
        r1 = min(n_rows, r0 + step_rows)
        text[r0:r1, :60] = lut[torch.randint(0, 4, (r1 - r0, 60), device=dev, generator=gen, dtype=torch.int64)]
    text[:, 60] = 10
    # N runs: base k of scaffold s sits at row first_row[s] + 1 + k // 60, column k % 60
    run_l = np.minimum(run_l, np.maximum(lens[run_s] - run_o - 1, 1))
    tot = int(run_l.sum())
    rs = torch.from_numpy(np.repeat(first_row[run_s] + 1, run_l)).to(dev)
    k = torch.from_numpy(np.repeat(run_o, run_l) + (np.arange(tot) - np.repeat(np.cumsum(run_l) - run_l, run_l))).to(dev)
    text[rs + k // 60, k % 60] = ord("N")
    # header rows: ">scfRRNNNNNNN " + padding + "\n"
    hdr = np.full((len(lens), 61), ord("x"), dtype=np.uint8)
    hdr[:, 0] = ord(">"); hdr[:, 1:4] = np.frombuffer(b"scf", dtype=np.uint8)
    ids = rank * 10_000_000 + np.arange(len(lens), dtype=np.int64)
    for d in range(9):
        hdr[:, 4 + d] = ord("0") + (ids // 10 ** (8 - d)) % 10
    hdr[:, 13] = ord(" "); hdr[:, 60] = 10
    text[torch.from_numpy(first_row).to(dev)] = torch.from_numpy(hdr).to(dev)
    host = engine._alloc(n_rows * 61, np.uint8, True)
    torch.from_numpy(host).copy_(text.reshape(-1))
    torch.cuda.synchronize(dev)
    del text, rs, k
    torch.cuda.empty_cache()
    return host, int(lens.sum()), int(run_l.sum())


def c5_block(rank, world, dev, peers_ok, steps=3):
    """BASELINE config C5 (wheat-scale fragmented assembly, many N gaps, --scaffoldsAll) at 125,000 scaffolds / 1.75 Gbp per
    GPU (1 M scaffolds / 14 Gbp on 8), from FASTA TEXT: every rank uploads and tokenises only its own byte range on its own
    GPU (dist.score_fasta_sharded), counts it, exchanges the counters once, scores its own windows."""
    import torch
    import torch.distributed as dist
    from frisk_b200 import engine
    from frisk_b200 import dist as fdist
    text, bases, n_unres = c5_text_on_device(rank, dev, 125_000, 14.0e9 / 8)
    params = dict(PARAMS, scaffolds_all=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    px = fdist.PeerExchange(PARAMS["kmax"], dev) if (world > 1 and peers_ok) else None
    res, _ = fdist.score_fasta_sharded(None, local_text=text, device=dev, fused=peers_ok, peers=px, row_names=False, **params)   # warm-up + the books
    books_ok = int(res.tables[:4].sum()) // 2 == res.meta[0] - res.meta[2]                               # order-1 total = resolved bases x 2 strands
    t_incl = []
    for _ in range(steps):
        barrier()
        t0 = time.perf_counter()
        res, _ = fdist.score_fasta_sharded(None, local_text=text, device=dev, fused=peers_ok, peers=px, row_names=False, **params)
        torch.cuda.synchronize(dev)
        t_incl.append((time.perf_counter() - t0) * 1e3)
    # kernel-only: the same shard resident
    dq = engine.DeviceGenome.from_fasta_bytes(text, dev)
    space = fdist.global_genome_space(dq.host.genome_space, dev) if world > 1 else dq.host.genome_space
    pipe = engine.Pipeline(dq, device=dev, allreduce=fdist.make_allreduce() if world > 1 else None, genome_space=space, peers=px, **params)
    pipe.enqueue()
    barrier()
    t_kern = []
    for _ in range(steps):
        barrier()
        marks = []
        pipe.enqueue(marks)
        torch.cuda.synchronize(dev)
        t_kern.append(marks[0].elapsed_time(marks[3]))
    n_win = len(pipe.wins)
    agg = torch.tensor([float(np.mean(t_incl)), float(np.mean(t_kern)), float(bases), float(n_win)], dtype=torch.float64, device=dev)
    mx = agg.clone(); sm = agg.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    out = None
    if rank == 0:
        tot_bases, tot_win = float(sm[2]), float(sm[3])
        out = {"workload": "C5: wheat-scale fragmented stand-in, 125,000 scaffolds / 1.75 Gbp per GPU (lognormal, median ~9 kbp), N runs in 30 %% "
                           "of them, --scaffoldsAll, from FASTA text (61-byte lines), %d GPU(s)" % world,
               "scaling": "weak", "bases": int(tot_bases), "scaffolds": 125_000 * world, "windows": int(tot_win),
               "text_bytes_per_gpu": int(text.shape[0]),
               "ingest_inclusive": {"ms": float(mx[0]), "value": tot_bases / float(mx[0]) / 1e6, "unit": "Gbp/s",
                                    "what": "pinned FASTA text -> H2D -> tokenise + 2-bit pack on the GPU -> record table to the host -> "
                                            "window list -> count, exchange, score -> rows on the host (wall clock, max over ranks)"},
               "kernel_only": {"ms": float(mx[1]), "value": tot_bases / float(mx[1]) / 1e6, "unit": "Gbp/s",
                               "what": "planes + window list resident: count, exchange, finalise, score (CUDA events, max over ranks)"},
               "imbalance": {"bases_max_over_mean": float(mx[2]) / (tot_bases / world), "windows_max_over_mean": float(mx[3]) / (tot_win / world)},
               "books": "order-1 total == 2 x resolved bases" if books_ok else "MISMATCH", "steps": steps}
    del pipe, dq
    torch.cuda.empty_cache()
    return out


def c3_sweep_block(rank, world, dev, steps=3):
    """BASELINE config C3 (120 Mbp plant-style, 12 chromosomes, 30 % repeats): scores for every kmax' = 1..8 (eight
    reference runs `-m 1 -k k'`) from ONE counting pass.  N > 1: the chromosomes' windows are split across ranks like C4."""
    import torch
    import torch.distributed as dist
    from frisk_b200 import engine, synth
    from frisk_b200 import dist as fdist
    sc = synth.make("C3", 1.0)
    g = engine.PackedGenome.from_scaffolds(sc)
    sweep = engine.Sweep(g, device=dev, rank=rank, world=world, allreduce=fdist.make_allreduce() if world > 1 else None, **{k: v for k, v in PARAMS.items() if k not in ("kmax", "kmin")})

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    sweep.enqueue()
    barrier()
    ms = []
    for _ in range(steps):
        barrier()
        marks = []
        sweep.enqueue(marks)
        torch.cuda.synchronize(dev)
        ms.append(marks[0].elapsed_time(marks[-1]))
    t = torch.tensor([float(np.mean(ms))], dtype=torch.float64, device=dev)
    chk = sweep.checksums()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(chk, op=dist.ReduceOp.SUM)
    out = None
    if rank == 0:
        out = {"workload": "C3: 120 Mbp plant-style assembly, kmax' = 1..8 (kmin 1), w=5000 step=2500, one counting pass",
               "bases": int(g.total_len), "windows": len(sweep.wins_all), "k_runs": 8, "ms_per_sweep": float(t[0]),
               "value": 8 * g.total_len / float(t[0]) / 1e6, "unit": "Gbp/s (bases x 8 k-runs per second)",
               "launches": sweep.launches, "kld_sums_by_kmax": [repr(float(x)) for x in chk.tolist()], "steps": steps}
    del sweep
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------- GPU arm
def dump_outputs(out_dir, res, prefix=""):
    """The arrays a caller of the timed path receives (Pipeline.result(): rows windowKLD/GC/PI/SI/CRI, row status bits,
    background tables, window coordinates, totalLen/exMax/nnTotal), all of them, as float64: counts and coordinates stay
    below 2**53, so the conversion is exact.  About 2 MB per GPU for C2."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"rows": res.rows, "status": res.status, "tables": res.tables, "coords": res.coords, "meta": np.array(res.meta)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from frisk_b200 import _lib, engine, synth
    from frisk_b200 import dist as fdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.require_device()
    for item in args.option or []:           # A/B of kernel choices: frisk_b200_set_option (e.g. force_bucket_kernel=1)
        name, _, val = item.partition("=")
        _lib.check(_lib.lib().frisk_b200_set_option(name.encode(), int(val or 1)), "set_option " + item)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # this rank's shard: 40 Mbp, packed into pinned planes (ingest is outside the timed region)
    scaffolds = synth.make("C2", 1.0, seed=2002 + rank)
    t0 = time.perf_counter()
    genome = engine.PackedGenome.from_scaffolds(scaffolds, pinned=True)
    t_pack = time.perf_counter() - t0
    bases = genome.total_len
    allreduce, space = None, genome.genome_space
    peers = None
    peers_ok = False
    if world > 1:
        space = fdist.global_genome_space(space, dev)
        allreduce = fdist.make_allreduce()
        if not args.nccl:
            peers = fdist.PeerExchange(PARAMS["kmax"], dev)
            ok = torch.tensor([int(peers.available)], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)                     # all ranks or none
            if not int(ok.item()):
                if rank == 0:
                    print("fused peer exchange unavailable (%s): NCCL all-reduce" % peers.reason, file=sys.stderr)
                peers = None
            peers_ok = peers is not None
    pipe = engine.Pipeline(genome, device=dev, allreduce=allreduce, genome_space=space, peers=peers, **PARAMS)
    collective = "none" if world == 1 else ("counters summed inside the finalise kernel over NVLink peer memory" if pipe.peers is not None
                                            else "1 NCCL all-reduce")
    n_win = len(pipe.wins)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        pipe.enqueue()
    barrier()

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.35)
    marks_all = []
    t_wall0 = time.time()
    barrier()
    for _ in range(args.steps):
        flush.fill_(1)                       # evict the planes and tables from L2 (not timed)
        marks = []
        pipe.enqueue(marks)                  # marks[0] precedes the zeroing of the counters: the whole step is timed
        marks_all.append(marks)
    barrier()
    t_wall1 = time.time()
    stage = np.array([[m[i].elapsed_time(m[i + 1]) for i in range(3)] for m in marks_all])   # ms
    step_ms = np.array([m[0].elapsed_time(m[3]) for m in marks_all])
    total_ms = float(step_ms.sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pipe.result(names=False), "" if world == 1 else "rank%d_" % rank)

    # ---- end to end through ONE C-ABI call from pinned host buffers; H2D of planes + window list and D2H of the rows
    # ---- inside the timer.  No cross-rank host barrier between steps (a pipeline has none): the ranks meet inside the call.
    out = engine.HostOutputs(n_win, PARAMS["kmax"])
    wins = pipe.wins
    e2e_steps = args.steps

    def e2e_once():
        if world == 1:
            return engine.run_host(genome, wins=wins, out=out, assemble_result=False, **PARAMS)
        if pipe.peers is not None:
            return pipe.peers.run_host(genome, wins, out, space, stream_ptr=engine._stream_ptr(dev), **PARAMS)
        return pipe.step_from_host(out)

    def last_call_stages():
        ms = (C.c_float * 6)()
        n = C.c_int(0)
        if _lib.lib().frisk_b200_last_run_timing(ms, 6, C.byref(n)) != 0:
            return None
        return [float(ms[i]) for i in range(n.value)]

    if args.profile:
        e2e_steps = 0
    else:
        e2e_once()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e2e_ms = 0.0
    stage_rows = []
    for _ in range(e2e_steps):
        flush.fill_(1)
        e0.record()
        e2e_once()
        e1.record()
        torch.cuda.synchronize(dev)
        e2e_ms += e0.elapsed_time(e1)
        st = last_call_stages() if (world == 1 or pipe.peers is not None) else None
        if st:
            stage_rows.append(st)
    # ---- end to end from FASTA TEXT (what the reference's CLI is given): pinned text -> H2D ->
    # ---- device-side tokenise + pack -> windows -> same kernels -> rows on the host (N = 1 only)
    fasta_ms, fasta_bytes_n, ingest_ms, fasta_stages = 0.0, 0, [], None
    if world == 1 and e2e_steps:
        raw = np.frombuffer(synth.fasta_bytes(scaffolds), dtype=np.uint8)
        text = engine._alloc(raw.shape[0], np.uint8, True)
        text[:] = raw
        fasta_bytes_n = int(text.shape[0])
        engine.run_fasta(text, out=out, assemble_result=False, **PARAMS)
        ingest_ms = []
        for _ in range(5):                              # the ingest alone: text upload + tokenise + pack on the device
            torch.cuda.synchronize(dev)
            t0i = time.perf_counter()
            dgi = engine.DeviceGenome.from_fasta_bytes(text, dev)
            torch.cuda.synchronize(dev)
            ingest_ms.append((time.perf_counter() - t0i) * 1e3)
            del dgi
        fasta_stage_rows = []
        for _ in range(e2e_steps):
            flush.fill_(1)
            barrier()
            e0.record()
            engine.run_fasta(text, out=out, assemble_result=False, **PARAMS)
            e1.record()
            torch.cuda.synchronize(dev)
            fasta_ms += e0.elapsed_time(e1)
            st = last_call_stages()
            if st:
                fasta_stage_rows.append(st)
        fasta_ms /= e2e_steps
        if fasta_stage_rows:
            m = np.mean(np.array(fasta_stage_rows), axis=0)
            fasta_stages = {"text_uploaded": float(m[0]), "tokenised+packed+counted": float(m[1]), "tables+ivom": float(m[2]),
                            "window_kernel_started": float(m[5]) if len(m) > 5 else None,
                            "scored": float(m[3]), "rows_on_host": float(m[4]),
                            "note": "ms since the start of the one C call (device-side events on the call's streams), mean over the "
                                    "timed steps; tokenise, pack and count of a chunk run while the next chunk is on the bus"}
    clocks = sampler.finish(t_wall0, t_wall1)

    h2d = genome.plane_bytes + wins.off.nbytes + wins.length.nbytes
    if world == 1 or pipe.peers is not None:      # the C call uploads the invalid plane as (index, word) pairs
        h2d += 8 * len(genome.inv_sparse()[0]) - genome.inv.nbytes
    d2h = n_win * 44 + _lib.table_size(1, PARAMS["kmax"]) * 8 + 8

    # max over ranks of the timed totals; sum over ranks of the bases
    tot = torch.tensor([total_ms, e2e_ms / max(e2e_steps, 1)], dtype=torch.float64, device=dev)
    cnt = torch.tensor([bases, n_win], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    total_ms, e2e_step_ms = float(tot[0]), float(tot[1])
    all_bases, all_win = int(cnt[0]), int(cnt[1])
    # per-rank stage breakdown of the e2e call: max and min over ranks of each stage's mean
    breakdown = None
    if stage_rows:
        mean = np.array(stage_rows).mean(0)                      # [uploaded, counted, finalised, scored, end, window kernel started] since call start
        per = np.array([mean[0], mean[1], mean[2] - mean[1], mean[3] - mean[2], mean[4] - mean[3], mean[4]])
        tmax = torch.tensor(per, dtype=torch.float64, device=dev); tmin = tmax.clone()
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        names = ["upload_done", "count_done", "tables+ivom (incl. wait for the peers)", "score", "download_tail", "call_total"]
        breakdown = {n: {"max_ms": float(a), "min_ms": float(b)} for n, a, b in zip(names, tmax.tolist(), tmin.tolist())}
        breakdown["note"] = ("device-side event times inside the one C call, mean over the e2e steps, max / min over ranks; upload and count overlap "
                             "(chunked copy stream), so count_done ~ upload_done + the last chunk's count")

    # ---- the other blocks (each rank takes part; rank 0 reports)
    extra = {}

    def guarded(name, fn, *a):
        """An extra block must never cost the headline line: a failure is reported in its place."""
        try:
            extra[name] = fn(*a)
        except Exception as e:                      # noqa: BLE001
            import traceback
            traceback.print_exc(file=sys.stderr)
            extra[name] = {"error": "%s: %s" % (type(e).__name__, e)}
            try:
                torch.cuda.empty_cache()
            except Exception:
                pass

    if not args.profile and not args.quick:
        if world > 1:
            guarded("parity", parity_block, rank, world, dev, scaffolds, genome, pipe, allreduce, space)
        del flush
        torch.cuda.empty_cache()
        guarded("strong", strong_block, rank, world, dev, peers_ok)
        if world > 1 or args.c5:
            guarded("c5", c5_block, rank, world, dev, peers_ok)
        guarded("c3_sweep", c3_sweep_block, rank, world, dev)

    occ = None
    try:
        a, b = C.c_int(0), C.c_int(0)
        _lib.check(_lib.lib().frisk_b200_score_occupancy(PARAMS["kmax"], wins.max_len, C.byref(a), C.byref(b)), "score_occupancy")
        occ = {"ctas_per_sm": a.value, "threads_per_cta": b.value}
    except Exception:
        pass
    if rank == 0:
        value = all_bases * args.steps / (total_ms * 1e-3) / 1e9
        peak, peak_kind = measured_peak_gbs()
        score_ms = float(stage[:, 2].mean())
        kernel = score_kernel_name(PARAMS["kmin"], PARAMS["kmax"], wins.max_len)
        low_b = 0.125 if genome.low is not None else 0.0
        alg_bytes = bases * (0.375 + low_b) + n_win * 40.0          # SURVEY 8(d): packed read once + one row/window
        hbm_achieved = alg_bytes / (score_ms * 1e-3) / 1e9
        # SURVEY 8(d): algorithmic histogram updates = one per (order, valid position)
        alg_updates = float(sum(max(int(l) - k + 1, 0) for l in wins.length for k in range(1, 9))) if n_win < 200000 else n_win * 39972.0
        n_kmers = float(sum(max(int(l) - 7, 0) for l in wins.length)) if n_win < 200000 else n_win * 4993.0
        atomic_peak = measure_smem_atomic_rate()
        gather_rand, gather_sorted = measure_l2_gather_rate(0), measure_l2_gather_rate(1)
        cap = committed_capture(kernel)
        # lower bounds on the kernel's time from the three candidate resources, each at its MEASURED rate
        t_atomic = alg_updates / atomic_peak if atomic_peak else None
        t_gather = n_kmers / gather_rand if gather_rand else None
        fp64_rate = 148 * 64 * 1.965e9                              # DFMA lanes/s: 64 per SM per clock at the maximum SM clock (nominal)
        t_fp64 = n_kmers * 42.0 / fp64_rate                          # 42 fp64 instructions per K-mer in the epilogue (SASS count, DESIGN.md)
        bounds = {"smem_atomic_s": t_atomic, "l2_gather_s": t_gather, "fp64_s": t_fp64}
        comp = max(v for v in bounds.values() if v)
        line = {
            "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u4/u16/u64 counts + f64 scores", "data": "synthetic",
            "config": dict(CONFIG),
            "run": {"bases_per_gpu": bases, "windows_per_gpu": n_win, "score_kernel": kernel, "score_kernel_occupancy": occ,
                    "parallelism": "scaffold shards x%d, %s" % (world, collective)},
            "windows_per_s": all_win * args.steps / (total_ms * 1e-3),
            "stage_ms": {"background": float(stage[:, 0].mean()), "tables+ivom(+exchange)": float(stage[:, 1].mean()),
                         "score": score_ms},
            "roofline": {
                "kernel": kernel, "bound": "smem_atomic",
                "achieved": alg_updates / (score_ms * 1e-3), "peak": atomic_peak, "unit": "updates/s",
                "frac": (alg_updates / (score_ms * 1e-3) / atomic_peak) if atomic_peak else None,
                "peak_source": "measured live: frisk_b200_bench_smem_atomics, uniformly random bins of a 64 KiB table",
                "algorithmic_updates_per_launch": alg_updates,
                "traffic": cap.get("dram_bytes") if isinstance(cap, dict) else None,
                "note": "SURVEY 8(d): the applicable bound is the lower-throughput one, the shared-memory histogram: algorithmic = one update per "
                        "(order, valid position) = 39,972 per 5 kb window.  The kernel issues ONE atomic per position (4-bit counters, orders "
                        "below K by marginalisation), so the algorithmic count overstates its atomic work 8-fold; what it is limited by is in "
                        "`limiter` and `composite`",
                "hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": peak, "peak_source": peak_kind, "unit": "GB/s", "frac": hbm_achieved / peak,
                        "algorithmic_bytes_per_launch": alg_bytes,
                        "note": "not binding: window tables never leave shared memory; every packed base is read once (traffic ~= algorithmic bytes)"},
                "composite": {"lower_bounds_ms": {k: (v * 1e3 if v else None) for k, v in bounds.items()}, "binding_ms": comp * 1e3,
                              "frac": comp * 1e3 / score_ms,
                              "l2_gather_16B_per_s": {"random": gather_rand, "sorted": gather_sorted},
                              "smem_random_loads_per_s": {"8B": measure_smem_load_rate(8), "16B": measure_smem_load_rate(16)},
                              "note": "time the kernel would need if ONLY that resource mattered, at the rate a micro-benchmark reaches on this GPU: "
                                      "algorithmic atomics; one random 16-byte gather per K-mer position from the 1 MiB genome IVOM table; 42 fp64 "
                                      "instructions per K-mer at 64 lanes/SM/clock.  frac = the largest of them / the measured kernel time"}},
            "limiter": cap,
            "e2e": {"value": (all_bases / (e2e_step_ms * 1e-3) / 1e9) if e2e_steps else None, "unit": "Gbp/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_step_ms, "steps": e2e_steps,
                    "api": "frisk_b200_run_host_sparse (C ABI, one call; pinned host planes, invalid plane as its non-zero words)" if world == 1 else ("frisk_b200_run_host_peers (C ABI, one call per rank; pinned host planes, fused peer exchange)" if pipe.peers is not None
                                else "engine.Pipeline.step_from_host (pinned host planes, NCCL all-reduce between kernels)"),
                    "stages": breakdown},
            "e2e_fasta": ({"value": all_bases / (fasta_ms * 1e-3) / 1e9, "unit": "Gbp/s", "ms_per_step": fasta_ms,
                           "h2d_bytes_per_step": fasta_bytes_n + wins.off.nbytes + wins.length.nbytes, "d2h_bytes_per_step": d2h,
                           "api": "frisk_b200_run_fasta (C ABI, one call: chunked upload of pinned FASTA text, device-side tokenise + "
                                  "layout + pack + count per chunk while the next is on the bus; genome space and window list built on the device, so tables, "
                                  "IVOM and window kernel are queued before the host has seen the record table; rows)",
                           "stages": fasta_stages}
                          if fasta_ms else None),
            "gpu_launches": pipe.launches_per_step * args.steps,
            "clocks": clocks,
            "ingest": {"device_ms": (sorted(ingest_ms)[len(ingest_ms) // 2] if ingest_ms else None),
                       "device_gbps": (bases / (sorted(ingest_ms)[len(ingest_ms) // 2] * 1e-3) / 1e9 if ingest_ms else None),
                       "host_pack_seconds": t_pack, "host_pack_gbps": bases / t_pack / 1e9,
                       "note": "device: pinned FASTA text -> H2D -> tokenise + 2-bit pack on the GPU (frisk_ingest.cu), median of 5 "
                               "wall-clock runs; host: the C++ packer used to build this bench's pinned planes (outside the timed region)"},
        }
        line.update({k: v for k, v in extra.items() if v is not None})
        if world == 1 and not args.profile:
            threads = os.cpu_count() or 1
            sample, tot_s = cpu_port_sample(scaffolds, 12.0, threads)
            t0 = time.perf_counter()
            nw = _one_cpu_pass(sample, threads)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {
                "value": tot_s / dt / 1e9, "unit": "Gbp/s", "cores": threads, "kind": "port",
                "sample": "first %d scaffolds of C2 = %d bp, %d windows (C oracle, background + all windows of the sample)" % (len(sample), tot_s, nw),
                "python_port_1core_gbps": python_port_rate(scaffolds),
            }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="frisk_b200", choices=["frisk_b200", "reference"])
    ap.add_argument("--nccl", action="store_true", help="N > 1: combine the counters with an NCCL all-reduce instead of the fused peer sum")
    ap.add_argument("--option", action="append", help="library option name=value (frisk_b200_set_option), repeatable")
    ap.add_argument("--profile", action="store_true", help="kernels only: skip the e2e, extra-block and CPU-baseline legs (for ncu)")
    ap.add_argument("--quick", action="store_true", help="skip the parity / strong / c5 / c3_sweep blocks")
    ap.add_argument("--c5", action="store_true", help="N = 1: run the c5 block too (1.75 Gbp from FASTA text)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step to DIR/<name>.npy "
                                                          "(float64), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
