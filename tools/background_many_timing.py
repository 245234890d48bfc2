"""One query against B stored backgrounds in one call (engine.run_backgrounds, frisk_b200_background_run_many) against
the loop of one Background.run per background, on one GPU, seeded inputs generated in the run:

  backgrounds  8, from distinct seeded C2-sized hosts (synth "C2", seeds 101..108), opened once, outside the timed calls
  queries      synth.config_c2() (40 Mbp) as FASTA text and as .2bit; the C4 stand-in of synth_device (3 Gbp) as .2bit;
               page-locked
  arms         for B = 1, 2, 4, 8: the fused call over the first B backgrounds against the loop over the same B; median of
               --reps calls each, alternating, both warmed up first, row buffers reused; every pair's rows and status
               compared bit for bit (block b of the fused call against background b's own call)
  stages       the window-kernel stage (ms[3] - ms[5] of frisk_b200_last_run_timing): of the fused call, and summed over
               the loop's calls

The card's name and power limit come from the same run.  Writes one JSON file (--out).

    python tools/background_many_timing.py --out profiles/r08_background_many_timing.json
"""
from __future__ import annotations

import argparse
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
from background_timing import marks  # noqa: E402
from bgzf_timing import device_info, pinned  # noqa: E402

COUNTS = (1, 2, 4, 8)


def kernel_ms() -> float:
    m = marks()
    return float(m[3] - m[5])


def compare(kind: str, bgs, query: np.ndarray, reps: int) -> dict:
    probe = bgs[0].run(query, kind=kind, assemble_result=False)
    n = int(probe.n_win)
    cap = n + 64
    res = {"windows": n, "by_backgrounds": {}}
    for nb in COUNTS:
        sub = bgs[:nb]
        out_many = engine.HostOutputs(nb * cap, 0)
        outs = [engine.HostOutputs(cap, 0) for _ in sub]

        def fused():
            engine.run_backgrounds(sub, query, kind=kind, out=out_many, assemble_result=False)
            return kernel_ms()

        def loop():
            k = 0.0
            for bg, o in zip(sub, outs):
                bg.run(query, kind=kind, out=o, assemble_result=False)
                k += kernel_ms()
            return k

        for _ in range(2):
            fused()
            loop()
        times = {"fused": [], "loop": []}
        kern = {"fused": [], "loop": []}
        identical = True
        for _ in range(reps):
            for name, f in (("fused", fused), ("loop", loop)):
                t0 = time.perf_counter()
                k = f()
                times[name].append((time.perf_counter() - t0) * 1e3)
                kern[name].append(k)
            for b in range(nb):
                identical &= bool(np.array_equal(out_many.rows[b * cap:b * cap + n], outs[b].rows[:n], equal_nan=True) and
                                  np.array_equal(out_many.status[b * cap:b * cap + n], outs[b].status[:n]))
        r = {"rows_identical_every_pair": identical,
             "call_ms": {k: {"median": float(np.median(v)), "min": float(min(v)), "all": v} for k, v in times.items()},
             "window_kernel_stage_ms": {k: float(np.median(v)) for k, v in kern.items()}}
        r["loop_over_fused"] = r["call_ms"]["loop"]["median"] / r["call_ms"]["fused"]["median"]
        res["by_backgrounds"][str(nb)] = r
        print(kind, nb, "identical:", identical, "median ms fused / loop: %.3f / %.3f" % (r["call_ms"]["fused"]["median"],
              r["call_ms"]["loop"]["median"]), "kernel stage:", r["window_kernel_stage_ms"], flush=True)
    return res


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--skip-c4", action="store_true")
    a = ap.parse_args(argv)
    import torch  # noqa: F401  (page-locked row buffers)
    _lib.require_device()
    res = {"info": device_info(), "backgrounds": "8 x synth C2 (40 Mbp), seeds 101..108, kmin 1, kmax 8",
           "pair_table_bytes_per_background": 32 * 4 ** 9}
    bgs = [engine.Background.from_result(engine.run_fasta(synth.fasta_bytes(synth.make("C2", 1.0, seed=101 + i))))
           for i in range(8)]
    c2 = synth.config_c2()
    queries = [("c2_text", "text", lambda: pinned(synth.fasta_bytes(c2))), ("c2_2bit", "2bit", lambda: pinned(synth.twobit_bytes(c2)))]
    if not a.skip_c4:
        def c4():
            from frisk_b200.synth_device import build_device_genome, c4_spec
            from test_twobit_gpu import planes_to_2bit
            lens, runs = c4_spec()
            dg = build_device_genome(engine, lens, runs, seed=44, at_rich_block=300_000 // 16)
            buf = pinned(planes_to_2bit(dg, runs).tobytes())
            del dg
            torch.cuda.empty_cache()
            return buf
        queries.append(("c4_2bit", "2bit", c4))
    for name, kind, make in queries:
        q = make()
        res[name] = {"query_bytes": int(q.shape[0]), **compare(kind, bgs, q, a.reps)}
        del q
    for bg in bgs:
        bg.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(res["info"])


if __name__ == "__main__":
    main()
