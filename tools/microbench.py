"""Roofline denominators measured on the GPU at hand: shared-memory atomics, random shared-memory loads, random and
sorted 16-byte gathers from an L2-resident 1 MiB table (frisk_b200_bench_*).  One JSON line."""
import ctypes as C
import json
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from frisk_b200 import _lib

L = _lib.lib()
L.frisk_b200_last_cuda_error.restype = C.c_char_p
_lib.require_device()


def best(fn, n=3):
    return max(fn() for _ in range(n))


def atomics(mode):
    ms = C.c_float(0)
    blocks, iters = 148 * 2, 4096 if mode < 2 else 512
    _lib.check(L.frisk_b200_bench_smem_atomics(blocks, iters, mode, C.byref(ms), None), "bench_smem_atomics")
    return blocks * 1024 * iters / (ms.value * 1e-3)


def gathers(mode, table_bytes=1 << 20):
    ms = C.c_float(0)
    blocks, iters = 148 * 4, 2048
    _lib.check(L.frisk_b200_bench_l2_gather(blocks, iters, table_bytes, mode, C.byref(ms), None), "bench_l2_gather")
    return blocks * 256 * iters / (ms.value * 1e-3)


def loads(nbytes):
    ms = C.c_float(0)
    blocks, iters = 148 * 4, 8192
    _lib.check(L.frisk_b200_bench_smem_loads(blocks, iters, nbytes, C.byref(ms), None), "bench_smem_loads")
    return blocks * 256 * iters / (ms.value * 1e-3)


def gather4(mode):
    ms = C.c_float(0)
    blocks, iters = 148 * 4, 2048
    rc = L.frisk_b200_bench_l2_gather(blocks, iters, 1 << 20, mode, C.byref(ms), None)
    return blocks * 256 * iters / (ms.value * 1e-3) if rc == 0 else "rc=%d (%s)" % (rc, L.frisk_b200_strerror(rc).decode())


if len(sys.argv) > 1 and sys.argv[1] == "tex":
    print(json.dumps({"l2_gather_16B_per_s": {"ldg_random_1MiB": best(lambda: gathers(0)), "tex1Dfetch_random_1MiB": best(lambda: gathers(6)),
                                              "ldg_random_64KiB": best(lambda: gathers(0, 1 << 16)),
                                              "tex1Dfetch_random_64KiB": best(lambda: gathers(6, 1 << 16))}}))
    sys.exit(0)
if len(sys.argv) > 1 and sys.argv[1] == "pairs":
    # the nibble kernel's pair gather: one 256-bit load of a 32-byte entry out of the (K+1)-mer pair table (8 MiB at K = 8,
    # 2 MiB at K = 7) against today's 16-byte gather from the 1 MiB genome-IVOM table; the three alternate, 7 rounds
    import subprocess
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    legs = {"mode0_16B_1MiB": (0, 1 << 20), "mode7_32B_8MiB": (7, 1 << 23), "mode7_32B_2MiB": (7, 1 << 21)}
    runs = {k: [] for k in legs}
    for _ in range(7):
        for k, (mode, nbytes) in legs.items():
            runs[k].append(gathers(mode, nbytes))
    med = {k: sorted(v)[len(v) // 2] for k, v in runs.items()}
    print(json.dumps({"gpu": q.stdout.strip() if q.returncode == 0 else "not available",
                      "gathers_per_s_median": med, "gathers_per_s_runs": runs,
                      "ratio_to_mode0": {k: med[k] / med["mode0_16B_1MiB"] for k in med},
                      "note": "requests (one entry per lane) per second, 148 x 4 CTAs of 256 threads, 2,048 loads per thread, "
                              "uniformly random entries; mode 0 is __ldg of 16 B, mode 7 ld.global.cg.v4.f64 of 32 B"}))
    sys.exit(0)
if len(sys.argv) > 1 and sys.argv[1] == "gather4":
    # (probed and removed: a tensor-map box of 4 rows is rejected, and destinations that are only 64- or 80-byte aligned
    # fault with cudaErrorMisalignedAddress: every gather4 needs a 128-byte aligned 64-byte landing slot)
    r = {"box_rows_1": gather4(5)}
    print(json.dumps({"tma_gather4_rows_per_s": r}))
    sys.exit(0)

out = {
    "smem_atomic_updates_per_s": {n: best(lambda m=m: atomics(m)) for m, n in [(0, "conflict_free"), (1, "random"), (2, "single_address")]},
    "smem_random_loads_per_s": {"%dB" % b: best(lambda b=b: loads(b)) for b in (4, 8, 16)},
    "l2_gather_16B_per_s": {"random_1MiB": best(lambda: gathers(0)), "sorted_1MiB": best(lambda: gathers(1)),
                            "random_256KiB": best(lambda: gathers(0, 1 << 18)), "random_16MiB": best(lambda: gathers(0, 1 << 24)),
                            "random_1MiB_cp_async": best(lambda: gathers(2)), "random_8B_entries_512KiB": best(lambda: gathers(3)), "random_1MiB_cp_async_bulk": best(lambda: gathers(4))},
}
print(json.dumps(out))
