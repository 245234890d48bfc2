"""Outputs and kernel times of the nibble window kernel on C2 (40 Mbp, seed 2002) beyond bench.py's shape, for an A/B of
two builds (FRISK_B200_LIB selects the library):

    python tools/nibble_pairs_ab.py dump OUT.npz       rows + status of frisk_b200_score for kmax 8 / 7 at w = 5000, 2000,
                                                       8000 (the default kernel: nibble), NaN-aware comparable
    python tools/nibble_pairs_ab.py compare A.npz B.npz   np.array_equal on every array; exit 1 on a difference
    python tools/nibble_pairs_ab.py profile            torch.profiler: mean device time of every kernel of one
                                                       frisk_b200_score call (kmax 8, w = 5000), L2 flushed between calls
One JSON line per command."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

SHAPES = ((5000, 2500), (2000, 1000), (8000, 4000))


def _setup():
    import torch
    from frisk_b200 import engine, synth
    g = engine.PackedGenome.from_scaffolds(synth.make("C2", 1.0, seed=2002))
    dq = engine.DeviceGenome(g)
    d_tables, _ = engine.finalize(engine.background(dq, 8), 8)
    return torch, engine, g, dq, d_tables


def _score(torch, engine, g, dq, d_tables, w, step, k):
    from frisk_b200 import _lib
    wins = g.windows(w, step, False)
    n = len(wins)
    d_off = torch.from_numpy(wins.off.view(np.int64)).cuda()
    d_len = torch.from_numpy(wins.length.view(np.int32)).cuda()
    d_ig = engine.genome_ivom(d_tables[:_lib.table_size(1, k)], 1, k, g.genome_space)
    d_rows = torch.empty((n, 5), dtype=torch.float64, device="cuda")
    d_status = torch.empty(n, dtype=torch.int32, device="cuda")
    P = engine._ptr

    def call():
        _lib.check(_lib.lib().frisk_b200_score(P(dq.codes), P(dq.inv), P(dq.low), P(d_off), P(d_len), n, wins.max_len, P(d_ig), 1, k,
                                               1, P(d_rows), P(d_status), None, engine._stream_ptr(dq.device)), "score")
    return call, d_rows, d_status


def dump(path):
    torch, engine, g, dq, d_tables = _setup()
    out = {}
    for w, step in SHAPES:
        for k in (8, 7):
            call, d_rows, d_status = _score(torch, engine, g, dq, d_tables, w, step, k)
            call()
            torch.cuda.synchronize()
            out["rows_w%d_k%d" % (w, k)] = d_rows.cpu().numpy()
            out["status_w%d_k%d" % (w, k)] = d_status.cpu().numpy()
    np.savez(path, **out)
    print(json.dumps({"dumped": path, "arrays": len(out)}))


def compare(a, b):
    za, zb = np.load(a), np.load(b)
    res = {k: bool(np.array_equal(za[k], zb[k], equal_nan=k.startswith("rows"))) for k in za.files}
    res["same_keys"] = sorted(za.files) == sorted(zb.files)
    print(json.dumps({"equal": all(res.values()), "arrays": res}))
    return 0 if all(res.values()) else 1


def profile():
    torch, engine, g, dq, d_tables = _setup()
    call, _, _ = _score(torch, engine, g, dq, d_tables, 5000, 2500, 8)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    reps = 20
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            flush.fill_(1)
            call()
        torch.cuda.synchronize()
    times = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "fill" not in e.name and "elementwise" not in e.name:
            times.setdefault(e.name, []).append(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total)
    print(json.dumps({"kernels_us_mean": {k: float(np.mean(v)) for k, v in times.items()}, "calls": reps,
                      "gpu": torch.cuda.get_device_name(0), "note": "kmax 8, w = 5000, C2; L2 flushed before every call"}))


if __name__ == "__main__":
    cmd = sys.argv[1]
    if cmd == "dump":
        dump(sys.argv[2])
    elif cmd == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        profile()
