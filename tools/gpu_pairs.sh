#!/bin/bash
# The nibble kernel's pair gather, against a build of the parent commit ($PARENT_LIB, a libfrisk_b200.so): the gather
# micro-benchmark (mode 7 vs mode 0), the GPU suite and smoke, outputs of both builds compared array for array
# (bench.py --quick --dump-outputs, and kmax 7 / w = 2000, 8000 through tools/nibble_pairs_ab.py), the kernel times of one
# score call, and the nibble rows of tools/k8_ab.py for both builds.  Results under OUT_DIR.
#   PARENT_LIB=path/to/parent/libfrisk_b200.so bash tools/gpu_pairs.sh OUT_DIR
O=${1:?usage: PARENT_LIB=... bash tools/gpu_pairs.sh OUT_DIR}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $O/gpu.txt
timeout 300 python tools/microbench.py pairs | tee $O/pairs_microbench.json
timeout 1500 python -m pytest tests -m gpu -q 2>&1 | tail -8 | tee $O/pytest_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
for arm in parent new; do
    lib=""; [ $arm = parent ] && lib=$PARENT_LIB
    FRISK_B200_LIB=$lib timeout 600 python bench.py --quick --steps 20 --dump-outputs $O/dump_$arm > $O/quick_$arm.json 2> $O/quick_$arm.err
    FRISK_B200_LIB=$lib timeout 600 python tools/nibble_pairs_ab.py dump $O/shapes_$arm.npz
done
python - "$O" <<'EOF'
import numpy as np, json, os, sys
O = sys.argv[1]
r = {n: bool(np.array_equal(np.load(os.path.join(O, "dump_parent", n + ".npy")), np.load(os.path.join(O, "dump_new", n + ".npy")), equal_nan=True))
     for n in ("rows", "status", "tables", "coords", "meta")}
print(json.dumps({"bench_dump_equal": r}))
for a in ("parent", "new"):
    d = json.loads(open(os.path.join(O, "quick_%s.json" % a)).read().strip().splitlines()[-1])
    print(a, "value", round(d["value"], 3), "stage_ms", {k: round(v, 4) for k, v in d["stage_ms"].items()})
EOF
python tools/nibble_pairs_ab.py compare $O/shapes_parent.npz $O/shapes_new.npz
for arm in parent new; do
    lib=""; [ $arm = parent ] && lib=$PARENT_LIB
    FRISK_B200_LIB=$lib timeout 600 python tools/nibble_pairs_ab.py profile | tee $O/profile_$arm.json
    FRISK_B200_LIB=$lib FRISK_AB_ONLY=nibble timeout 900 python tools/k8_ab.py | tee $O/k8_ab_$arm.jsonl
done
