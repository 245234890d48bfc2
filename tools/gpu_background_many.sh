#!/bin/bash
# One query against several stored backgrounds on one B200: build, then the steps named in $2 (default: all) with their logs
# in $1 --
#   tests   tests/test_background_many_gpu.py and tests/test_background_gpu.py
#   timing  tools/background_many_timing.py (fused call against the loop of Background.run, B = 1, 2, 4, 8)
#   suite   the whole GPU suite
#   smoke   __graft_entry__.smoke()
#   bench   bench.py --gpus 1 --steps 50 --warmup 5
set -u
OUT=${1:?usage: tools/gpu_background_many.sh OUT_DIR [STEPS]}
STEPS=${2:-"tests timing suite smoke bench"}
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT/build.log" 2>&1 || { tail -50 "$OUT/build.log"; exit 1; }
for s in $STEPS; do
    case $s in
        tests) python -m pytest -q -m gpu tests/test_background_many_gpu.py tests/test_background_gpu.py > "$OUT/pytest_background_many.log" 2>&1 ;;
        timing) python tools/background_many_timing.py --out "$OUT/r08_background_many_timing.json" > "$OUT/timing.log" 2>&1 ;;
        suite) python -m pytest -q -m gpu > "$OUT/pytest_gpu.log" 2>&1 ;;
        smoke) python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT/smoke.log" 2>&1 ;;
        bench) python bench.py --gpus 1 --steps 50 --warmup 5 > "$OUT/bench.log" 2>&1 ;;
    esac
    echo "$s: exit $?"
done
for f in "$OUT"/*.log; do echo "== $f"; tail -15 "$f"; done
