#!/bin/bash
# Scoring against a stored background on one B200: build, then the steps named in $2 (default: all) with their logs in $1 --
#   tests   tests/test_background_gpu.py
#   timing  tools/background_timing.py (C4 stand-in host, C2 and C1 queries, text and .2bit; the CLI with and without pickle)
#   suite   the whole GPU suite
#   smoke   __graft_entry__.smoke()
#   bench   bench.py --gpus 1 --steps 50 --warmup 5
set -u
OUT=${1:?usage: tools/gpu_background.sh OUT_DIR [STEPS]}
STEPS=${2:-"tests timing suite smoke bench"}
mkdir -p "$OUT"
python -c 'import __graft_entry__ as g; g.build()' > "$OUT/build.log" 2>&1 || { tail -50 "$OUT/build.log"; exit 1; }
for s in $STEPS; do
    case $s in
        tests) python -m pytest -q -m gpu tests/test_background_gpu.py > "$OUT/pytest_background.log" 2>&1 ;;
        timing) python tools/background_timing.py --out "$OUT/r07_background_timing.json" > "$OUT/timing.log" 2>&1 ;;
        suite) python -m pytest -q -m gpu > "$OUT/pytest_gpu.log" 2>&1 ;;
        smoke) python -c 'import __graft_entry__ as g; g.smoke()' > "$OUT/smoke.log" 2>&1 ;;
        bench) python bench.py --gpus 1 --steps 50 --warmup 5 > "$OUT/bench.log" 2>&1 ;;
    esac
    echo "$s: exit $?"
done
for f in "$OUT"/*.log; do echo "== $f"; tail -15 "$f"; done
