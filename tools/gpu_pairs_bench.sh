#!/bin/bash
# Speed A/B of two builds: full bench.py --steps 100 runs, parent ($PARENT_LIB) and this tree alternately, three each, one
# JSON line per run appended to OUT_DIR/bench_ab.jsonl with the arm and the card in front.
#   PARENT_LIB=path/to/parent/libfrisk_b200.so bash tools/gpu_pairs_bench.sh OUT_DIR
O=${1:?usage: PARENT_LIB=... bash tools/gpu_pairs_bench.sh OUT_DIR}
mkdir -p $O
gpu=$(nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | head -1)
echo "$gpu"
timeout 300 python -m pytest tests/test_nibble_pairs_gpu.py -q 2>&1 | tail -3
for i in 1 2 3; do
    for arm in parent new; do
        lib=""; [ $arm = parent ] && lib=$PARENT_LIB
        line=$(FRISK_B200_LIB=$lib timeout 170 python bench.py --gpus 1 --steps 100 --warmup 3 2> $O/bench_${arm}_$i.err | tail -1)
        python -c "import json,sys; d=json.loads(sys.argv[3]); print(json.dumps({'arm': sys.argv[1], 'gpu': sys.argv[2], **d}))" \
            "$arm" "$gpu" "$line" >> $O/bench_ab.jsonl || echo "run $arm $i failed: $(tail -2 $O/bench_${arm}_$i.err)"
        python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().splitlines()[-1]); g=lambda b: (b or {}).get('value'); print(d['arm'], round(d['value'], 3), 'score', round(d['stage_ms']['score'], 4), 'e2e', g(d.get('e2e')), 'e2e_fasta', g(d.get('e2e_fasta')), 'strong', g(d.get('strong')), 'c3', g(d.get('c3_sweep')))" $O/bench_ab.jsonl
    done
done
