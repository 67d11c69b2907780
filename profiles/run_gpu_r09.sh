#!/bin/bash
# Round 9 (1 GPU): one host loop and one keyed graph cache in capi.cu, against its parent commit.
# Builds, runs the whole GPU suite and smoke(), then alternates the parent and this tree: bench.py on
# the default schedule and with --schedule 0 (parent, new, new, parent), profiles/block_bench.py and
# profiles/device_solve_bench.py (parent, new; both repeat inside).  The card is read before and
# after in the same job.
#   bash profiles/run_gpu_r09.sh OUTDIR PARENT_TREE
# PARENT_TREE: a checkout of the parent commit on which __graft_entry__.build() has run.
set +e
OUT=$(realpath -m "${1:?usage: run_gpu_r09.sh OUTDIR PARENT_TREE}")
PARENT=$(realpath "${2:?usage: run_gpu_r09.sh OUTDIR PARENT_TREE}")
NEW=$(pwd)
mkdir -p "$OUT"
q() { nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,power.draw,temperature.gpu --format=csv >> "$OUT/card.csv"; }
q
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1; echo "build exit $?" >> "$OUT/build.log"
timeout 1500 python -m pytest -q -rs tests > "$OUT/pytest_gpu_g1.log" 2>&1; echo "pytest exit $?" >> "$OUT/pytest_gpu_g1.log"
timeout 300 python __graft_entry__.py smoke > "$OUT/smoke.log" 2>&1; echo "smoke exit $?" >> "$OUT/smoke.log"
run() { # run BUILD ROUND [all]
    local dir=$NEW
    [ "$1" = parent ] && dir=$PARENT
    cd "$dir" || return
    timeout 600 python bench.py --gpus 1 --steps 200 --warmup 10 > "$OUT/bench_$1_default_$2.json" 2> "$OUT/bench_$1_default_$2.err"
    timeout 600 python bench.py --gpus 1 --steps 200 --warmup 10 --schedule 0 > "$OUT/bench_$1_schedule0_$2.json" 2> "$OUT/bench_$1_schedule0_$2.err"
    [ "$3" = all ] || { cd "$NEW"; return; }
    timeout 600 python profiles/block_bench.py --sizes 40000,1000000 --nrhs 1,8 > "$OUT/block_bench_$1_$2.jsonl" 2>&1
    timeout 900 python profiles/device_solve_bench.py > "$OUT/device_solve_bench_$1_$2.jsonl" 2>&1
    cd "$NEW"
}
run parent 1 all
run new 1 all
run new 2
run parent 2
q
echo done > "$OUT/done.txt"
