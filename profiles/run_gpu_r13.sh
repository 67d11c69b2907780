#!/bin/bash
# Round 13 (1 GPU): one COO staging pipeline for cgb_set_matrix_coo (last-write fold) and cgb_assemble_coo (sum
# fold).  Reads the card before and after, builds, keeps the ptxas reports of spmv.cu and capi.cu, runs the whole
# GPU suite and smoke(), then profiles/build_bench.py against the parent's library (4 rounds), then alternates
# profiles/assemble_bench.py and bench.py of the parent tree and this one (two rounds of parent, new, new,
# parent each: same bits, same speed).
#   bash profiles/run_gpu_r13.sh OUTDIR PARENT_TREE
# PARENT_TREE: a checkout of the parent commit on which __graft_entry__.build() has run; its libcgb200.so is also
# copied to profiles/_parent/ as build_bench.py's docstring says.
set +e
OUT=$(realpath -m "${1:?usage: run_gpu_r13.sh OUTDIR PARENT_TREE}")
PARENT=$(realpath "${2:?usage: run_gpu_r13.sh OUTDIR PARENT_TREE}")
NEW=$(pwd)
mkdir -p "$OUT/ptxas"
q() { nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,power.draw,temperature.gpu --format=csv >> "$OUT/card.csv"; }
q
NGPU=$(nvidia-smi -L | wc -l)
echo "gpus $NGPU" >> "$OUT/card.csv"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1; echo "build exit $?" >> "$OUT/build.log"
cp conjugate-gradient_b200/csrc/_build/spmv.ptxas.log conjugate-gradient_b200/csrc/_build/capi.ptxas.log "$OUT/ptxas/"
timeout 1500 python -m pytest -q -rs --durations=15 tests > "$OUT/pytest_gpu_g1.log" 2>&1; echo "pytest exit $?" >> "$OUT/pytest_gpu_g1.log"
timeout 300 python __graft_entry__.py smoke > "$OUT/smoke.log" 2>&1; echo "smoke exit $?" >> "$OUT/smoke.log"
timeout 1800 python profiles/build_bench.py --rounds 4 --out "$OUT" > "$OUT/build_bench.log" 2>&1
echo "build_bench exit $?" >> "$OUT/build_bench.log"
asm() { # asm BUILD ROUND
    local dir=$NEW
    [ "$1" = parent ] && dir=$PARENT
    mkdir -p "$OUT/assemble_$1_$2"
    (cd "$dir" && timeout 1200 python profiles/assemble_bench.py --out "$OUT/assemble_$1_$2" > "$OUT/assemble_$1_$2/log" 2>&1
     echo "assemble_bench exit $?" >> "$OUT/assemble_$1_$2/log")
}
for r in 1 2; do
    asm parent "${r}a"
    asm new "${r}a"
    asm new "${r}b"
    asm parent "${r}b"
done
bench() { # bench BUILD ROUND
    local dir=$NEW
    [ "$1" = parent ] && dir=$PARENT
    (cd "$dir" && timeout 600 python bench.py --gpus 1 --steps 200 --warmup 10 > "$OUT/bench_$1_$2.json" 2> "$OUT/bench_$1_$2.err")
}
for r in 1 2; do
    bench parent "${r}a"
    bench new "${r}a"
    bench new "${r}b"
    bench parent "${r}b"
done
q
echo done > "$OUT/done.txt"
