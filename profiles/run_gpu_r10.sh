#!/bin/bash
# Round 10 (1 GPU): matrices from device memory (cgb_set_matrix_csr) and value refreshes
# (cgb_update_matrix_values).  Builds, keeps the ptxas report of spmv.cu (the new kernels), runs the whole
# GPU suite and smoke(), alternates bench.py of the parent and this tree (parent, new, new, parent: the
# default dense path must keep its digest and its speed), then profiles/matrix_update_bench.py.  The card
# is read before and after in the same job.
#   bash profiles/run_gpu_r10.sh OUTDIR PARENT_TREE
# PARENT_TREE: a checkout of the parent commit on which __graft_entry__.build() has run.
set +e
OUT=$(realpath -m "${1:?usage: run_gpu_r10.sh OUTDIR PARENT_TREE}")
PARENT=$(realpath "${2:?usage: run_gpu_r10.sh OUTDIR PARENT_TREE}")
NEW=$(pwd)
mkdir -p "$OUT/ptxas"
q() { nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,power.draw,temperature.gpu --format=csv >> "$OUT/card.csv"; }
q
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1; echo "build exit $?" >> "$OUT/build.log"
cp conjugate-gradient_b200/csrc/_build/spmv.ptxas.log conjugate-gradient_b200/csrc/_build/capi.ptxas.log "$OUT/ptxas/"
timeout 1500 python -m pytest -q -rs --durations=15 tests > "$OUT/pytest_gpu_g1.log" 2>&1; echo "pytest exit $?" >> "$OUT/pytest_gpu_g1.log"
timeout 300 python __graft_entry__.py smoke > "$OUT/smoke.log" 2>&1; echo "smoke exit $?" >> "$OUT/smoke.log"
bench() { # bench BUILD ROUND
    local dir=$NEW
    [ "$1" = parent ] && dir=$PARENT
    (cd "$dir" && timeout 600 python bench.py --gpus 1 --steps 200 --warmup 10 > "$OUT/bench_$1_$2.json" 2> "$OUT/bench_$1_$2.err")
}
bench parent 1
bench new 1
bench new 2
bench parent 2
timeout 900 python profiles/matrix_update_bench.py --out "$OUT" --steps 10 --repeats 3 > "$OUT/matrix_update_bench.log" 2>&1
echo "matrix_update_bench exit $?" >> "$OUT/matrix_update_bench.log"
q
echo done > "$OUT/done.txt"
