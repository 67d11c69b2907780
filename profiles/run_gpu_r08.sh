#!/bin/bash
# Round 8 (1 GPU): build, the whole GPU suite, smoke(), bench.py once (default dense path), then
# profiles/device_solve_bench.py; the card is read before and after in the same job.
#   bash profiles/run_gpu_r08.sh OUTDIR      (every log and result goes under OUTDIR)
set +e
OUT=${1:?usage: run_gpu_r08.sh OUTDIR}
mkdir -p "$OUT"
q() { nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,power.draw,temperature.gpu --format=csv >> $OUT/card.csv; }
q
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1; echo "build exit $?" >> $OUT/build.log
cp conjugate-gradient_b200/csrc/_build/loop.ptxas.log conjugate-gradient_b200/csrc/_build/capi.ptxas.log $OUT/ 2>/dev/null
timeout 600 python -m pytest -q -rs -x tests/test_gpu_device_solve.py > $OUT/pytest_device_solve_g1.log 2>&1; echo "pytest exit $?" >> $OUT/pytest_device_solve_g1.log
timeout 1500 python -m pytest -q -rs tests > $OUT/pytest_gpu_g1.log 2>&1; echo "pytest exit $?" >> $OUT/pytest_gpu_g1.log
timeout 300 python __graft_entry__.py smoke > $OUT/smoke.log 2>&1; echo "smoke exit $?" >> $OUT/smoke.log
timeout 600 python bench.py --gpus 1 --steps 200 --warmup 10 > $OUT/bench_g1.json 2> $OUT/bench_g1.err; echo "bench exit $?" >> $OUT/bench_g1.err
timeout 900 python profiles/device_solve_bench.py --out $OUT > $OUT/device_solve_bench.log 2>&1; echo "device_solve_bench exit $?" >> $OUT/device_solve_bench.log
q
echo done > $OUT/done.txt
