#!/bin/bash
# One B200 visit for the stage-by-stage multigrid checks: card, fp32-vs-fp64 spread of the smoother and the cycle
# (mg_operator_spread.py), the new test file, the whole GPU suite, smoke(), and bench.py alternated with the tree at BASE
# (built there first) when one is given.  Everything it writes goes under OUTDIR.
#     bash scripts/mg_operator_gpu.sh OUTDIR [BASE]
set -x
O=${1:?usage: mg_operator_gpu.sh OUTDIR [BASE]}
BASE=$2
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/mg_gpu.csv; cat $O/mg_gpu.csv
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1; echo "build exit $?"
if [ -n "$BASE" ]; then (cd $BASE && python -c "import __graft_entry__ as g; g.build()") > $O/build_base.log 2>&1; echo "base build exit $?"; fi
timeout 600 python scripts/mg_operator_spread.py > $O/mg_operator_spread.jsonl 2> $O/mg_operator_spread.err; tail -1 $O/mg_operator_spread.jsonl; tail -3 $O/mg_operator_spread.err
timeout 1500 python -m pytest tests/test_gpu_multigrid_operator.py -q -m gpu -p no:cacheprovider -rf > $O/mg_pytest_new.txt 2>&1; echo "new tests exit $?"; tail -12 $O/mg_pytest_new.txt
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_multigrid_operator.py > $O/mg_pytest_gpu.txt 2>&1; echo "pytest exit $?" >> $O/mg_pytest_gpu.txt
tail -8 $O/mg_pytest_gpu.txt
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $O/mg_smoke.log 2>&1; echo "smoke exit $?"; tail -2 $O/mg_smoke.log
for k in 1 2; do
  if [ -n "$BASE" ]; then (cd $BASE && timeout 500 python bench.py --gpus 1 --no-cpu-baseline) > $O/bench_base_$k.json 2> $O/bench_base_$k.err; tail -c 1500 $O/bench_base_$k.json; fi
  timeout 500 python bench.py --gpus 1 --no-cpu-baseline > $O/bench_new_$k.json 2> $O/bench_new_$k.err; tail -c 1500 $O/bench_new_$k.json
done
