#!/bin/bash
# One B200 visit for the stage-by-stage Jacobi-PCG checks: card, error / bound spread (pcg_stage_spread.py), the new test
# file, the whole GPU suite and smoke().  Everything it writes goes under OUTDIR.
#     bash scripts/pcg_stage_gpu.sh OUTDIR
set -x
O=${1:?usage: pcg_stage_gpu.sh OUTDIR}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/pcg_gpu.csv; cat $O/pcg_gpu.csv
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1; echo "build exit $?"
timeout 900 python scripts/pcg_stage_spread.py > $O/pcg_stage_spread.jsonl 2> $O/pcg_stage_spread.err; echo "spread exit $?"; tail -1 $O/pcg_stage_spread.jsonl; tail -3 $O/pcg_stage_spread.err
timeout 1500 python -m pytest tests/test_gpu_pcg_stages.py -q -m gpu -p no:cacheprovider -rf --durations=8 > $O/pcg_pytest_new.txt 2>&1; echo "new tests exit $?"; tail -25 $O/pcg_pytest_new.txt
timeout 1800 python -m pytest tests -q -m gpu -p no:cacheprovider --ignore=tests/test_gpu_pcg_stages.py > $O/pcg_pytest_gpu.txt 2>&1; echo "pytest exit $?" >> $O/pcg_pytest_gpu.txt
tail -8 $O/pcg_pytest_gpu.txt
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $O/pcg_smoke.log 2>&1; echo "smoke exit $?"; tail -2 $O/pcg_smoke.log
