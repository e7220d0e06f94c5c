#!/bin/bash
# One B200 visit for the x ring of the fused Jacobi-PCG (FI_B200_X_RING): card, spread of two m = 2 solves on the test
# lattices, bench default against m = 2 alternated three times (with --dump-outputs), fp64 bench both ways, per-form
# update timings, the whole GPU suite and smoke().  Everything it writes goes under the directory given as its argument.
#     bash scripts/x_ring_gpu.sh OUTDIR
set -x
O=${1:?usage: x_ring_gpu.sh OUTDIR}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/x_ring_gpu.csv; cat $O/x_ring_gpu.csv
timeout 300 python scripts/x_ring_spread.py > $O/x_ring_spread.jsonl 2> $O/x_ring_spread.err; grep summary $O/x_ring_spread.jsonl; tail -3 $O/x_ring_spread.err
for k in 1 2 3; do
  FI_B200_X_RING=2 timeout 400 python bench.py --no-cpu-baseline --dump-outputs $O/dump_m2_$k > $O/x_ring_bench_m2_$k.json 2> $O/x_ring_bench_m2_$k.err
  timeout 400 python bench.py --no-cpu-baseline --dump-outputs $O/dump_def_$k > $O/x_ring_bench_default_$k.json 2> $O/x_ring_bench_default_$k.err
done
python scripts/x_ring_compare.py $O
for k in 1 2; do
  FI_B200_X_RING=2 timeout 300 python bench.py --no-cpu-baseline --no-configs --no-time-to-tol --precision f64 > $O/x_ring_bench_f64_m2_$k.json 2> $O/x_ring_bench_f64_m2_$k.err
  timeout 300 python bench.py --no-cpu-baseline --no-configs --no-time-to-tol --precision f64 > $O/x_ring_bench_f64_default_$k.json 2> $O/x_ring_bench_f64_default_$k.err
done
python scripts/x_ring_compare.py $O f64
timeout 600 python scripts/time_x_ring.py > $O/x_ring_time.jsonl 2> $O/x_ring_time.err; cat $O/x_ring_time.jsonl | cut -c 1-400; tail -3 $O/x_ring_time.err
timeout 1200 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/x_ring_pytest_gpu.txt 2>&1; echo "pytest exit $?" >> $O/x_ring_pytest_gpu.txt
tail -8 $O/x_ring_pytest_gpu.txt
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > $O/x_ring_smoke.log 2>&1; echo "smoke exit $?"; tail -2 $O/x_ring_smoke.log
