#!/bin/bash
# Scoring visit (one GPU): parity tests of the scoring paths, the cfg3 micro-benchmark in every mode, and full ncu
# captures (raw + source pages) of the tensor-core kernel.  TAG names the output directory under gpurun_out/.
#   NCU_MODES="matrix_lm topk both_lm"  NCU_DIMS="10"  VARIANTS="name:-DFLAG ..." (rebuild lec_score_mma.o and re-time)
set -u
TAG=${TAG:-r2s}
O=gpurun_out/$TAG
mkdir -p $O
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $O/gpu.txt 2>&1
if [ "${PYTEST:-1}" = "1" ]; then
  timeout 900 python -m pytest tests -m gpu -q --no-header -p no:cacheprovider -k "scor or smoke or classif or pipeline" > $O/pytest_score.log 2>&1
  echo "pytest exit $?" >> $O/pytest_score.log
  tail -8 $O/pytest_score.log
fi
timeout 300 python scripts/score_bench.py --dims ${DIMS:-10,50} --iters 9 --modes ${MODES:-topk,matrix_lm,both_lm} --engines tc > $O/score_bench.log 2>&1
cat $O/score_bench.log
for spec in ${VARIANTS:-}; do
  name=${spec%%:*}; flags=${spec#*:}
  rm -f learning_embeddings_b200/csrc/build/lec_score_mma.o
  make -C learning_embeddings_b200/csrc EXTRA="$(echo $flags | tr ',' ' ')" > $O/make_$name.log 2>&1 || { tail -5 $O/make_$name.log; continue; }
  timeout 300 python scripts/score_bench.py --dims ${DIMS:-10,50} --iters 9 --modes ${MODES:-topk,matrix_lm,both_lm} --engines tc > $O/score_bench_$name.log 2>&1
  echo "== variant $name ($flags)"; cat $O/score_bench_$name.log
done
if [ -n "${VARIANTS:-}" ]; then
  rm -f learning_embeddings_b200/csrc/build/lec_score_mma.o
  make -C learning_embeddings_b200/csrc > $O/make_restore.log 2>&1
fi
for D in ${NCU_DIMS-10}; do
  # score_bench runs 2 warm-up + 1 timed launch per mode: launch 2 of the kernel is the timed one
  for m in ${NCU_MODES-matrix_lm}; do
    timeout 300 ncu --set full --clock-control none --import-source on -k regex:score_mma_kernel -s 2 -c 1 -o /tmp/prof_tc_d${D}_$m \
        python scripts/score_bench.py --images 303104 --dims $D --iters 1 --modes $m --engines tc > $O/ncu_tc_d${D}_$m.log 2>&1
    ncu -i /tmp/prof_tc_d${D}_$m.ncu-rep --page raw --csv > $O/tc_d${D}_${m}_raw.csv 2>/dev/null
    ncu -i /tmp/prof_tc_d${D}_$m.ncu-rep --page source --csv > $O/tc_d${D}_${m}_source.csv 2>/dev/null
  done
done
