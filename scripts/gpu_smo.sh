#!/bin/bash
# SMO (K11) evidence on one B200: build, the GPU suite, smoke, the default bench line, the grid-size sweep and the
# bench_smo configs, written to the directory given as the first argument (SMO_SWEEP=0 skips the sweep).
set -u
cd "$(dirname "$0")/.."
OUT="${1:?usage: scripts/gpu_smo.sh OUTPUT_DIR}"
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1
python -c "import __graft_entry__ as e; print(e.build())" > $OUT/build.log 2>&1 || { cat $OUT/build.log; exit 1; }
python -m pytest tests -q -m gpu -p no:cacheprovider > $OUT/pytest_gpu.log 2>&1; echo "pytest exit $?" >> $OUT/pytest_gpu.log
tail -3 $OUT/pytest_gpu.log
python -c "import __graft_entry__ as e; e.smoke()" > $OUT/smoke.log 2>&1; echo "smoke exit $?" >> $OUT/smoke.log
tail -2 $OUT/smoke.log
python bench.py --gpus 1 --steps 3 --warmup 3 > $OUT/bench_n1.json 2> $OUT/bench_n1.err; tail -c 400 $OUT/bench_n1.json
if [ "${SMO_SWEEP:-1}" = 1 ]; then
  for g in 148 74 37 16; do
    python scripts/bench_smo.py --configs C1,C4 --no-sklearn --grid $g >> $OUT/smo_grid_sweep.jsonl 2>> $OUT/smo.err
  done
  cut -c1-300 $OUT/smo_grid_sweep.jsonl
fi
python scripts/bench_smo.py --configs C1,C4,C2 >> $OUT/smo_bench.jsonl 2>> $OUT/smo.err
cat $OUT/smo_bench.jsonl; tail -5 $OUT/smo.err
