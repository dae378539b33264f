#!/bin/bash
# SMO computed rows (K12) evidence on one B200: build (ptxas lines of both SMO instantiations), the GPU suite, smoke, the
# default bench line, C4 resident vs computed (default cache and cache 0), and C5-shaped fits at n = 200 000 and 500 000
# that only the computed form runs -- written to the directory given as the first argument.
set -u
cd "$(dirname "$0")/.."
OUT="${1:?usage: scripts/gpu_smo_rows.sh OUTPUT_DIR}"
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1
python -c "import __graft_entry__ as e; print(e.build())" > $OUT/build.log 2>&1 || { cat $OUT/build.log; exit 1; }
timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider -rA -s > $OUT/pytest_gpu.log 2>&1; echo "pytest exit $?" >> $OUT/pytest_gpu.log
tail -3 $OUT/pytest_gpu.log
python -c "import __graft_entry__ as e; e.smoke()" > $OUT/smoke.log 2>&1; echo "smoke exit $?" >> $OUT/smoke.log
tail -2 $OUT/smoke.log
python bench.py --gpus 1 --steps 3 --warmup 3 > $OUT/bench_n1.json 2> $OUT/bench_n1.err; tail -c 400 $OUT/bench_n1.json
python scripts/bench_smo.py --configs C4 --no-sklearn --rows resident >> $OUT/smo_rows_c4.jsonl 2>> $OUT/smo.err
python scripts/bench_smo.py --configs C4 --no-sklearn --rows computed >> $OUT/smo_rows_c4.jsonl 2>> $OUT/smo.err
python scripts/bench_smo.py --configs C4 --no-sklearn --rows computed --cache-mb 0 >> $OUT/smo_rows_c4.jsonl 2>> $OUT/smo.err
cut -c1-600 $OUT/smo_rows_c4.jsonl
for n in 200000 500000; do
  timeout 720 python scripts/bench_smo.py --configs C5 --n $n --large >> $OUT/smo_rows_large.jsonl 2>> $OUT/smo.err || echo "C5 n=$n: exit $?" >> $OUT/smo_rows_large.jsonl
done
cat $OUT/smo_rows_large.jsonl; tail -5 $OUT/smo.err
