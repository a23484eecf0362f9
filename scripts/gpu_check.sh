#!/bin/bash
# One GPU-box pass: parity tests, bench line, ncu launch list, ncu full capture of the evaluation kernels.
# usage (through gpurun): bash scripts/gpu_check.sh <tag> [skip_tests]
TAG=${1:-run}
OUT=gpurun_out/$TAG
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.max.sm,clocks.max.mem,power.limit --format=csv > $OUT/gpu.txt 2>&1
nproc >> $OUT/gpu.txt
if [ -z "$2" ]; then
  timeout 900 python -m pytest tests -m gpu -q > $OUT/pytest.log 2>&1; echo "pytest rc=$?" | tee -a $OUT/pytest.log
  tail -3 $OUT/pytest.log
fi
timeout 900 python bench.py --steps 50 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
cat $OUT/bench.json
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file $OUT/launches.csv python bench.py --quick --steps 3 --warmup 3 > $OUT/ncu_launches.log 2>&1; echo "ncu launches rc=$?"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'DynOut|RomNodeOut|TransposeIn' --launch-skip 12 --launch-count 4 -o $OUT/full python bench.py --quick --steps 3 --warmup 3 > $OUT/ncu_full.log 2>&1; echo "ncu full rc=$?"
ls -la $OUT
