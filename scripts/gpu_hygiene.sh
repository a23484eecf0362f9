#!/bin/bash
# One GPU-box pass of round-2 evidence: compute-sanitizer (memcheck, racecheck) over the config-2 / config-4 parity tests,
# the bench line, the ncu launch list of the same command and a --set full capture of the evaluation kernels.
# usage (through gpurun): bash scripts/gpu_hygiene.sh <tag>
TAG=${1:-r2_hyg}; OUT=gpurun_out/$TAG; mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.max.sm,clocks.max.mem,power.limit --format=csv > $OUT/gpu.txt 2>&1; nproc >> $OUT/gpu.txt
for tool in memcheck racecheck; do
  timeout 1500 compute-sanitizer --tool $tool --error-exitcode 9 python -m pytest tests/test_gpu_parity.py -x -q -k "config2 or config4 or batch_of_one" > $OUT/sanitizer_$tool.log 2>&1
  echo "$tool rc=$?" | tee -a $OUT/sanitizer_$tool.log; tail -4 $OUT/sanitizer_$tool.log
done
timeout 900 python bench.py --steps 50 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file $OUT/launches.csv env TWB_NO_CONFIG5=1 python bench.py --quick --steps 3 --warmup 3 > $OUT/ncu_launches.log 2>&1; echo "ncu launches rc=$?"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'DynOut|RomNodeOut|TransposeIn' --launch-skip 12 --launch-count 4 -o $OUT/full python bench.py --quick --steps 3 --warmup 3 > $OUT/ncu_full.log 2>&1; echo "ncu full rc=$?"
ls -la $OUT
