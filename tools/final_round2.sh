#!/bin/bash
# Final records of round 2 on one B200: tests, smoke, the driver's bench command, one bench line per
# BASELINE config, the reference arm, the knob matrix.
O=gpurun_out
python -m pytest tests -m gpu -x -q > $O/r02_final_tests.txt 2>&1; tail -2 $O/r02_final_tests.txt
python -c "import __graft_entry__ as g; g.smoke()" > $O/r02_final_smoke.txt 2>&1; tail -1 $O/r02_final_smoke.txt
python bench.py --steps 20 --warmup 5 > $O/r02_bench_n1.json 2> $O/r02_bench_n1.err
python bench.py --impl reference --steps 20 --warmup 5 > $O/r02_bench_reference_arm.json 2>> $O/r02_bench_n1.err
: > $O/r02_bench_all_configs.jsonl
for a in "--config 1" "--config 2" "--config 3" "--config 4 --format RGBA" "--config 4 --format BGRA" "--config 4 --format AYUV" "--config 5"; do
  python bench.py $a --steps 200 --warmup 5 --no-cpu-baseline >> $O/r02_bench_all_configs.jsonl 2>> $O/r02_bench_n1.err
done
bash tools/knob_matrix.sh > $O/r02_knob_matrix.txt 2>&1
grep -c passed $O/r02_knob_matrix.txt; grep -c failed $O/r02_knob_matrix.txt
build/latency_probe > $O/r02_latency_probe.txt 2>&1
{ for t in 4 8 12; do FLUC_TTMLBLEND_STAGE_THREADS=$t build/e2e_multi --gpus 0 --pageable --secs 1.5; done; build/e2e_multi --gpus 0 --secs 1.5; } > $O/r02_pageable_probe.txt 2>&1
build/launch_floor > $O/r02_launch_floor.txt 2>&1
bash tools/ab_opaque.sh > $O/r02_opaque_skip.txt 2>&1
