#!/bin/bash
# Runs the GPU suite in separate processes (a sticky CUDA error in one group must not mask the others).
# Usage (on the GPU box): bash tests/run_gpu_suite.sh [outdir]
OUT=${1:-gpurun_out}
mkdir -p $OUT
run() { name=$1; shift; echo "=== $name" ; timeout 900 "$@" > $OUT/$name.log 2>&1; echo "exit $?" | tee -a $OUT/$name.log; tail -n 25 $OUT/$name.log; }
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $OUT/gpu.csv 2>&1
run t1_bottleneck python -m pytest tests/test_gpu_bottleneck.py -q --no-header -rfE -p no:cacheprovider
run t2_exact python -m pytest tests/test_gpu_attention.py -q --no-header -rfE -p no:cacheprovider -k "exact"
run t3_dump python -m pytest tests/test_gpu_attention.py -q --no-header -rfE -p no:cacheprovider -k "raw_scores"
run t4_sm100 python -m pytest tests/test_gpu_attention.py -q --no-header -rfE -p no:cacheprovider -k "sm100 and not raw_scores or masked or validation"
run t4b_probes python -m pytest tests/test_gpu_attention_probes.py -q --no-header -rfE -p no:cacheprovider
run t5_full python -m pytest tests/test_gpu_attention.py -q --no-header -rfE -p no:cacheprovider -k "full_size"
run t6_model python -m pytest tests/test_gpu_model.py -q --no-header -rfE -p no:cacheprovider
run t7_smoke python -c "import __graft_entry__ as g; g.smoke()"
