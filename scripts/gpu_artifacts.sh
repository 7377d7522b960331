#!/bin/bash
# Final-state artefacts: bench line, launch list, ncu --set full of the tensor-core / scatter / optimiser kernels, components.
mkdir -p gpurun_out
cd "${GRAFT_REPO_ROOT:-.}"
T0=$(date +%s)
ADER_B200_TRACE=gpurun_out/trace_final.json timeout 120 python bench.py > gpurun_out/bench_final.json 2> gpurun_out/bench_final.err
echo "bench rc=$? t=$(( $(date +%s) - T0 ))" >> gpurun_out/legs_artifacts.txt
timeout 100 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
    --log-file gpurun_out/launches_final.csv python scripts/ncu_step.py 2 > gpurun_out/ncu_launches_final.log 2>&1
echo "launches rc=$? t=$(( $(date +%s) - T0 ))" >> gpurun_out/legs_artifacts.txt
timeout 150 ncu --profile-from-start off --set full --clock-control none --import-source on \
    -k regex:'k_tc2|k_scatter_apply|k_adam|k_merge_stats|k_sort_scatter' \
    -f -o gpurun_out/final_full python scripts/ncu_step.py 1 > gpurun_out/ncu_final_full.log 2>&1
echo "full rc=$? t=$(( $(date +%s) - T0 ))" >> gpurun_out/legs_artifacts.txt
[ -f gpurun_out/final_full.ncu-rep ] && ncu -i gpurun_out/final_full.ncu-rep --page raw --csv > gpurun_out/final_full.raw.csv 2>/dev/null
timeout 120 python scripts/bench_components.py > gpurun_out/components_final.jsonl 2> gpurun_out/components_final.err
echo "components rc=$? t=$(( $(date +%s) - T0 ))" >> gpurun_out/legs_artifacts.txt
cat gpurun_out/legs_artifacts.txt; head -c 300 gpurun_out/bench_final.json; echo; tail -3 gpurun_out/components_final.err
