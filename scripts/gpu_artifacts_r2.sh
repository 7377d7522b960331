#!/bin/bash
# Round-2 artefacts: launch list of one train step, ncu --set full of the tcgen05 loss kernels / fused eval kernel / Adam /
# herding kernels, compute-sanitizer memcheck over a subset of the GPU tests.
mkdir -p gpurun_out
cd "${GRAFT_REPO_ROOT:-.}"
T0=$(date +%s)
timeout 150 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
    --log-file gpurun_out/r2_launches_step.csv python scripts/ncu_step.py 2 > gpurun_out/r2_ncu_launches.log 2>&1
echo "launches rc=$? t=$(( $(date +%s) - T0 ))"
timeout 240 ncu --profile-from-start off --set full --clock-control none --import-source on \
    -k regex:'k_tc2|k_adam|k_scatter_apply|k_qkv_fwd|k_attn_ln_fwd|k_wgrad' \
    -f -o gpurun_out/r2_step_full python scripts/ncu_step.py 1 > gpurun_out/r2_ncu_step_full.log 2>&1
echo "step full rc=$? t=$(( $(date +%s) - T0 ))"
[ -f gpurun_out/r2_step_full.ncu-rep ] && ncu -i gpurun_out/r2_step_full.ncu-rep --page raw --csv > gpurun_out/r2_step_full.raw.csv 2>/dev/null
timeout 240 ncu --set full --clock-control none --import-source on -k regex:'k_eval_tc|k_refine|k_herding_small|k_herding_mid|k_herding_big|k_fisher_table|k_dp_adam' -c 12 \
    -f -o gpurun_out/r2_components_full python -c "
import bench, torch
print(bench.gpu_components(torch.device('cuda', 0)))" > gpurun_out/r2_ncu_components_full.log 2>&1
echo "components full rc=$? t=$(( $(date +%s) - T0 ))"
[ -f gpurun_out/r2_components_full.ncu-rep ] && ncu -i gpurun_out/r2_components_full.ncu-rep --page raw --csv > gpurun_out/r2_components_full.raw.csv 2>/dev/null
rm -f gpurun_out/r2_step_full.ncu-rep gpurun_out/r2_components_full.ncu-rep
# compute-sanitizer (memcheck) over the kernel-level parity tests (SURVEY section 5: race / memory checking)
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 --print-limit 20 python -m pytest tests/test_gpu_parity.py tests/test_gpu_encoder_fused.py tests/test_gpu_eval.py tests/test_gpu_herding.py -m gpu -x -q \
    -k "encoder_forward or train_grad_kd or tc_loss_path or fused_forward or fused_ranks or second_generation or batched_fisher or adam_matches" \
    > gpurun_out/r2_sanitizer_memcheck.log 2>&1
echo "sanitizer rc=$? t=$(( $(date +%s) - T0 ))"; tail -8 gpurun_out/r2_sanitizer_memcheck.log
ls -la gpurun_out/r2_*
