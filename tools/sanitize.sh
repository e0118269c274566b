#!/bin/bash
# compute-sanitizer over the kernels that alias shared-memory regions across barriers (k_inner_cem_fast) or hand-roll mbarrier protocols
# (k_project, k_project_tc).  One log per tool, sanitize_<tool>.log, in the output directory created below.
set -u
mkdir -p gpurun_out
SEL_MEM='inner_cem_kernel_variants or stage_project_bit_exact or solve_small or tensor_core_within or stage_risk_bit_exact or injected'
SEL_RACE='(inner_cem_kernel_variants and 5-30-gaussian) or stage_project_bit_exact or tensor_core_within'
timeout 1500 compute-sanitizer --tool memcheck --error-exitcode 86 python -m pytest tests/test_gpu_parity.py -x -q -k "$SEL_MEM" > gpurun_out/sanitize_memcheck.log 2>&1
echo "memcheck rc=$?" | tee -a gpurun_out/sanitize_memcheck.log
timeout 1500 compute-sanitizer --tool racecheck --racecheck-report all --error-exitcode 86 python -m pytest tests/test_gpu_parity.py -x -q -k "$SEL_RACE" > gpurun_out/sanitize_racecheck.log 2>&1
echo "racecheck rc=$?" | tee -a gpurun_out/sanitize_racecheck.log
timeout 900 compute-sanitizer --tool synccheck --error-exitcode 86 python -m pytest tests/test_gpu_parity.py -x -q -k "$SEL_RACE" > gpurun_out/sanitize_synccheck.log 2>&1
echo "synccheck rc=$?" | tee -a gpurun_out/sanitize_synccheck.log
tail -5 gpurun_out/sanitize_memcheck.log gpurun_out/sanitize_racecheck.log gpurun_out/sanitize_synccheck.log
