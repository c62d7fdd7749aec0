#!/bin/bash
# compute-sanitizer (memcheck / racecheck / synccheck) over the hand-written tcgen05 / TMA / mbarrier kernels, through small GPU tests.
# Usage (on the GPU box): bash tools/run_sanitizer.sh [outdir]   -- logs go to <outdir>/sanitizer_<tool>.log
out=${1:-gpurun_out}
mkdir -p "$out"
TESTS="tests/test_gpu_conv_umma.py::test_every_conv_umma_vs_simt_and_cpu[shape1] tests/test_gpu_output_parity.py::test_every_conv_tf32_vs_exact_tf32_arithmetic[shape1] tests/test_gpu_conv_umma.py::test_fused_basic_block_vs_separate_convs_and_cpu[shape2] tests/test_gpu_vitpose.py::test_gemm_umma[2100-1152-384-0-False-True] tests/test_gpu_vitpose.py::test_gemm_umma[300-384-384-0-True-False] tests/test_gpu_vitpose.py::test_gemm_umma[130-128-64-2-False-True] tests/test_gpu_vitpose.py::test_attention_umma[2-128] tests/test_gpu_vitpose.py::test_attention_umma[3-60] tests/test_gpu_parity.py::test_uplift_bf16_tensor_core_bound tests/test_gpu_parity.py::test_uplift_golden[connectstage-tf32x3] tests/test_gpu_vitpose.py::test_gemm_x3[300-384-384-0-True-False] tests/test_gpu_vitpose.py::test_gemm_x3[24-1152-384-0-False-True] tests/test_gpu_vitpose.py::test_attention_x3[2-128] tests/test_gpu_vitpose.py::test_attention_x3[3-60] tests/test_gpu_vitpose.py::test_vitpose_x3_vs_oracle[res0-2] tests/test_gpu_conv_umma.py::test_network_block_fusion_tf32 tests/test_gpu_rally_cameras.py::test_reproject_clips_equals_project_per_clip tests/test_gpu_rally_cameras.py::test_reproject_clips_invalid_clips_are_nan"
# gemm3_umma_kernel (uplift tf32x3) uses 232 064 of the 232 448 bytes of shared memory a CTA can have; synccheck keeps its barrier
# bookkeeping in shared memory too and then reports "Missing init" for every mbarrier wait of that kernel (and kills it), while the
# same kernel built with a 2-stage ring (32 KB less) is clean.  So synccheck runs without the tf32x3 uplift tests on the stock library,
# and on them with the 2-stage build (the barrier protocol does not depend on the ring depth).
G3="tests/test_gpu_parity.py::test_uplift_golden[connectstage-tf32x3]"
for tool in memcheck synccheck racecheck; do
  log="$out/sanitizer_$tool.log"
  echo "== compute-sanitizer --tool $tool ==" > "$log"
  T="$TESTS"
  if [ $tool = synccheck ]; then T="${TESTS/"$G3"/}"; T="${T/tests\/test_gpu_parity.py::test_uplift_bf16_tensor_core_bound/}"; fi
  timeout 1500 compute-sanitizer --tool $tool --print-limit 20 --error-exitcode 9 python -m pytest $T -x -q -m gpu -p no:cacheprovider >> "$log" 2>&1
  echo "exit code $?" >> "$log"
  tail -4 "$log"
done
log="$out/sanitizer_synccheck.log"
echo "== synccheck of the tf32x3 uplift with gemm3 built with a 2-stage ring (-DTTK_GEMM3_STAGES=2) ==" >> "$log"
touch upliftingtabletennis_b200/csrc/gemm3_umma.cu
TTK_NVCC_FLAGS=-DTTK_GEMM3_STAGES=2 python -m upliftingtabletennis_b200.build >> "$log" 2>&1
timeout 900 compute-sanitizer --tool synccheck --print-limit 20 --error-exitcode 9 python -m pytest "$G3" tests/test_gpu_parity.py::test_uplift_bf16_tensor_core_bound -x -q -m gpu -p no:cacheprovider >> "$log" 2>&1
echo "exit code $?" >> "$log"
tail -4 "$log"
touch upliftingtabletennis_b200/csrc/gemm3_umma.cu
python -m upliftingtabletennis_b200.build >> "$log" 2>&1
