#!/usr/bin/env bash
# compute-sanitizer over the small parity tests (SURVEY.md section 5, "race detection / sanitizers"): every blend-kernel variant,
# the three binning methods, the fused smoothing / sampling ops and the KNN.  memcheck = out-of-bounds /
# misaligned accesses; racecheck = shared-memory hazards; synccheck = divergent barriers.  One GPU.
set -u
mkdir -p gpurun_out
SEL='test_blend_kernel_variants_agree or test_depth_first_binning_is_bit_identical or test_tile_sort_binning_is_bit_identical or test_edge_cases or test_mask_only_path or test_cuda_matches_oracle'
for tool in memcheck racecheck synccheck; do
  echo "== compute-sanitizer --tool $tool =="
  timeout 200 compute-sanitizer --tool $tool --error-exitcode 77 --log-file gpurun_out/r2_sanitizer_${tool}.log \
      python -m pytest tests/test_parity_gpu.py tests/test_sampling_gpu.py tests/test_smoothing_gpu.py -m gpu -q -x -k "$SEL or sample_rays or smooth" \
      > gpurun_out/r2_sanitizer_${tool}.pytest.log 2>&1
  echo "rc=$?"; tail -3 gpurun_out/r2_sanitizer_${tool}.pytest.log; grep -c "=========" gpurun_out/r2_sanitizer_${tool}.log; grep "ERROR SUMMARY\|RACECHECK SUMMARY" gpurun_out/r2_sanitizer_${tool}.log | tail -2
done
