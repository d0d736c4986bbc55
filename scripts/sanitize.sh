#!/bin/bash
# compute-sanitizer passes over the fast GPU tests (run through gpurun; logs land in gpurun_out/).
# memcheck: out-of-bounds / misaligned accesses of every kernel; racecheck: shared-memory hazards; initcheck: reads of
# uninitialised global memory.  Big-shape tests are deselected (the tools slow kernels down 10-100x).
O=gpurun_out
mkdir -p $O
SEL='not full_size and not full_shape and not full_batch and not large_keystream and not statistics'
for tool in memcheck racecheck; do
  timeout ${SAN_TIMEOUT:-900} compute-sanitizer --tool $tool --error-exitcode 9 --launch-timeout 0 \
    --print-limit 30 \
    python -m pytest tests/test_gpu_svi.py tests/test_gpu_minibatch.py tests/test_gpu_random.py tests/test_gpu_device_keys.py \
      tests/test_gpu_vae.py tests/test_gpu_vae_inputs.py tests/test_gpu_gmm.py tests/test_gpu_epoch.py tests/test_gpu_gemm.py \
      -x -q -k "$SEL" \
      > $O/sanitize_$tool.log 2>&1
  echo "$tool rc=$?" >> $O/sanitize_summary.txt
  tail -5 $O/sanitize_$tool.log
done
cat $O/sanitize_summary.txt
