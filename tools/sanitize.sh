#!/bin/bash
# compute-sanitizer over the GPU parity tests (SURVEY section 5): memcheck, then racecheck (shared-memory hazards of the cp.async / TMA
# staging, the in-place state tiles, the per-warp scans of the long-string pass), then initcheck on the witness columns.  Everything
# except the largest batches (2^20 strings, 16 MiB string, 30 000-string fuzz, the `huge` DFA shapes).  The summaries are copied to profiles/.
mkdir -p gpurun_out
SKIP="not large_batches and not 16_mib and not fuzz and not full_size and not multi_device and not huge"
FILES="tests/test_gpu_parity.py tests/test_fr_feed.py tests/test_host_paths.py tests/test_cpp_host.py tests/test_dfa_shapes.py tests/test_batch_chunked.py tests/test_knob_matrix.py"
for tool in memcheck racecheck; do
    extra=""; [ $tool = racecheck ] && extra="--racecheck-report all"
    timeout 3000 compute-sanitizer --tool $tool $extra --error-exitcode 9 --target-processes all python -m pytest $FILES -m gpu -q -k "$SKIP" > gpurun_out/r2_$tool.log 2>&1
    echo "$tool exit code $?" >> gpurun_out/r2_$tool.log
done
grep -E "ERROR SUMMARY|RACECHECK SUMMARY|passed|failed|exit code" gpurun_out/r2_memcheck.log gpurun_out/r2_racecheck.log
