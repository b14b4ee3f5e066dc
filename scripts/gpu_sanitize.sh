#!/bin/bash
# compute-sanitizer over the GPU parity tests: memcheck, racecheck (shared-memory hazards) and synccheck on the parity files (the
# full-size config-3 case excluded: minutes under the tools).
# Usage: gpurun --timeout 1200 -- bash scripts/gpu_sanitize.sh [tag]
set -u
OUT=gpurun_out/${1:-sanitize}
mkdir -p "$OUT"
SMALL="tests/test_curve_gpu.py tests/test_scene_gpu.py tests/test_post_gpu.py tests/test_lines_gpu.py tests/test_perlin_gpu.py tests/test_splat_gpu.py"
run() {   # tool, log name, test files, extra env
    env ${4:-X=1} timeout ${SAN_TIMEOUT:-240} compute-sanitizer --tool "$1" --error-exitcode 7 --print-limit 5 \
        python -m pytest $3 -m gpu -q -p no:cacheprovider -k "not full_size" > "$OUT/$2.log" 2>&1
    echo "$1 ($2) exit code: $?" | tee -a "$OUT/$2.log"
    grep -E "ERROR SUMMARY|RACECHECK SUMMARY|passed|failed" "$OUT/$2.log" | tail -4
}
run memcheck memcheck "$SMALL tests/test_configs_gpu.py"
run racecheck racecheck "$SMALL"
run synccheck synccheck "$SMALL"
