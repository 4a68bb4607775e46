#!/bin/bash
# compute-sanitizer over the GPU parity tests: bash scripts/sanitize.sh [output dir, default sanitize_out]
# memcheck on the whole -m gpu suite of the optimizer / ESDF / multi paths; racecheck on a reduced selection (it is ~50x slower).
set -u
OUT="${1:-sanitize_out}"
mkdir -p "$OUT"
export ALORE_SANITIZE_SMALL=1
compute-sanitizer --tool memcheck --error-exitcode 99 --log-file "$OUT"/memcheck_r02.log \
  python -m pytest tests/test_optimizer_gpu.py tests/test_esdf_gpu.py tests/test_golden.py -x -q -m gpu \
  -k "not division and not 4096 and not 8192 and not 2048 and not long_trajectories" > "$OUT"/memcheck_r02.pytest.txt 2>&1
echo "memcheck rc=$?" >> "$OUT"/memcheck_r02.pytest.txt
compute-sanitizer --tool racecheck --error-exitcode 99 --log-file "$OUT"/racecheck_r02.log \
  python -m pytest tests/test_optimizer_gpu.py -x -q -m gpu -k "cost_and_gradient_batch or small_piece_counts or penalty_batch or final_collision or config1" \
  > "$OUT"/racecheck_r02.pytest.txt 2>&1
echo "racecheck rc=$?" >> "$OUT"/racecheck_r02.pytest.txt
tail -n 3 "$OUT"/memcheck_r02.pytest.txt "$OUT"/racecheck_r02.pytest.txt
grep -h "ERROR SUMMARY" "$OUT"/memcheck_r02.log "$OUT"/racecheck_r02.log
# ESDF far-field path (K2 masks/flags, conditional K1b, K2e band envelope, warp-per-cell quirk column)
compute-sanitizer --tool memcheck --error-exitcode 99 --log-file "$OUT"/memcheck_esdf_r02.log \
  python -m pytest tests/test_esdf_gpu.py -x -q -m gpu -k "(small_maps or far_field or box_and_dense or sub_window or named_maps) and not 4096 and not 8192" \
  > "$OUT"/memcheck_esdf_r02.pytest.txt 2>&1
echo "memcheck(esdf) rc=$?" >> "$OUT"/memcheck_esdf_r02.pytest.txt
compute-sanitizer --tool racecheck --error-exitcode 99 --log-file "$OUT"/racecheck_esdf_r02.log \
  python -m pytest tests/test_esdf_gpu.py -x -q -m gpu -k "far_field_maps" \
  > "$OUT"/racecheck_esdf_r02.pytest.txt 2>&1
echo "racecheck(esdf) rc=$?" >> "$OUT"/racecheck_esdf_r02.pytest.txt
tail -n 3 "$OUT"/memcheck_esdf_r02.pytest.txt "$OUT"/racecheck_esdf_r02.pytest.txt
grep -h "ERROR SUMMARY" "$OUT"/memcheck_esdf_r02.log "$OUT"/racecheck_esdf_r02.log
