#!/bin/bash
# compute-sanitizer over the kernel modes (profiles/round2_sanitizer_*.log).
mkdir -p gpurun_out/sanitizer
S=/usr/local/cuda/bin/compute-sanitizer
if [ "${1:-}" = reservations ]; then
  # the capacity-reservation suite (tests/golden/reservations.json); logs go
  # to $SANITIZE_DIR (default: a new temporary directory)
  D=${SANITIZE_DIR:-$(mktemp -d)}
  mkdir -p "$D"
  for mode in auto fast-split; do
    for tool in memcheck racecheck; do
      log="$D/${tool}_reservations_${mode}.log"
      timeout 600 $S --tool $tool --print-limit 20 python tools/sanitize_reservations.py $mode > "$log" 2>&1
      echo "$tool reservations $mode rc=$? $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY' "$log" | tail -1)"
    done
  done
  echo "logs in $D"
  exit 0
fi
for mode in auto fast-split fast-noprune tile queue; do
  for tool in memcheck racecheck; do
    timeout 600 $S --tool $tool --print-limit 20 python tools/sanitize_target.py $mode \
      > gpurun_out/sanitizer/${tool}_${mode}.log 2>&1
    echo "$tool $mode rc=$? $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY' gpurun_out/sanitizer/${tool}_${mode}.log | tail -1)"
  done
done
for tool in synccheck initcheck; do
  timeout 600 $S --tool $tool --print-limit 20 python tools/sanitize_target.py auto \
    > gpurun_out/sanitizer/${tool}_auto.log 2>&1
  echo "$tool auto rc=$? $(grep -E 'ERROR SUMMARY' gpurun_out/sanitizer/${tool}_auto.log | tail -1)"
done
# the region allow-list and the forced full chain evaluation
SKYOPT_EXP=8 timeout 600 $S --tool memcheck --print-limit 20 python tools/sanitize_target.py auto \
  > gpurun_out/sanitizer/memcheck_auto_fullchain.log 2>&1
echo "memcheck auto fullchain rc=$? $(grep -E 'ERROR SUMMARY' gpurun_out/sanitizer/memcheck_auto_fullchain.log | tail -1)"
