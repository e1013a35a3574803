#!/bin/bash
# Sanitizer evidence for the per-column kernel code (SURVEY.md section 5, row "race detection / sanitizers").
#
# compute-sanitizer is CLOSED on the B200 pool this repository is built on ("runs under it have left GPUs needing a
# reset"; profiles/r2_sanitizer_pool_closed.txt), so the device code is checked in the two ways that remain:
#  1. the SAME per-column sources (csrc/*.cuh) are compiled for the host with AddressSanitizer +
#     UndefinedBehaviorSanitizer (tests/hostsim, XP_HOSTSIM_SANITIZE=1) and the whole CPU test-suite of that code runs
#     under them: every stash / table / level index the kernels compute is bounds-checked against real allocations;
#  2. on the GPU, a -DXP_BOUNDS_CHECK build of libxparcel.so turns every shared-memory stash / coefficient-table /
#     list access of the fast kernels into a device assert (tests/test_gpu_bounds_check.py).
set -e
cd "$(dirname "$0")/.."
export XP_HOSTSIM_SANITIZE=1
export ASAN_OPTIONS=detect_leaks=0:abort_on_error=1
LD_PRELOAD="$(gcc -print-file-name=libasan.so):$(gcc -print-file-name=libubsan.so)" \
    python -m pytest tests/test_fast_hostsim.py tests/test_hostsim_vs_oracle.py tests/test_layers_hostsim.py \
    tests/test_levels_hostsim.py tests/test_specific_humidity_input.py tests/test_kinematics_hostsim.py -q -m "not gpu" -p no:cacheprovider "$@"
