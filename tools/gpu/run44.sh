#!/bin/bash
# exact per-primitive ray-query answers under every tree walk and traversal knob (tests/test_walk_exact_gpu.py, with its
# CPU check of the expectations and the existing ray-query tests)
OUT=${OUT:-out}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r04a_gpu.txt"
timeout 2400 python -m pytest tests/test_walk_cases.py tests/test_walk_exact_gpu.py tests/test_cast_gpu.py -q -rs --durations=10 \
    > "$OUT/r04a_walk_tests.log" 2>&1; echo "tests rc=$?" >> "$OUT/r04a_walk_tests.log"
tail -16 "$OUT/r04a_walk_tests.log" | cut -c1-220
