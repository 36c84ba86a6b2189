#!/bin/bash
# batched ray queries (g19_cast_rays): their tests, then their throughput on their own (tools/cast_bench.py)
OUT=${OUT:-out}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r03a_gpu.txt"
timeout 1200 python -m pytest tests/test_cast_gpu.py tests/test_cast_oracle.py -q -rs > "$OUT/r03a_cast_tests.log" 2>&1; echo "tests rc=$?" >> "$OUT/r03a_cast_tests.log"
tail -6 "$OUT/r03a_cast_tests.log" | cut -c1-220
timeout 900 python tools/cast_bench.py --out "$OUT/r03a_cast_bench.jsonl" > "$OUT/r03a_cast_bench.log" 2>&1; echo "cast_bench rc=$?" >> "$OUT/r03a_cast_bench.log"
cut -c1-300 "$OUT/r03a_cast_bench.log"
