#!/bin/bash
# Noise-targeted adaptive sampling (g19_render_adaptive): bit identity of the existing renders against a parent checkout
# built in $PARENT (bench.py --dump-outputs on c2 / c3 / c5), the new and the existing GPU tests, bench.py alternating
# parent and this tree (C2 value, other_configs), and tools/adaptive_bench.py (overhead and benefit tables).
# PHASES (default all) picks from: parity adaptive_tests bench adaptive_bench suite.
OUT=${OUT:-out}
PARENT=${PARENT:-out/parent}
PHASES=${PHASES:-parity adaptive_tests bench adaptive_bench suite}
has() { [[ " $PHASES " == *" $1 "* ]]; }
mkdir -p "$OUT"
LOG="$OUT/r46.log"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee -a "$OUT/r46_gpu.txt" >> "$LOG"
echo "phases: $PHASES" >> "$LOG"
HERE=$(pwd)
DUMPS=$(mktemp -d)  # the dumped frames stay out of $OUT
has parity && for cfg in c2 c3 c5; do
    (cd "$PARENT" && timeout 600 python bench.py --no-others --no-cpu --steps 1 --warmup 1 --config $cfg \
        --dump-outputs "$DUMPS/dump_parent_$cfg" > "$HERE/$OUT/dump_parent_$cfg.json" 2>>"$HERE/$LOG")
    timeout 600 python bench.py --no-others --no-cpu --steps 1 --warmup 1 --config $cfg \
        --dump-outputs "$DUMPS/dump_new_$cfg" > "$OUT/dump_new_$cfg.json" 2>>"$LOG"
    python - "$OUT" $cfg "$DUMPS" >> "$LOG" 2>&1 <<'EOF'
import json, os, sys
out, cfg, dumps = sys.argv[1], sys.argv[2], sys.argv[3]
a, b = os.path.join(dumps, "dump_parent_" + cfg), os.path.join(dumps, "dump_new_" + cfg)
ok = True
for f in ("radiance.npy", "rgb.npy"):
    same = open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read()
    ok &= same
    print(cfg, f, "byte-equal" if same else "DIFFERENT")
ja = json.loads(open(os.path.join(out, "dump_parent_%s.json" % cfg)).read().strip().split("\n")[-1])
jb = json.loads(open(os.path.join(out, "dump_new_%s.json" % cfg)).read().strip().split("\n")[-1])
def find(j, k):  # every value stored under key k, depth first
    if isinstance(j, dict):
        return [v for x, y in j.items() for v in ([y] if x == k else []) + find(y, k)]
    if isinstance(j, list):
        return [v for y in j for v in find(y, k)]
    return []
for k in ("segments_per_sample", "windows"):  # parity windows: relRMSE against the oracle per window
    va, vb = find(ja, k), find(jb, k)
    print(cfg, k, "equal" if va == vb else "DIFFERENT: %s vs %s" % (va, vb))
    ok &= va == vb and len(va) > 0
print(cfg, "bit identity", "OK" if ok else "FAILED")
EOF
done
has adaptive_tests && timeout 900 python -m pytest tests/test_adaptive_gpu.py tests/test_adaptive_oracle.py -q -rs -s --durations=5 > "$OUT/r46_adaptive_tests.log" 2>&1
has adaptive_tests && echo "adaptive tests rc=$?" | tee -a "$OUT/r46_adaptive_tests.log" >> "$LOG"
has adaptive_tests && grep -E "relRMSE|ratio|tile counts|passed|failed" "$OUT/r46_adaptive_tests.log" | cut -c1-200 >> "$LOG"
has bench && for i in 1 2 3; do
    (cd "$PARENT" && timeout 600 python bench.py --gpus 1 --no-cpu > "$HERE/$OUT/bench_parent_$i.json" 2>/dev/null)
    timeout 600 python bench.py --gpus 1 --no-cpu > "$OUT/bench_new_$i.json" 2>/dev/null
done
has bench && python - "$OUT" >> "$LOG" 2>&1 <<'EOF'
import glob, json, os, statistics, sys
out = sys.argv[1]
def load(f):
    return json.loads(open(f).read().strip().split("\n")[-1])
for tag in ("parent", "new"):
    runs = [load(f) for f in sorted(glob.glob(os.path.join(out, "bench_%s_[0-9].json" % tag)))]
    if not runs:
        continue
    v = [r["value"] for r in runs]
    line = "%-8s C2 %s median %.1f (spread %.2f %%)" % (tag, ["%.1f" % x for x in v], statistics.median(v),
                                                        100 * (max(v) - min(v)) / statistics.median(v))
    for oc in (runs[0].get("other_configs") or []):
        c = oc["config"]
        vs = [next(o["value"] for o in r["other_configs"] if o["config"] == c) for r in runs]
        line += " | %s %s" % (c, ["%.1f" % x for x in vs])
    print(line)
EOF
has adaptive_bench && timeout 900 python tools/adaptive_bench.py > "$OUT/r46_adaptive_bench.jsonl" 2>>"$LOG"
has adaptive_bench && echo "adaptive_bench rc=$?" >> "$LOG" && cat "$OUT/r46_adaptive_bench.jsonl" >> "$LOG"
if has suite; then
    timeout 1500 python -m pytest tests -m gpu -q -rs --durations=10 > "$OUT/r46_all_tests.log" 2>&1
    echo "GPU suite rc=$?" | tee -a "$OUT/r46_all_tests.log" >> "$LOG"
    tail -3 "$OUT/r46_all_tests.log" >> "$LOG"
    python -c "import __graft_entry__ as g; g.smoke()" >> "$LOG" 2>&1; echo "smoke rc=$?" >> "$LOG"
fi
rm -rf "$DUMPS"
cut -c1-400 "$LOG"
