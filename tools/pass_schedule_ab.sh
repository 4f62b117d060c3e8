#!/bin/bash
# A/B of the pass plan (nn_sched.h): the default plan against C3R_PASS_SCHEDULE=rounds, in one process tree.
#   tools/pass_schedule_ab.sh OUT [RUNS] [CONFIGS]
# 1. bench.py --dump-outputs under both plans; the dumps must be bit-identical.
# 2. RUNS alternating bench.py runs of each plan per config; one line per run with value, e2e, k5_network, shard_cfg5.
set -e
OUT=${1:?usage: tools/pass_schedule_ab.sh OUT [RUNS] [CONFIGS]}
RUNS=${2:-3}
CONFIGS=${3:-"2 4"}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
for plan in default rounds; do
    env $([ $plan = rounds ] && echo C3R_PASS_SCHEDULE=rounds) python bench.py --gpus 1 --steps 3 --warmup 1 --cfg5_scale 0 \
        --no_cpu_baseline --dump-outputs "$OUT/dump_$plan" 2>"$OUT/dump_$plan.err" | grep '^{"metric"' > "$OUT/dump_$plan.json"
done
python - "$OUT" <<'EOF'
import os, sys
import numpy as np
out = sys.argv[1]
a, b = os.path.join(out, "dump_default"), os.path.join(out, "dump_rounds")
names = sorted(f for f in os.listdir(a) if f.endswith(".npy"))
assert names and names == sorted(f for f in os.listdir(b) if f.endswith(".npy")), "dump file lists differ"
for f in names:
    x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
    same = x.shape == y.shape and x.dtype == y.dtype and x.tobytes() == y.tobytes()
    print("dump %-28s %-16s %s" % (f, str(x.shape), "identical" if same else "DIFFERENT"))
    assert same, f
EOF
for cfg in $CONFIGS; do
    for r in $(seq 1 "$RUNS"); do
        for plan in default rounds; do
            line=$(env $([ $plan = rounds ] && echo C3R_PASS_SCHEDULE=rounds) python bench.py --gpus 1 --config "$cfg" \
                --no_cpu_baseline $([ "$cfg" != 2 ] && echo --cfg5_scale 0) 2>>"$OUT/bench.err" | grep '^{"metric"')
            echo "$line" > "$OUT/bench_c${cfg}_${plan}_$r.json"
            python -c '
import json, sys
d = json.loads(sys.argv[1])
sm = d.get("stage_ms", {})
s5 = d.get("shard_cfg5", {})
s5 = s5.get("value", s5) if isinstance(s5, dict) else s5
print("config %s run %s %-8s value %.4g e2e %.4g k5_network %.4f ms shard_cfg5 %s" % (sys.argv[2], sys.argv[3], sys.argv[4],
      d["value"], d["e2e"]["value"], sm.get("k5_network", float("nan")), s5))' "$line" "$cfg" "$r" "$plan"
        done
    done
done
