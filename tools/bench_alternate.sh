#!/bin/bash
# bench.py on two trees alternately, in one GPU session:
#   tools/bench_alternate.sh PARENT_TREE OUT_DIR [ROUNDS]
# PARENT_TREE is a built checkout of the commit to compare against (its own build() run first).  Each round runs
#   bench.py --gpus 1 --steps 10 --warmup 3
# in PARENT_TREE and then in this tree; afterwards each tree writes its --dump-outputs files once and the two sets are
# compared byte for byte.  OUT_DIR gets every bench line and alternation.json: per tree the resident ms_per_step of each
# round, the median and spread, e2e pinned and pageable, and the card's name, power limit and maximum SM clock.
set -u
PARENT=$(cd "$1" && pwd)
mkdir -p "$2"
OUT=$(cd "$2" && pwd)
ROUNDS=${3:-3}
HERE=$(cd "$(dirname "$0")/.." && pwd)
TMP=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader -i 0 > "$OUT/card.txt"
for r in $(seq 1 "$ROUNDS"); do
  (cd "$PARENT" && python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT/parent_$r.json" 2> "$OUT/parent_$r.err")
  (cd "$HERE" && python bench.py --gpus 1 --steps 10 --warmup 3 > "$OUT/new_$r.json" 2> "$OUT/new_$r.err")
done
(cd "$PARENT" && python bench.py --gpus 1 --steps 3 --warmup 3 --no-cpu-baseline --no-configs --dump-outputs "$TMP/parent" > /dev/null 2>&1)
(cd "$HERE" && python bench.py --gpus 1 --steps 3 --warmup 3 --no-cpu-baseline --no-configs --dump-outputs "$TMP/new" > /dev/null 2>&1)
diff -r "$TMP/parent" "$TMP/new" > /dev/null 2>&1 && SAME=true || SAME=false
python - "$OUT" "$ROUNDS" "$SAME" <<'PY'
import json, statistics, sys
out_dir, rounds, same = sys.argv[1], int(sys.argv[2]), sys.argv[3] == "true"
res = {"what": f"bench.py --gpus 1 --steps 10 --warmup 3, the parent tree and this one alternately, {rounds} rounds",
       "card": open(f"{out_dir}/card.txt").read().strip(), "dump_outputs_identical": same, "rounds": {}}
for t in ("parent", "new"):
    rs = []
    for r in range(1, rounds + 1):
        j = json.loads(open(f"{out_dir}/{t}_{r}.json").read().strip().splitlines()[-1])
        rs.append({"ms_per_step": j["ms_per_step"], "e2e_pinned_ms": j["e2e"]["ms_per_step"],
                   "e2e_pageable_ms": j["e2e"]["pageable"]["ms_per_step"], "gpu_launches": j["gpu_launches"],
                   "argmax_index": j["argmax"]["index"]})
    ms = [r["ms_per_step"] for r in rs]
    res["rounds"][t] = rs
    res[t + "_median_ms"] = statistics.median(ms)
    res[t + "_spread_ms"] = max(ms) - min(ms)
json.dump(res, open(f"{out_dir}/alternation.json", "w"), indent=1)
print(json.dumps({k: v for k, v in res.items() if k != "rounds"}))
PY
rm -rf "$TMP"
