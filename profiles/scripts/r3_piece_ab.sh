#!/bin/bash
# Round 3 A/B of reader piece staging against the parent commit's 512 MiB IN ring,
# on one GPU, in one session:
#   config 2A alternately for the two builds (ABBA order, ROUNDS times each), then per build one VMIG_TRACE=1 pass of 2A
#   and one run each of 2B and 4, all four with --dump-outputs, and an output-for-output comparison of those dumps.
# usage: profiles/scripts/r3_piece_ab.sh BASE_TREE NEW_TREE OUT_DIR [ROUNDS]
#   BASE_TREE: `git archive` of the parent commit, NEW_TREE: of the commit under test (or the parent with a patch
#   applied), each built in place (__graft_entry__.build())
set -u
BASE=$(cd "$1" && pwd); NEW=$(cd "$2" && pwd); mkdir -p "$3"; OUT=$(cd "$3" && pwd); ROUNDS=${4:-4}
export PYTHONDONTWRITEBYTECODE=1
tree_of() { [ "$1" = base ] && echo "$BASE" || echo "$NEW"; }
bench() {   # arm tag args...
    local arm=$1 tag=$2; shift 2
    (cd "$(tree_of "$arm")" && python bench.py --gpus 1 "$@") >> "$OUT/${tag}_$arm.jsonl" 2>> "$OUT/${tag}_$arm.err"
    echo "$arm $tag rc=$? $(tail -n 1 "$OUT/${tag}_$arm.jsonl" | python -c 'import json,sys; d=json.loads(sys.stdin.read()); print(d["value"], d["unit"], d["ms_per_step"], "ms/step")' 2>/dev/null)"
}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
for i in $(seq "$ROUNDS"); do
    if [ $((i % 2)) = 1 ]; then order="base new"; else order="new base"; fi
    for arm in $order; do bench $arm 2A --config 2A --steps 5 --warmup 3 --no-cpu-baseline; done
done
for arm in base new; do
    VMIG_TRACE=1 bench $arm 2A_trace --config 2A --steps 5 --warmup 3 --no-cpu-baseline --dump-outputs "$OUT/dump_2A_$arm"
    bench $arm 2B --config 2B --steps 5 --warmup 3 --no-cpu-baseline --dump-outputs "$OUT/dump_2B_$arm"
    bench $arm 4 --config 4 --steps 3 --warmup 1 --dump-outputs "$OUT/dump_4_$arm"
done
python - "$OUT" <<'EOF'
import sys
from pathlib import Path
import numpy as np
out = Path(sys.argv[1])
for cfg in ("2A", "2B", "4"):
    a, b = out / f"dump_{cfg}_base", out / f"dump_{cfg}_new"
    names = sorted(p.name for p in a.glob("*.npy"))
    same = bool(names) and names == sorted(p.name for p in b.glob("*.npy")) and all(
        np.array_equal(np.load(a / n), np.load(b / n)) for n in names)
    print(f"outputs {cfg}: {'identical' if same else 'DIFFER'} ({', '.join(names)})")
EOF
