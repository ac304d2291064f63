#!/bin/bash
# Round 3: piece staging variants on one GPU, in one session.  PATCHED_TREE is the parent commit with
# profiles/r03_piece_staging.patch applied and built; the patch reads VMIG_PIECES (pieces of 1 MiB per reader) and
# VMIG_PIECE_SPIN (1 = poll the piece's event instead of a blocking wait).  Every run carries VMIG_TRACE=1.
# usage: profiles/scripts/r3_piece_variants.sh BASE_TREE PATCHED_TREE OUT_DIR
set -u
BASE=$(cd "$1" && pwd); EXP=$(cd "$2" && pwd); mkdir -p "$3"; OUT=$(cd "$3" && pwd)
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
run() {  # tag tree env...
    local tag=$1 dir=$2; shift 2
    (cd "$dir" && env "$@" VMIG_TRACE=1 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline --config $CFG) >> "$OUT/${CFG}_$tag.jsonl" 2>> "$OUT/${CFG}_$tag.err"
    echo "$CFG $tag $(tail -n 1 "$OUT/${CFG}_$tag.jsonl" | python -c 'import json,sys; d=json.loads(sys.stdin.read()); print(d["value"], d["ms_per_step"])' 2>/dev/null)"
}
for CFG in 2A 2B 2A; do
    run base "$BASE" X=1
    run p4block "$EXP" VMIG_PIECES=4
    run p16block "$EXP" VMIG_PIECES=16
    run p4spin "$EXP" VMIG_PIECES=4 VMIG_PIECE_SPIN=1
    run p16spin "$EXP" VMIG_PIECES=16 VMIG_PIECE_SPIN=1
done
