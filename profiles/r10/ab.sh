#!/bin/bash
# A/B of the in-place level 2 on one GPU. A = a built checkout of the parent commit in $1, B = this tree (built).
# Runs config 5 as A B repeated ROUNDS times, then config 2 the same way, with the outputs of every run dumped; then
# checks that all dumps of a config are identical and prints ms_per_step, e2e ms_per_step, device_bytes, scatter1
# (ms and launches per step), scatter2 and the page-list kernels per run and the spread.
# usage: profiles/r10/ab.sh PARENT_TREE OUT_DIR ROUNDS
set -u
BASE=$(cd "$1" && pwd); OUT=$(mkdir -p "$2" && cd "$2" && pwd); ROUNDS=$3; HERE=$(pwd)
DUMP=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
run() {   # tag tree config
    (cd "$2" && timeout 900 python bench.py --config "$3" --no-cpu-baseline --dump-outputs "$DUMP/$1") > "$OUT/$1.json" 2> "$OUT/$1.err"
    echo "$1 exit $?"
}
for cfg in 5 2; do
    for i in $(seq 1 "$ROUNDS"); do
        run "c${cfg}_A$i" "$BASE" $cfg
        run "c${cfg}_B$i" "$HERE" $cfg
    done
done
python "$HERE/profiles/r10/ab_summary.py" "$OUT" "$DUMP" | tee "$OUT/summary.txt"
rm -rf "$DUMP"
