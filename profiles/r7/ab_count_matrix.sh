#!/bin/bash
# A/B of the -rc / prediction counts on one GPU: A = a built checkout of the parent commit in $1 (one ps_lookup per
# sample), B = this tree (built; one ps_count_matrix call). Config 5 as A B A B A B, then config 2 the same way;
# then prints the times per side and whether every run's counts were identical.
# usage: profiles/r7/ab_count_matrix.sh PARENT_TREE OUT_DIR
set -u
BASE=$(cd "$1" && pwd); OUT=$(mkdir -p "$2" && cd "$2" && pwd); HERE=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
run() {   # tag tree config
    timeout 1200 python "$HERE/profiles/r7/count_matrix.py" --tree "$2" --config "$3" > "$OUT/$1.json" 2> "$OUT/$1.err"
    echo "$1 exit $?"
}
for cfg in 5 2; do
    for i in 1 2 3; do run "c${cfg}_A$i" "$BASE" $cfg; run "c${cfg}_B$i" "$HERE" $cfg; done
done
python "$HERE/profiles/r7/count_matrix.py" --summary "$OUT" | tee "$OUT/summary.txt"
