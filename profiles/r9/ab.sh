#!/bin/bash
# A/B of the level-2 stage on one GPU. A = a built checkout of the parent commit in $1, B = this tree (built);
# extra arms "TAG=ENV" run this tree with one environment variable set (variants/ was taken with a build whose
# PSKMER_SC2=dbuf selected the double-buffered k_scatter2, arm D; that form was removed after it lost).
# Runs config 5 as A B [..] repeated ROUNDS times, then config 2 the same way, with the outputs of every run dumped;
# then checks that all dumps of a config are identical and prints ms_per_step, scatter2 and the page-list kernels per
# run and the spread.
# usage: profiles/r9/ab.sh PARENT_TREE OUT_DIR ROUNDS [TAG=ENV ...]
set -u
BASE=$(cd "$1" && pwd); OUT=$(mkdir -p "$2" && cd "$2" && pwd); ROUNDS=$3; shift 3; HERE=$(pwd)
DUMP=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
run() {   # tag tree config [env]
    (cd "$2" && env ${4:-} timeout 900 python bench.py --config "$3" --no-cpu-baseline --dump-outputs "$DUMP/$1") > "$OUT/$1.json" 2> "$OUT/$1.err"
    echo "$1 exit $?"
}
for cfg in 5 2; do
    for i in $(seq 1 "$ROUNDS"); do
        run "c${cfg}_A$i" "$BASE" $cfg
        run "c${cfg}_B$i" "$HERE" $cfg
        for arm in "$@"; do run "c${cfg}_${arm%%=*}$i" "$HERE" $cfg "${arm#*=}"; done
    done
done
python "$HERE/profiles/r9/ab_summary.py" "$OUT" "$DUMP" | tee "$OUT/summary.txt"
rm -rf "$DUMP"
