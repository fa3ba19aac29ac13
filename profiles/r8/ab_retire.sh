#!/bin/bash
# A/B after retiring the losing variants (bucket-kernel TMA ring, staged-byte FASTA write pass, PSKMER_PAGED,
# PSKMER_CHI2=masked) on one GPU. A = a built checkout of the parent commit in $1, B = this tree (built).
# Runs config 5 as A B A B A B, then config 2 the same way, with the outputs of every run dumped; then checks that all
# dumps of a config are identical and prints ms_per_step, bucket_count, bucket_build and decode_write per run and the
# spread.
# usage: profiles/r8/ab_retire.sh PARENT_TREE OUT_DIR
set -u
BASE=$(cd "$1" && pwd); OUT=$(mkdir -p "$2" && cd "$2" && pwd); HERE=$(pwd)
DUMP=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
run() {   # tag tree config
    (cd "$2" && timeout 900 python bench.py --config "$3" --no-cpu-baseline --dump-outputs "$DUMP/$1") > "$OUT/$1.json" 2> "$OUT/$1.err"
    echo "$1 exit $?"
}
for cfg in 5 2; do
    for i in 1 2 3; do run "c${cfg}_A$i" "$BASE" $cfg; run "c${cfg}_B$i" "$HERE" $cfg; done
done
python "$HERE/profiles/r8/ab_summary.py" "$OUT" "$DUMP" | tee "$OUT/summary.txt"
rm -rf "$DUMP"
