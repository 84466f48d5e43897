#!/bin/bash
# One-visit A/B of the RANSAC scoring change: a built tree of the parent commit ($1) against this tree,
# `bench.py` runs alternating between the two (RUNS per side), then --dump-outputs of both compared byte
# for byte, the card's name and power limit read in the same visit.  Summary: profiles/rs_ab_summary.py.
# usage: bash profiles/rs_ab.sh PARENT_TREE OUT_DIR [TAG] [RUNS]
set -u
PARENT=$(cd "$1" && pwd); mkdir -p "$2"; O=$(cd "$2" && pwd); TAG=${3:-rs_ab}; RUNS=${4:-3}
NEW=$PWD
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $O/${TAG}_gpu.txt
for i in $(seq 1 $RUNS); do
  for side in parent new; do
    if [ $side = parent ]; then d=$PARENT; else d=$NEW; fi
    (cd $d && timeout 600 python bench.py --no-cpu-baseline --no-e2e) > $O/${TAG}_${side}_$i.json 2> $O/${TAG}_${side}_$i.err
    echo "$side $i rc=$?"
  done
done
for side in parent new; do
  if [ $side = parent ]; then d=$PARENT; else d=$NEW; fi
  (cd $d && timeout 600 python bench.py --no-cpu-baseline --no-e2e --no-configs --steps 3 --warmup 1 \
     --dump-outputs $O/${TAG}_dump_$side) > /dev/null 2> $O/${TAG}_dump_$side.err
  echo "dump $side rc=$?"
done
python profiles/rs_ab_summary.py $O $TAG $RUNS | tee $O/${TAG}.json
