#!/bin/bash
# ncu --set full capture (with source counters) of the chain's symbol-stage kernel; usage: bash tools/gpu_ncu_chain.sh <tag> [chain|fll]
set -u
TAG=${1:-r02}
WHICH=${2:-chain}
OUT=gpurun_out
mkdir -p $OUT
python tools/chain_only.py $WHICH 2 > $OUT/${TAG}_plain_${WHICH}.log 2>&1 || { echo "plain run failed"; tail -5 $OUT/${TAG}_plain_${WHICH}.log; exit 1; }
timeout 900 ncu --set full --clock-control none --import-source on -k regex:"symsync|fll_duo|fll_pair" -c 3 -f -o $OUT/${TAG}_prof_${WHICH} \
  python tools/chain_only.py $WHICH 2 > $OUT/${TAG}_ncu_${WHICH}.log 2>&1
echo "ncu rc=$?"; tail -3 $OUT/${TAG}_ncu_${WHICH}.log
