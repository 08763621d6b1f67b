#!/bin/bash
# ncu evidence of one round (run under gpurun on ONE GPU, after the same commands have exited 0 without ncu).
# usage: bash tools/gpu_profiles.sh <tag>
set -u
TAG=${1:-r02}
OUT=gpurun_out
mkdir -p $OUT
B="python bench.py --steps 2 --warmup 3 --no-e2e --no-cpu --no-scaling-legs"
$B > $OUT/${TAG}_plain_bench.json 2> $OUT/${TAG}_plain_bench.err || { echo "plain bench failed"; exit 1; }
# 1. launch list of the bench (cold-cache, serialised: shares, not absolutes)
ncu --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file $OUT/${TAG}_launches_bench.csv $B > $OUT/${TAG}_ncu_launch.log 2>&1
echo "launch list rc=$?"
# 2. FIR kernel, one launch per tap count (the timed region: skip warm-up launches 3 x 4)
timeout 900 ncu --set full --clock-control none --import-source on -k regex:"fir_tma|fir_split2" -s 12 -c 4 -f -o $OUT/${TAG}_prof_fir $B --no-chain --no-decimate > $OUT/${TAG}_ncu_fir.log 2>&1
echo "fir rc=$?"
# 3. decimating FIR: one launch per (taps, D) of the bench's `decimate` leg
python tools/decim_probe.py > $OUT/${TAG}_plain_decim.log 2>&1
timeout 900 ncu --set full --clock-control none -k regex:fir_dec -c 6 -f -o $OUT/${TAG}_prof_decim python tools/decim_probe.py > $OUT/${TAG}_ncu_decim.log 2>&1
echo "decim rc=$?"
# 4. chain at 2048 channels: FLL (duo), fused MF + symbol stage, TSC strip, BER
python tools/chain_only.py fll 2 > $OUT/${TAG}_plain_chain_fll.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:"fll_duo|symsync|tsc_strip|ber_kernel" -s 12 -c 4 -f \
  -o $OUT/${TAG}_prof_chain python tools/chain_only.py fll 2 > $OUT/${TAG}_ncu_chain.log 2>&1
echo "chain rc=$?"
# 5. the 16384-channel FLL on one GPU: fll_pair_kernel
timeout 900 ncu --set full --clock-control none --import-source on -k regex:"fll_pair" -s 3 -c 1 -f \
  -o $OUT/${TAG}_prof_chain16k python tools/fll_only.py 16384 > $OUT/${TAG}_ncu_chain16k.log 2>&1
echo "chain16k rc=$?"
# 6. modulator leg: mod_shape_kernel, one launch of 512 frames
timeout 600 ncu --set full --clock-control none --import-source on -k regex:mod_shape -s 3 -c 1 -f -o $OUT/${TAG}_prof_mod python tools/mod_probe.py 512 2 > $OUT/${TAG}_ncu_mod.log 2>&1
echo "mod rc=$?"
# condense on the box: the reports themselves are too big to travel back (64 MiB limit)
for k in fir decim chain chain16k mod; do
  python tools/ncu_summary.py $OUT/${TAG}_prof_$k.ncu-rep $OUT/${TAG}_ncu_full_${k}_summary.csv
done
for k in chain chain16k mod fir; do
  python tools/ncu_src.py $OUT/${TAG}_prof_$k.ncu-rep 40 > $OUT/${TAG}_ncu_src_$k.txt 2>&1
done
ls -la $OUT/${TAG}_prof_*.ncu-rep
rm -f $OUT/${TAG}_prof_*.ncu-rep
du -sh $OUT
