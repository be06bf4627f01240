#!/bin/bash
# Round-2 measurement recipe (each block is one run on a B200; outputs land in OUTDIR, the summaries that are
# judged are copied to profiles/ -- see profiles/r02_summary.md).  1 GPU unless a line says otherwise.
# Usage: bash tools/final_measure.sh OUTDIR
OUT=${1:?usage: bash tools/final_measure.sh OUTDIR}
mkdir -p "$OUT"
# parity + sanitizer
(time python -m pytest tests -m gpu -q) > $OUT/final_pytest.log 2>&1; tail -3 $OUT/final_pytest.log
bash tools/sanitize.sh
# bench lines (driver-style: --steps 20 --warmup 5, and long runs)
for wl in default scannet c4 grid c5; do
  python bench.py --workload $wl --steps 20 --warmup 5 --no-cpu-baseline 2>/dev/null | tail -1 > $OUT/final_bench_$wl.json
done
python bench.py --steps 100 --warmup 5 2>/dev/null | tail -1 > $OUT/final_bench_default_100.json
python bench.py --impl reference --steps 20 --warmup 5 2>/dev/null | tail -1 > $OUT/final_bench_reference.json
# launch list of the bench command (shares, not absolutes) and ncu captures of the dominant kernels
ncu --metrics gpu__time_duration.sum --clock-control none -s 60 -c 120 --csv --log-file $OUT/final_launches.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2>&1
# kernel_time.py times with eng.profile(True), which runs every chunk as one wave; its 3 warm-up steps before that run
# the 211-tile chunk as two waves (2 chain + 2 dW launches each), so the 211-tile captures skip 6 launches
ncu --set full --clock-control none --import-source on -k regex:tc_chain -s 6 -c 1 -o $OUT/final_chain_211 -f \
    python tools/kernel_time.py bf16x3g 1000 > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:tc_chain -s 3 -c 1 -o $OUT/final_chain_148 -f \
    python tools/kernel_time.py bf16x3g 701 > /dev/null 2>&1
ncu --set full --clock-control none -k regex:tc_dw -s 6 -c 1 -o $OUT/final_dw_211 -f \
    python tools/kernel_time.py bf16x3g 1000 > /dev/null 2>&1
# here (no GPU): python tools/update_traffic.py bf16x3g default $OUT/final_chain_211.ncu-rep "<command>"
#                python tools/ncu_summary.py $OUT/final_chain_148.ncu-rep profiles/<name>.json "<note>"
# multi-GPU (N GPUs): N=2|8 bash tools/n2_check.sh
