#!/bin/bash
# ncu.sh -- the committed Nsight Compute captures behind profiles/ (the reference's ncu.sh:1 profiles its own binary the
# same way). Run on a B200 box (./ncu.sh <tag> [encode|decode|metrics|launches]); read the reports on the
# CPU box with scripts/ncu_export.py. Every profiled command first runs plain and must exit 0.
#   encode   : --set full of one launch of every encode kernel, headline config (8320x40000 4:2:2 q95 optimised)
#   decode   : --set full of one decode of the headline JPEG
#   metrics  : --set full of k_diff_psnr (difference map + SSD), k_idct and k_upcolor on the secondary-compression path
#   launches : per-launch device times of bench.py (gpu__time_duration only)
set -e
TAG=${1:-r02}
WHAT=${2:-encode}
OUT=gpurun_out
mkdir -p $OUT
NCU="ncu --clock-control none"
case $WHAT in
encode)
    python scripts/stage_times.py --iters 3 > $OUT/${TAG}_stage_times.jsonl
    $NCU --set full --import-source on -k regex:"k_fdct|k_pack|k_stuff|k_tables|k_scan_tiles|k_dc_edge" -s 6 -c 6 \
        -f -o $OUT/prof_${TAG} python scripts/stage_times.py --iters 3 > $OUT/${TAG}_ncu.log 2>&1
    ;;
decode)
    python scripts/decode_times.py > $OUT/${TAG}_decode_times.jsonl
    $NCU --set full --import-source on -k regex:"k_destuff|k_dec_|k_scan_u32|k_dc_scan|k_idct|k_upcolor" -s 23 -c 23 \
        -f -o $OUT/prof_${TAG}_decode python scripts/decode_times.py > $OUT/${TAG}_decode_ncu.log 2>&1
    ;;
metrics)
    python scripts/secondary_multi.py --iters 1 > $OUT/${TAG}_secondary.jsonl
    $NCU --set full --import-source on -k regex:"k_diff_psnr|k_idct|k_upcolor" -s 3 -c 3 \
        -f -o $OUT/prof_${TAG}_metrics python scripts/secondary_multi.py --iters 1 > $OUT/${TAG}_metrics_ncu.log 2>&1
    ;;
launches)
    python bench.py --steps 2 --warmup 3 > $OUT/${TAG}_bench_plain.json
    $NCU --metrics gpu__time_duration.sum -k regex:"^k_|b2j" -c 400 --csv --log-file $OUT/launches_${TAG}.csv \
        python bench.py --steps 2 --warmup 3 > $OUT/${TAG}_launches.log 2>&1
    ;;
*) echo "usage: $0 <tag> [encode|decode|metrics|launches]"; exit 2;;
esac
echo "ncu.sh $TAG $WHAT done"
