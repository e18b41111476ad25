#!/bin/bash
# Round-2 profile on the GPU box: ncu launch list of the default bench command (C4 on one GPU), then ncu --set full of one
# forward's kernels of a C2 step (tools/step_profile.py).  Usage (under gpurun): bash tools/gpu_profile2.sh <tag> [skip] [count]
TAG=${1:-r2}
O=gpurun_out; mkdir -p $O
timeout 1200 ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file $O/${TAG}_launches.csv \
    python bench.py --steps 3 --warmup 3 > $O/${TAG}_ncu_bench.log 2>&1
tail -1 $O/${TAG}_ncu_bench.log | cut -c1-200
# kernels of one eager step (skip the text-context / finalize launches and the first steps)
timeout 1200 ncu --set full --clock-control none --import-source on \
    -k regex:'tc_gemm|flash_attn768|cross_fused|layernorm|adaln|cfg_update_kernel' -s ${2:-40} -c ${3:-14} -f -o /tmp/${TAG}_full \
    python tools/step_profile.py --steps 3 > $O/${TAG}_ncu_full.log 2>&1
tail -2 $O/${TAG}_ncu_full.log
ncu -i /tmp/${TAG}_full.ncu-rep --page raw --csv > $O/${TAG}_full_raw.csv 2>/dev/null
SZ=$(stat -c %s /tmp/${TAG}_full.ncu-rep); echo "report size $SZ"
if [ "$SZ" -lt 40000000 ]; then cp /tmp/${TAG}_full.ncu-rep $O/; fi
