#!/bin/bash
# Round profile on the GPU box: bench line, ncu launch list of the bench command, ncu --set full of one layer's kernels.
TAG=${1:-r1}
O=gpurun_out; mkdir -p $O
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $O/${TAG}_gpu.txt
timeout 600 python bench.py 2> $O/${TAG}_bench.err | tee $O/${TAG}_bench.json | cut -c1-600
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 700 --csv --log-file $O/${TAG}_launches.csv \
    python bench.py --steps 3 --warmup 3 > $O/${TAG}_ncu_bench.log 2>&1
tail -1 $O/${TAG}_ncu_bench.log | cut -c1-200
# one forward's kernels of the eager warm-up step inside step_profile (skip the text-context / finalize launches)
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'tc_gemm|tc_scores|layernorm|adaln|cfg_update_kernel|softmax' -s ${2:-20} -c ${3:-14} -f -o /tmp/${TAG}_full \
    python tools/step_profile.py --steps 3 > $O/${TAG}_ncu_full.log 2>&1
tail -2 $O/${TAG}_ncu_full.log
ncu -i /tmp/${TAG}_full.ncu-rep --page raw --csv > $O/${TAG}_full_raw.csv 2>/dev/null
SZ=$(stat -c %s /tmp/${TAG}_full.ncu-rep); echo "report size $SZ"
if [ "$SZ" -lt 40000000 ]; then cp /tmp/${TAG}_full.ncu-rep $O/; fi
timeout 300 python bench.py --impl reference --steps 5 --warmup 1 | tee $O/${TAG}_bench_ref.json | cut -c1-300
