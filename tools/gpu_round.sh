#!/bin/bash
# One GPU-box session: GPU parity tests, smoke, bench (ours + reference arm), ncu launch list, ncu --set full of the top kernels.
# Usage (under gpurun): bash tools/gpu_round.sh [tag]      outputs -> gpurun_out/<tag>_*
TAG=${1:-r1}
O=gpurun_out
mkdir -p $O
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $O/${TAG}_gpu.txt
echo "##### pytest -m gpu"
timeout 900 python -m pytest tests -x -q -m gpu 2>&1 | tail -15 | tee $O/${TAG}_pytest.log
echo "##### smoke"
timeout 300 python __graft_entry__.py smoke 2>&1 | tail -5 | tee $O/${TAG}_smoke.log
echo "##### bench"
timeout 600 python bench.py 2> $O/${TAG}_bench.err | tee $O/${TAG}_bench.json
tail -5 $O/${TAG}_bench.err
if [ "${SKIP_NCU:-0}" != "1" ]; then
echo "##### ncu launch list"
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/${TAG}_launches.csv \
    python bench.py --steps 3 --warmup 3 > $O/${TAG}_ncu_bench.log 2>&1
tail -2 $O/${TAG}_ncu_bench.log
echo "##### ncu full"
# one forward's kernels of the eager warm-up step (one DiT block and a half); the report stays in /tmp unless it is small:
# gpurun copies back at most 64 MiB
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'tc_gemm|tc_scores|cross_fused|softmax|adaln|layernorm|cfg_update_kernel' -s 20 -c 12 \
    -o /tmp/${TAG}_prof -f python tools/step_profile.py --steps 3 > $O/${TAG}_ncu_full.log 2>&1
tail -2 $O/${TAG}_ncu_full.log
ncu -i /tmp/${TAG}_prof.ncu-rep --page raw --csv > $O/${TAG}_full_raw.csv 2>/dev/null
SZ=$(stat -c %s /tmp/${TAG}_prof.ncu-rep); echo "report size $SZ"
if [ "$SZ" -lt 30000000 ]; then cp /tmp/${TAG}_prof.ncu-rep $O/; fi
fi
echo "##### reference arm"
timeout 600 python bench.py --impl reference --steps 5 --warmup 1 | tee $O/${TAG}_bench_ref.json
ls -la $O
