#!/bin/bash
# flash_attn768q experiments: timelines (trace build) + timings with and without the LayerNorm stage at the C2 and the C4 problem size
O=gpurun_out; mkdir -p $O
TL=ditto_tts_b200/libditto_b200_trace.so
timeout 200 python tools/f7_trace.py --lib $TL --n 32 --limit 300 > $O/f7x_trace_n32.txt 2>&1; tail -2 $O/f7x_trace_n32.txt
timeout 200 python tools/f7_trace.py --lib $TL --n 256 --limit 300 > $O/f7x_trace_n256.txt 2>&1; tail -2 $O/f7x_trace_n256.txt
for n in 32 256; do
  echo "n=$n:       $(timeout 120 python tools/attn768_bench.py --n $n --iters 7 | tail -1)"
  echo "n=$n noln:  $(timeout 120 python tools/attn768_bench.py --n $n --iters 7 --noln 1 | tail -1)"
done 2>&1 | tee $O/f7x_switches.txt
