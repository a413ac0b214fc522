#!/bin/bash
mkdir -p gpurun_out
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29712"
for cfg in "own64 X=1"; do
  set -- $cfg; name=$1; shift
  env "$@" PHASE=prefill LAYERS=4 ROWS=90 timeout 300 $TR tools/timeline.py > gpurun_out/r02_tl_prefill_tp2_$name.txt 2>&1
  echo "== $name"; grep -E "step span|other" gpurun_out/r02_tl_prefill_tp2_$name.txt | head -8 | cut -c1-120
done
timeout 600 python -m pytest tests/test_tp_gpu.py -m gpu -q --timeout 800 -x -k tp2 2>&1 | tail -2
