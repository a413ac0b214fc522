#!/bin/bash
# 8-GPU pass: TP=2/4/8 parity tests, TP=8 bench, decode timeline
mkdir -p gpurun_out
timeout 1200 python -m pytest tests/test_tp_gpu.py -m gpu -q --timeout 900 > gpurun_out/r02_tp_tests.log 2>&1
echo "tp tests rc=$?"; tail -4 gpurun_out/r02_tp_tests.log | cut -c1-600
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29713"
for cfg in "default X=1"; do
  set -- $cfg; name=$1; shift
  env "$@" timeout 600 $TR bench.py --gpus 8 --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/r02_tp8_$name.json 2> gpurun_out/r02_tp8_$name.err
  python -c "
import json;d=json.load(open('gpurun_out/r02_tp8_$name.json'))
print('$name', d['value'],'tok/s ttft',d['ttft_p50_ms'],'ms/step',d['decode_ms_per_token_step'],'prefill frac',d['roofline_prefill']['frac'], d['parity_check'])" || tail -5 gpurun_out/r02_tp8_$name.err
done
for cfg in "default X=1"; do
  set -- $cfg; name=$1; shift
  env "$@" LAYERS=8 ROWS=24 timeout 300 $TR tools/timeline.py > gpurun_out/r02_tl_tp8_$name.txt 2>&1
  echo "== $name"; grep -E "step span" gpurun_out/r02_tl_tp8_$name.txt; grep -vE "^\[|^\*|NCCL|OMP|^$" gpurun_out/r02_tl_tp8_$name.txt | sed -n 12,22p | cut -c1-115
done
