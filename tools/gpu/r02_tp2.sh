#!/bin/bash
# 2-GPU sanity of the round-2 tensor-parallel changes (two-shot not active at tp=2)
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_tp_gpu.py -m gpu -q --timeout 800 -x -k tp2 > gpurun_out/r02_tp2_tests.log 2>&1
echo "tp2 tests rc=$?"; tail -5 gpurun_out/r02_tp2_tests.log | cut -c1-400
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29711"
for cfg in "default X=1"; do
  set -- $cfg; name=$1; shift
  env "$@" timeout 600 $TR bench.py --gpus 2 --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/r02_tp2_$name.json 2> gpurun_out/r02_tp2_$name.err
  python -c "
import json;d=json.load(open('gpurun_out/r02_tp2_$name.json'))
print('$name', d['value'],'tok/s ttft',d['ttft_p50_ms'],'ms/step',d['decode_ms_per_token_step'],'prefill frac',d['roofline_prefill']['frac'], d['parity_check'])" || tail -5 gpurun_out/r02_tp2_$name.err
done
