#!/bin/bash
mkdir -p gpurun_out
timeout 900 python bench.py --steps 3 --warmup 3 --no-cpu-baseline > gpurun_out/r02_bench_quick.json 2> gpurun_out/r02_bench_quick.err
python -c "
import json;d=json.load(open('gpurun_out/r02_bench_quick.json'))
print('N=1', d['value'],'tok/s e2e',d['e2e']['value'],'ttft',d['ttft_p50_ms'],'ms/step',d['decode_ms_per_token_step'],'frac',d['roofline']['frac'],'prefill frac',d['roofline_prefill']['frac'],d['clocks'], d['parity_check']['ok'])" || tail -5 gpurun_out/r02_bench_quick.err
echo "prefill gemm: $(python tools/prefill_gemm.py 2>&1 | tail -1)"
timeout 600 python -m pytest tests/test_engine_gpu.py tests/test_kernels_gpu.py -m gpu -q --timeout 500 2>&1 | tail -2
