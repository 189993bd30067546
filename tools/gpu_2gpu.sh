#!/bin/bash
set -u
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name --format=csv > gpurun_out/gpus.txt
T="timeout 1500 python -m pytest -q --timeout 600 --timeout-method thread -p no:cacheprovider"
$T tests/test_gpu_dist.py tests/test_gpu_gemm.py -m gpu > gpurun_out/t_dist.log 2>&1; echo "dist rc=$?" > gpurun_out/rc.txt
grep -E "passed|failed|^FAILED|^E  " gpurun_out/t_dist.log | cut -c1-300 | tail -12
python tools/patch_embed_bench.py 256 224 768 2>&1 | grep -v Warn > gpurun_out/patch_embed3.txt; cat gpurun_out/patch_embed3.txt
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511"
timeout 600 $TR bench.py --gpus 2 --steps 20 --warmup 5 --no-cpu-baseline > gpurun_out/r02_bench_2gpu_c3.json 2> gpurun_out/b2.err; echo "b2 rc=$?" >> gpurun_out/rc.txt
python - <<'PY'
import json
for f in ('r02_bench_2gpu_c3',):
    try:
        d=json.load(open('gpurun_out/%s.json'%f)); print(f, round(d['value'],1), round(d['ms_per_step'],2), d['e2e'] and round(d['e2e']['value'],1), d['config']['grad_allreduce'])
    except Exception as e: print(f,'ERR',e)
PY
cat gpurun_out/rc.txt
