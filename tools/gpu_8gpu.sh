#!/bin/bash
set -u
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name --format=csv,noheader | wc -l > gpurun_out/ngpus.txt
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29521"
timeout 400 $TR bench.py --gpus 8 --steps 30 --warmup 5 --no-cpu-baseline > gpurun_out/r02_bench_8gpu_c3.json 2> gpurun_out/b8_c3.err; echo "c3 rc=$?" > gpurun_out/rc.txt
timeout 500 $TR bench.py --gpus 8 --config 4 --steps 20 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/r02_bench_8gpu_c4.json 2> gpurun_out/b8_c4.err; echo "c4 rc=$?" >> gpurun_out/rc.txt
timeout 500 $TR bench.py --gpus 8 --config 5 --steps 20 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/r02_bench_8gpu_c5.json 2> gpurun_out/b8_c5.err; echo "c5 rc=$?" >> gpurun_out/rc.txt
timeout 300 python bench.py --steps 30 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/r02_bench_1of8_c3.json 2>/dev/null; echo "1gpu rc=$?" >> gpurun_out/rc.txt
python - <<'PY'
import json
for f in ('r02_bench_8gpu_c3','r02_bench_8gpu_c4','r02_bench_8gpu_c5','r02_bench_1of8_c3'):
    try:
        d=json.load(open('gpurun_out/%s.json'%f)); print(f, 'n', d['n_gpus'], round(d['value'],1), 'img/s', round(d['ms_per_step'],2), 'ms e2e', d['e2e'] and round(d['e2e']['value'],1), d['config']['grad_allreduce'], 'clk', d['clocks']['sm_mhz'], 'teacher', d['config']['teacher_fwd_ms_per_step'])
    except Exception as e: print(f,'ERR',e)
PY
cat gpurun_out/rc.txt
