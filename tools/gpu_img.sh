#!/bin/bash
set -u
mkdir -p gpurun_out
T="timeout 1500 python -m pytest -q --timeout 300 --timeout-method thread -p no:cacheprovider"
$T tests/test_gpu_gemm.py -m gpu -k "patch_embed_image" > gpurun_out/t_img.log 2>&1; echo "img rc=$?" > gpurun_out/rc.txt
grep -E "passed|failed|^E  " gpurun_out/t_img.log | cut -c1-220 | head -12
$T tests -m gpu > gpurun_out/t_all.log 2>&1; echo "all rc=$?" >> gpurun_out/rc.txt
grep -E "passed|failed|^FAILED" gpurun_out/t_all.log | tail -6
GB_NOLIB=1 GB_ONLY=wgrad python tools/gemm_bench.py 384 768 1024 2>&1 | grep -v Warn > gpurun_out/wgrad_new.txt; cat gpurun_out/wgrad_new.txt
B="timeout 600 python bench.py --no-cpu-baseline --no-e2e --steps 20 --warmup 5"
$B --config 5 --steps 10 > gpurun_out/c5.json 2>/dev/null
$B --config 2 > gpurun_out/c2.json 2>/dev/null
python - <<'PY'
import json
for f in ('c5','c2'):
    try:
        d=json.load(open('gpurun_out/%s.json'%f)); print(f, round(d['value'],1), round(d['ms_per_step'],2), d['clocks']['sm_mhz'], d['roofline']['by_shape_us'])
    except Exception as e: print(f, 'ERR', e)
PY
cat gpurun_out/rc.txt
