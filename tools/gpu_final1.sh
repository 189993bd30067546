#!/bin/bash
set -u
mkdir -p gpurun_out
T="timeout 1500 python -m pytest -q --timeout 300 --timeout-method thread -p no:cacheprovider"
$T tests -m gpu > gpurun_out/t_all.log 2>&1; echo "all rc=$?" > gpurun_out/rc.txt
grep -E "passed|failed|^FAILED" gpurun_out/t_all.log | tail -6
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?" >> gpurun_out/rc.txt; tail -1 gpurun_out/smoke.log
python tools/patch_embed_bench.py 256 224 768 2>&1 | grep -v Warn > gpurun_out/patch_embed2.txt; cat gpurun_out/patch_embed2.txt
timeout 900 python bench.py --steps 50 --warmup 5 --breakdown > gpurun_out/r02_bench_c3.json 2> gpurun_out/r02_bench_c3.err; echo "c3 rc=$?" >> gpurun_out/rc.txt
for c in 2 4 5; do
  timeout 900 python bench.py --config $c --steps 50 --warmup 5 --breakdown > gpurun_out/r02_bench_c$c.json 2> gpurun_out/r02_bench_c$c.err; echo "c$c rc=$?" >> gpurun_out/rc.txt
done
python - <<'PY'
import json
for f in ('r02_bench_c3','r02_bench_c2','r02_bench_c4','r02_bench_c5'):
    try:
        d=json.load(open('gpurun_out/%s.json'%f)); r=d['roofline']
        print(f, round(d['value'],1), 'img/s', round(d['ms_per_step'],2), 'ms  e2e', d['e2e'] and round(d['e2e']['value'],1), ' clk', d['clocks']['sm_mhz'], ' frac_sust %.3f'%d['model_flops']['frac_of_measured_sustained'], ' roof %.3f %s %.1fus'%(r['frac'], r['kernel'][-30:], r['us_per_launch']), 'teacher', d['config']['teacher_fwd_ms_per_step'], 'cpu', d.get('cpu_baseline',{}).get('value'))
    except Exception as e: print(f, 'ERR', e)
PY
cat gpurun_out/rc.txt
