#!/bin/bash
# round 2, GPU pass c: fused conv1x1 + context network kernel, tiled encoder-flow kernel: op tests, parity suite, bench (A/B by env switches)
mkdir -p gpurun_out
true
true
B="python bench.py --steps 20 --warmup 5 --no-cpu-baseline --secondary="
$B > gpurun_out/r2c_bench.json 2> gpurun_out/r2c_bench.err; echo "bench rc=$?"
CFPP_C1X1_CTX=0 $B > gpurun_out/r2c_bench_noc1.json 2> gpurun_out/r2c_bench_noc1.err; echo "bench (two-kernel conv1x1) rc=$?"
python - <<'P'
import json
for f in ['r2c_bench','r2c_bench_noc1']:
    try:
        d=json.loads(open(f'gpurun_out/{f}.json').read().strip().splitlines()[-1])
        print(f, round(d['value']), d['ms_per_step'], d['parity_at_bench_batch'].get('ok'))
        for n,v in sorted(d['kernels'].items(), key=lambda kv:-kv[1]['ms_per_step'])[:9]:
            print('   ', n, v['ms_per_step'], {k: s['ms_per_launch'] for k, s in v.get('by_shape', {}).items()})
    except Exception as e:
        print(f, 'ERR', e)
P
