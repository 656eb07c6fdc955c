#!/bin/bash
mkdir -p gpurun_out
timeout 300 python -m pytest tests/test_gpu_training.py -q -m gpu -k "conv2d_family" --timeout 120 > gpurun_out/r2bb_conv.log 2>&1; echo "conv tests rc=$?"; tail -2 gpurun_out/r2bb_conv.log
timeout 600 python tools/bench_training.py --workload cfg2 --batch 8192 --steps 5 --warmup 2 --graph > gpurun_out/r2bb_train_cfg2.json 2> gpurun_out/r2bb_train.err; echo "train rc=$?"
python - <<P
import json
d=json.loads(open('gpurun_out/r2bb_train_cfg2.json').read().strip().splitlines()[-1])
ks=d['kernels']; print('cfg2 training', d['value'], d['ms_per_step'], d.get('loss'), {k: round(ks[k]['ms_per_step'],1) for k in ('conv2d_bwd_data','gmm_ctx_train_bwd','gmm_ctx_train_fwd')})
P
CFPP_PROFILE_RANGE=1 timeout 600 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
  --log-file gpurun_out/r2bb_launches_train_cfg2.csv python tools/bench_training.py --workload cfg2 --batch 8192 --steps 1 --warmup 2 > gpurun_out/r2bb_ncu_train.log 2>&1; echo "ncu launches rc=$?"
