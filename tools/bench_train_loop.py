"""Time the training loop body as the reference writes it (experiment_ad.py:204-213), eager against CUDA-graph replay of log_prob
(FlowSequential.enable_cuda_graphs(training=True)), the two arms interleaved in one process.

Per step: CPU batch .to(device), dim_inv * model.log_prob, NaN scrub, loss with constants built on the CPU per call, zero_grad(),
backward(), optimizer.step() with the optimizer the launcher installs (contextflow_b200.optim.FusedAdamW), .item() x 3.  Per arm:
median ms per step on the host clock (the .item() calls synchronise), libcfpp launches issued from the host per step, peak device memory,
and how often FusedAdamW rebuilt its pointer tables in the timed steps.

python tools/bench_train_loop.py [--configs cfg1,cfg2,cfg3,cfg4] [--batches 256,2048] [--steps 20] [--warmup 3] [--rounds 3] [--out FILE]"""
import argparse, copy, json, os, statistics, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.nn as nn
from contextflow_b200 import _cabi, builder, synth
from contextflow_b200.optim import FusedAdamW

# experiment_ad.py:56-61: the specialists and the image generalist with a classifier term, SMAP's generalist (M = 1) without
LOSS = {'cfg1': (1e-2, True), 'cfg2': (1e-2, True), 'cfg3': (1e-2, True), 'cfg4': (1e2, False)}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return {'torch_device_name': torch.cuda.get_device_name(0), 'nvidia_smi': q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


def loss_body(model, x, c, gt, data_size, alpha, criterion):
    """experiment_ad.py:204-209 as written: the constants are CPU tensors built on every call, the NaN scrub edits logp in place."""
    dim_inv = 1.0 / torch.prod(torch.tensor(data_size))
    log_theta = nn.LogSigmoid()
    logp = dim_inv * model.log_prob(x, context=c)
    logp[logp != logp] = 0.0
    if criterion:
        sup = nn.CrossEntropyLoss()(logp, gt)
        uns = -alpha * log_theta(torch.logsumexp(logp, -1)).mean()
    else:
        uns = -alpha * log_theta(logp).mean()
        sup = torch.zeros_like(uns)
    return sup + uns, sup, uns


class Arm:
    def __init__(self, name, model, dev):
        self.name, self.model, self.dev = name, model, dev
        self.opt = FusedAdamW([p for p in model.parameters() if p.requires_grad], lr=1e-4)
        self.ms, self.launches, self.rebuilds, self.peak = [], [], 0, 0

    def step(self, batch, conf, alpha, criterion):
        x, c, gt = batch
        x, c, gt = x.to(self.dev), c.to(self.dev), gt.to(self.dev)
        cost, sup, uns = loss_body(self.model, x, c, gt, conf['data_size'], alpha, criterion)
        self.opt.zero_grad()
        cost.backward()
        self.opt.step()
        return cost.item(), sup.item(), uns.item()


def measure(name, B, a, dev):
    conf = synth.CONFIGS[name]
    alpha, criterion = LOSS[name]
    base = builder.build_named(conf)
    sd = base.state_dict(); synth.fill_state(sd, 'bench'); base.load_state_dict(sd)
    base = base.to(dev).train()
    C, H, W = conf['data_size']
    g = torch.Generator().manual_seed(99)
    batches = [((torch.randint(0, 256, (B, C, H, W), generator=g).float() if conf['image'] else torch.rand(B, C, H, W, generator=g)),
                torch.stack([torch.randint(0, k, (B,), generator=g) for k in conf['contexts']], 1),
                torch.randint(0, conf['mixtures'], (B,), generator=g)) for _ in range(3)]
    with torch.no_grad():                                         # ActNorm's first-batch initialisation, shared by both arms
        base.log_prob(batches[0][0].to(dev), batches[0][1].to(dev))
    arms = [Arm('eager', copy.deepcopy(base), dev), Arm('graphed', copy.deepcopy(base).enable_cuda_graphs(training=True), dev)]
    del base
    torch.manual_seed(1)
    for arm in arms:
        for i in range(a.warmup):                                 # the graphed arm's first call runs eagerly, the second captures
            arm.step(batches[i % 3], conf, alpha, criterion)
    losses = {}
    for r in range(a.rounds):
        for arm in arms:
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats(dev)
            plans = dict(arm.opt._plans)
            l0 = _cabi.launch_count()
            for i in range(a.steps):
                t0 = time.perf_counter()
                losses[arm.name] = arm.step(batches[i % 3], conf, alpha, criterion)
                arm.ms.append(1e3 * (time.perf_counter() - t0))
                arm.rebuilds += sum(1 for gi, p in arm.opt._plans.items() if plans.get(gi) is not p)
                plans = dict(arm.opt._plans)
            arm.launches.append((_cabi.launch_count() - l0) / a.steps)
            arm.peak = max(arm.peak, torch.cuda.max_memory_allocated(dev))
    res = {'workload': name, 'batch': B, 'steps_per_round': a.steps, 'rounds': a.rounds,
           'note': 'both arms resident on the device during every timed step; peak = max_memory_allocated over an arm\'s timed steps'}
    for arm in arms:
        res[arm.name] = {'ms_per_step_median': round(statistics.median(arm.ms), 3), 'ms_per_step_min': round(min(arm.ms), 3),
                         'libcfpp_launches_per_step': max(arm.launches), 'peak_allocated_MB': round(arm.peak / 2 ** 20, 1),
                         'fused_adamw_table_rebuilds_in_timed_steps': arm.rebuilds, 'last_losses': losses[arm.name]}
        if arm.name == 'graphed':
            res[arm.name]['training_graph_entries'] = len(arm.model._graphed_train._entries)
    res['speedup_median'] = round(res['eager']['ms_per_step_median'] / res['graphed']['ms_per_step_median'], 3)
    del arms
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='cfg1,cfg2,cfg3,cfg4'); ap.add_argument('--batches', default='256,2048')
    ap.add_argument('--steps', type=int, default=20); ap.add_argument('--warmup', type=int, default=3); ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON result to this file')
    a = ap.parse_args()
    if a.warmup < 2:
        ap.error('--warmup must be at least 2: the graphed arm captures at its second call')
    if not torch.cuda.is_available():
        raise SystemExit('bench_train_loop.py measures on a CUDA device; none is visible')
    dev = torch.device('cuda', 0)
    out = {'tool': 'tools/bench_train_loop.py', 'card': card(), 'torch': torch.__version__, 'results': []}
    for name in a.configs.split(','):
        for B in (int(b) for b in a.batches.split(',')):
            r = measure(name, B, a, dev)
            out['results'].append(r)
            print(json.dumps(r), flush=True)
    print(json.dumps(out))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
