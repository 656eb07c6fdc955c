"""Time the training direction of StudentMixtureDistribution (`--dist tdist`) on the GPU.

1. The prior alone, forward + backward (training.StudentMixtureFn: cfpp_student_prep, cfpp_student_train_fwd, cfpp_student_train_bwd),
   against torch eager autograd over oracle.flow_oracle.student_mixture_log_prob in float32 on the same GPU; and the input-gradient pass
   (cfpp_student_train_bwd without parameter gradients) on its own, with the HBM floor of its traffic (x read, dx written: the table stays
   in L2) and its rate in component-element evaluations per second.
2. A whole training step (the loop body of tools/bench_train_loop.py, FusedAdamW) of a model whose `dist` is replaced by a Student-t
   mixture of the same size and M: the cfg1 stack (prior 32x8x8, M = 10) at B = 4096 and the cfg4 stack (prior 26x8x1, M = 1) at B = 8192,
   eager against FlowSequential.enable_cuda_graphs(training=True), the two arms interleaved.

python tools/bench_student_train.py [--configs cfg1,cfg4] [--iters 20] [--steps 10] [--warmup 3] [--rounds 3] [--out FILE]"""
import argparse, copy, json, os, statistics, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import torch
from bench_train_loop import LOSS, Arm, card
from contextflow_b200 import builder, ops, synth
from contextflow_b200.layers import StudentMixtureDistribution
from oracle import flow_oracle as O

BATCH = {'cfg1': 4096, 'cfg4': 8192}
HBM_BYTES_PER_S = 7.7e12            # HGX B200 data sheet, one GPU


def events_ms(fn, iters):
    """Median of `iters` CUDA-event timings of fn() (after two warm-up calls)."""
    for _ in range(2):
        fn()
    out = []
    for _ in range(iters):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record()
        torch.cuda.synchronize()
        out.append(s.elapsed_time(e))
    return statistics.median(out)


def student(size, M, dev):
    dist = StudentMixtureDistribution(tuple(size), mixtures=M)
    sd = dist.state_dict(); synth.fill_state(sd, 'bench_student'); dist.load_state_dict(sd)
    return dist.to(dev)


def prior_alone(size, M, B, iters, dev):
    dist = student(size, M, dev)
    gen = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn((B,) + tuple(size), device=dev, generator=gen).requires_grad_(True)
    g = torch.randn((B, M), device=dev, generator=gen)
    params = [getattr(dist, k) for k in ('mG', 'sG', 'wG', 'mS', 'sS', 'wS')]

    def kernels():
        dist.log_prob(x).backward(g)

    P = {k: getattr(dist, k) for k in ('mG', 'sG', 'wG', 'mS', 'sS', 'wS', 'vS')}

    def torch_eager():
        O.student_mixture_log_prob(P, x).backward(g)

    with torch.no_grad():
        table = dist._tables.get('student', params + [dist.vS], lambda: ops.student_table(*[p.detach() for p in params + [dist.vS]]))
    _, resp = ops.student_train_fwd(x.detach(), table, M, dist.K)

    def dx_pass():
        ops.student_train_bwd(x.detach(), table, *[p.detach() for p in (dist.sG, dist.wG, dist.sS, dist.wS)], resp, g, need_dx=True,
                              need_params=False)

    n = x[0].numel()
    res = {'size': list(size), 'M': M, 'K': dist.K, 'B': B, 'kernels_fwd_bwd_ms': round(events_ms(kernels, iters), 4)}
    dx_ms = events_ms(dx_pass, iters)
    evals = B * M * dist.K * n
    res['dx_pass'] = {'ms': round(dx_ms, 4), 'hbm_floor_ms': round(8.0 * B * n / HBM_BYTES_PER_S * 1e3, 4),
                      'component_element_evals_per_s': float(f'{evals / (dx_ms * 1e-3):.4g}')}
    del resp
    torch.cuda.empty_cache()
    try:
        res['torch_eager_autograd_fp32_ms'] = round(events_ms(torch_eager, max(3, iters // 4)), 4)
    except torch.cuda.OutOfMemoryError:
        res['torch_eager_autograd_fp32_ms'] = 'out of memory'
    res['speedup_vs_torch_eager'] = (round(res['torch_eager_autograd_fp32_ms'] / res['kernels_fwd_bwd_ms'], 2)
                                     if isinstance(res['torch_eager_autograd_fp32_ms'], float) else None)
    for p in params:
        p.grad = None
    torch.cuda.empty_cache()
    return res


def training_step(name, B, a, dev):
    conf = synth.CONFIGS[name]
    alpha, criterion = LOSS[name]
    base = builder.build_named(conf)
    sd = base.state_dict(); synth.fill_state(sd, 'bench'); base.load_state_dict(sd)
    base.dist = StudentMixtureDistribution(tuple(base.dist.size), mixtures=conf['mixtures'])
    sd = base.dist.state_dict(); synth.fill_state(sd, 'bench_student'); base.dist.load_state_dict(sd)
    base = base.to(dev).train()
    C, H, W = conf['data_size']
    g = torch.Generator().manual_seed(99)
    batches = [((torch.randint(0, 256, (B, C, H, W), generator=g).float() if conf['image'] else torch.rand(B, C, H, W, generator=g)),
                torch.stack([torch.randint(0, k, (B,), generator=g) for k in conf['contexts']], 1),
                torch.randint(0, conf['mixtures'], (B,), generator=g)) for _ in range(3)]
    with torch.no_grad():                                         # ActNorm's first-batch initialisation, shared by both arms
        base.log_prob(batches[0][0].to(dev), batches[0][1].to(dev))
    prior = {'size': list(base.dist.size), 'M': base.dist.M}
    arms = [Arm('eager', copy.deepcopy(base), dev), Arm('graphed', copy.deepcopy(base).enable_cuda_graphs(training=True), dev)]
    del base
    torch.manual_seed(1)
    for arm in arms:
        for i in range(a.warmup):                                 # the graphed arm's first call runs eagerly, the second captures
            arm.step(batches[i % 3], conf, alpha, criterion)
    losses = {}
    for _ in range(a.rounds):
        for arm in arms:
            torch.cuda.synchronize()
            for i in range(a.steps):
                t0 = time.perf_counter()
                losses[arm.name] = arm.step(batches[i % 3], conf, alpha, criterion)     # .item() synchronises
                arm.ms.append(1e3 * (time.perf_counter() - t0))
    res = {'workload': f'{name} with a Student-t mixture as dist', 'prior': prior, 'batch': B, 'steps_per_round': a.steps, 'rounds': a.rounds}
    for arm in arms:
        res[arm.name] = {'ms_per_step_median': round(statistics.median(arm.ms), 3), 'ms_per_step_min': round(min(arm.ms), 3),
                         'last_losses': losses[arm.name]}
    res['graphed']['training_graph_entries'] = len(arms[1].model._graphed_train._entries)
    res['speedup_median'] = round(res['eager']['ms_per_step_median'] / res['graphed']['ms_per_step_median'], 3)
    del arms
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='cfg1,cfg4'); ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--steps', type=int, default=10); ap.add_argument('--warmup', type=int, default=3); ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON result to this file')
    a = ap.parse_args()
    if a.warmup < 2:
        ap.error('--warmup must be at least 2: the graphed arm captures at its second call')
    if not torch.cuda.is_available():
        raise SystemExit('bench_student_train.py measures on a CUDA device; none is visible')
    dev = torch.device('cuda', 0)
    out = {'tool': 'tools/bench_student_train.py', 'card': card(), 'torch': torch.__version__, 'prior_alone': [], 'training_step': []}
    for name in a.configs.split(','):
        conf = synth.CONFIGS[name]
        size = builder.build_named(conf).dist.size
        r = prior_alone(size, conf['mixtures'], BATCH[name], a.iters, dev)
        out['prior_alone'].append(r)
        print(json.dumps(r), flush=True)
        r = training_step(name, BATCH[name], a, dev)
        out['training_step'].append(r)
        print(json.dumps(r), flush=True)
    print(json.dumps(out))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
