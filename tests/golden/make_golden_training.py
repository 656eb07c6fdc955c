"""Generate tests/golden/train_*.npz by executing the UNMODIFIED reference on CPU with torch autograd.

    CFPP_REFERENCE=<upstream checkout>/contextflow python tests/golden/make_golden_training.py
Training direction (SURVEY §8f-1).  For each case the reference model (hash-derived weights, inputs and noise, as in make_golden.py)
evaluates the training loss exactly as experiment_ad.py:204-209 writes it and calls .backward(); stored: the loss terms and the
gradient of every trainable parameter (full tensor up to 2048 elements, else (sum, sum|.|) and the first 512 values), plus the
parameters after ONE torch.optim.AdamW step with the settings of model.py:289 (lr 1e-3 here).
"""
import sys, os, argparse, json
import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from contextflow_b200 import synth  # noqa: E402
from tests.golden.cases import CASES, TRAINING_CASES  # noqa: E402
from tests.golden.make_golden import import_reference, patched_rng  # noqa: E402

FULL = 2048


def training_loss(net, x, ctx, gt, data_size, spec):
    """experiment_ad.py:204-209 (log_theta = nn.LogSigmoid(), :15; dim_inv :60)."""
    dim_inv = 1.0 / torch.prod(torch.tensor(data_size))
    log_theta = nn.LogSigmoid()
    criterion = nn.CrossEntropyLoss(weight=None if spec['weight'] is None else torch.tensor(spec['weight'])) if spec['criterion'] else None
    alpha = spec['alpha']
    logp = dim_inv * net.log_prob(x, context=ctx)
    logp[logp != logp] = 0.0
    cost_uns = -alpha * log_theta(torch.logsumexp(logp, -1)).mean() if criterion else -alpha * log_theta(logp).mean()
    cost_sup = criterion(logp, gt) if criterion else torch.zeros_like(cost_uns)
    return cost_sup + cost_uns, cost_sup, cost_uns


def labels(name, B, M):
    return (synth.NoiseTape(f'traingt:{name}').rand((B,)) * M).long().clamp(max=M - 1)


def run(M_, name, spec):
    case = CASES[name]
    conf = case['conf']
    M_.c = argparse.Namespace(dataset=conf['cfg']['dataset'])
    torch.manual_seed(0)
    net = M_.create_model(conf['cfg'], data_size=conf['data_size'], mixtures=conf['mixtures'], contexts=conf['contexts'])
    sd = net.state_dict(); synth.fill_state(sd, case.get('wseed', 'w0')); net.load_state_dict(sd)
    net.train()
    x, ctx = synth.make_inputs(conf, case['B'], case.get('iseed', 'in0'))
    gt = labels(name, case['B'], conf['mixtures'])
    opt = torch.optim.AdamW(filter(lambda p: p.requires_grad, net.parameters()), lr=1e-3)
    with patched_rng(synth.NoiseTape(case.get('nseed', 'noise0'))):
        cost, sup, uns = training_loss(net, x, ctx, gt, conf['data_size'], spec)
    cost.backward()
    rec = dict(loss=np.array([cost.item(), sup.item(), uns.item()]))
    names = []
    for k, p in net.named_parameters():
        if not p.requires_grad or p.grad is None:        # e.g. the embed table in front of probsample: unused by the reference's forward
            continue
        g = p.grad.detach()
        names.append(k)
        gd = g.double()
        rec[f'gsum:{k}'] = np.array([gd.sum().item(), gd.abs().sum().item(), gd.abs().max().item()])
        rec[f'g:{k}'] = g.numpy() if g.numel() <= FULL else g.flatten()[:512].numpy()
    opt.step()
    for k, p in net.named_parameters():
        if p.requires_grad and p.grad is not None:
            pd = p.detach().double()
            rec[f'psum:{k}'] = np.array([pd.sum().item(), pd.abs().sum().item()])
    # the same reference model and loss in float64: the yardstick for how far float32 summation order moves each gradient
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(0)
        net64 = M_.create_model(conf['cfg'], data_size=conf['data_size'], mixtures=conf['mixtures'], contexts=conf['contexts'])
        sd = net64.state_dict(); synth.fill_state(sd, case.get('wseed', 'w0')); net64.load_state_dict(sd)
        net64 = net64.double().train()

        class Tape64:
            def __init__(self, t): self.t = t
            def rand(self, shape, dtype=None, **kw): return self.t.rand(shape).double()
            def randn(self, shape, dtype=None, **kw): return self.t.randn(shape).double()
        with patched_rng(Tape64(synth.NoiseTape(case.get('nseed', 'noise0')))):
            cost64, _, _ = training_loss(net64, x.double(), ctx, gt, conf['data_size'], spec)
        cost64.backward()
        for k, p in net64.named_parameters():
            if p.requires_grad and p.grad is not None:
                g = p.grad.detach()
                rec[f'g64:{k}'] = g.numpy() if g.numel() <= FULL else g.flatten()[:512].numpy()
        rec['loss64'] = np.array(cost64.item())
    finally:
        torch.set_default_dtype(torch.float32)
    rec['names'] = np.array(json.dumps(names))
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', f'train_{name}.npz'), **rec)
    print(f'train_{name}: loss={cost.item():.6f} (sup {sup.item():.6f}, uns {uns.item():.6f}) params={len(names)}')


if __name__ == '__main__':
    M_ = import_reference()
    only = set(sys.argv[1:])                       # optional: case names to (re)generate
    for n, spec in TRAINING_CASES.items():
        if not only or n in only:
            run(M_, n, spec)
