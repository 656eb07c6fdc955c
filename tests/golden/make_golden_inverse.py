"""Generate tests/golden/inv_*.npz and score_*.npz by executing the UNMODIFIED reference on CPU.

    CFPP_REFERENCE=<upstream checkout>/contextflow python tests/golden/make_golden_inverse.py
Inverse direction (SURVEY §8f-3).  Two kinds of fixture:
  * full chain (models whose every layer has an executable .reverse in the reference: generalists without split priors):
    the latent z of the forward golden is pushed through `module.reverse` from the last layer to the first, exactly the loop
    of FlowSequential.sample (flowsequential.py:34-37).  Stored: the result, the value entering Dequantization.reverse (before
    the floor), per-layer (sum, sum|.|) checksums.
  * per-layer Coupling / TransCoupling reverse with a context encoder (specialists): each coupling module's .reverse on a
    hash-derived input of its own output shape, encoder noise served from a NoiseTape.
Score epilogue (SURVEY §8f-2): the torch expressions of experiment_ad.py:204-211,270-278 / experiment_cl.py:127-133,193-200
evaluated on hash-derived log-probs (nn.LogSigmoid, nn.CrossEntropyLoss(weight), torch.logsumexp/softmax/argmax).
"""
import sys, os, argparse, json
import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from contextflow_b200 import synth  # noqa: E402
from tests.golden.cases import CASES, INVERSE_CHAIN, INVERSE_COUPLING, SCORE_CASES  # noqa: E402
from tests.golden.make_golden import import_reference, patched_rng  # noqa: E402


def build(M, case):
    conf = case['conf']
    M.c = argparse.Namespace(dataset=conf['cfg']['dataset'])
    torch.manual_seed(0)
    net = M.create_model(conf['cfg'], data_size=conf['data_size'], mixtures=conf['mixtures'], contexts=conf['contexts'])
    net.eval()
    sd = net.state_dict(); synth.fill_state(sd, case.get('wseed', 'w0')); net.load_state_dict(sd)
    return net


def chk(t):
    d = t.detach().double()
    return np.array([d.sum().item(), d.abs().sum().item()])


def run_chain(M, name):
    case = CASES[name]
    net = build(M, case)
    _, ctx = synth.make_inputs(case['conf'], case['B'], case.get('iseed', 'in0'))
    z = torch.from_numpy(np.load(os.path.join(ROOT, 'tests', 'golden', f'{name}.npz'))['z'])
    rec = {}
    out = z
    mods = list(net.sequence_modules)
    with torch.no_grad():
        for i in reversed(range(len(mods))):
            if type(mods[i]).__name__ == 'Dequantization':
                rec['x_prefloor'] = out.numpy().copy()
            out = mods[i].reverse(out, ctx)
            rec[f'rsum_{i}'] = chk(out)
    rec['x_rec'] = out.numpy()
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', f'inv_{name}.npz'), **rec)
    print(f'inv_{name}: layers={len(mods)} x_rec{tuple(out.shape)} [0,:4]={out.flatten()[:4].tolist()}')


def run_coupling(M, name):
    case = CASES[name]
    net = build(M, case)
    x, ctx = synth.make_inputs(case['conf'], case['B'], case.get('iseed', 'in0'))
    shapes = {}
    hooks = [m.register_forward_hook(lambda mod, inp, out, i=i: shapes.__setitem__(i, tuple(out[0].shape)))
             for i, m in enumerate(net.sequence_modules)]
    with torch.no_grad(), patched_rng(synth.NoiseTape('noise0')):
        net(x, ctx)
    for h in hooks:
        h.remove()
    rec, idx = {}, []
    for i, m in enumerate(net.sequence_modules):
        if type(m).__name__ not in ('Coupling', 'TransCoupling'):
            continue
        zin = synth.NoiseTape(f'invin{i}').randn(shapes[i])
        tape = synth.NoiseTape(f'invnoise{i}')
        with torch.no_grad(), patched_rng(tape):
            xr = m.reverse(zin, ctx)
        rec[f'rsum_{i}'] = chk(xr)
        if len(idx) < 2:
            rec[f'x_{i}'] = xr.numpy()
        idx.append(i)
    rec['layers'] = np.array(idx)
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', f'inv_{name}.npz'), **rec)
    print(f'inv_{name}: coupling layers {idx}')


def run_score(name, spec):
    B, Mx = spec['B'], spec['M']
    logp = synth.NoiseTape(f'score:{name}').randn((B, Mx)) * spec['spread'] + spec['shift']
    if spec.get('nan'):
        logp[1, 0] = float('nan'); logp[B - 1, Mx - 1] = float('nan')
    gt = (synth.NoiseTape(f'scoregt:{name}').rand((B,)) * Mx).long().clamp(max=Mx - 1)
    dim_inv = 1.0 / torch.prod(torch.tensor(spec['size']))                 # experiment_ad.py:60 / experiment_cl.py:55
    log_theta = nn.LogSigmoid()                                             # experiment_ad.py:15
    w = torch.tensor(spec['weight'], dtype=torch.float32) if spec.get('weight') else None
    criterion = nn.CrossEntropyLoss(weight=w)                               # model.py:294
    s = dim_inv * logp
    s[s != s] = 0.0                                                         # experiment_ad.py:205
    rec = dict(logp=logp.numpy(), gt=gt.numpy(), dim_inv=np.array(float(dim_inv), dtype=np.float32),
               scaled=s.numpy(), lse=torch.logsumexp(s, -1).numpy(),
               uns_crit=log_theta(torch.logsumexp(s, -1)).mean().numpy(),   # :207 with a criterion (without alpha)
               uns_none=log_theta(s).mean().numpy(),                        # :207 without
               sup=criterion(s, gt).numpy(),                                # :208
               argmax=torch.argmax(s, dim=-1).numpy(),                      # experiment_cl.py:200
               last=s[:, -1].numpy())                                       # experiment_ad.py:278 (theta = Identity)
    if Mx > 1:
        rec['softmax1'] = torch.softmax(s, dim=-1)[:, 1].numpy()            # experiment_ad.py:278
    if w is not None:
        rec['weight'] = w.numpy()
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', f'score_{name}.npz'), **rec)
    print(f'score_{name}: B={B} M={Mx} sup={float(rec["sup"]):.6f} uns={float(rec["uns_crit"]):.6f}')


if __name__ == '__main__':
    M = import_reference()
    for n in INVERSE_CHAIN:
        run_chain(M, n)
    for n in INVERSE_COUPLING:
        run_coupling(M, n)
    for n, spec in SCORE_CASES.items():
        run_score(n, spec)
