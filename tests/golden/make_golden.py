"""Generate tests/golden/*.npz by executing the UNMODIFIED reference on CPU.

    CFPP_REFERENCE=<upstream checkout>/contextflow python tests/golden/make_golden.py
The reference is imported through the shim of SURVEY App. B (no reference file is edited or copied).
Weights are overwritten with contextflow_b200.synth.fill_state (hash-derived, portable), inputs come
from synth.make_inputs, and the reference's own torch.rand/torch.randn calls are served from a
synth.NoiseTape for the duration of the forward, so the fixtures depend on no RNG implementation.
Stored per case: final z, logp (B,M), per-layer ldj, per-layer (sum z, sum |z|), the noise-draw log.
"""
import sys, os, types, argparse, json
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from contextflow_b200 import synth  # noqa: E402
from tests.golden.cases import CASES  # noqa: E402

REF = os.environ.get('CFPP_REFERENCE', '')


def import_reference():
    if not os.path.isfile(os.path.join(REF, 'model.py')):
        sys.exit('set CFPP_REFERENCE to the upstream contextflow package directory')
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    pkg = types.ModuleType('datasets'); pkg.__path__ = [REF + '/datasets']; pkg.corrupt = None
    sys.modules['datasets'] = pkg

    class _Stub(types.ModuleType):
        __path__ = []
        def __getattr__(self, k):
            if k.startswith('__'):
                raise AttributeError(k)
            return lambda *a, **kw: None
    for n in ('matplotlib', 'matplotlib.pyplot', 'torchinfo', 'ood_metrics'):
        sys.modules[n] = _Stub(n)
    import model as M
    return M


class patched_rng:
    """Serve torch.rand / torch.randn from a NoiseTape while the reference runs."""
    def __init__(self, tape):
        self.tape = tape
    def __enter__(self):
        self._rand, self._randn = torch.rand, torch.randn
        def shape_of(a):
            return tuple(a[0]) if len(a) == 1 and isinstance(a[0], (tuple, list, torch.Size)) else tuple(a)
        torch.rand = lambda *a, **kw: self.tape.rand(shape_of(a), dtype=kw.get('dtype') or torch.float32)
        torch.randn = lambda *a, **kw: self.tape.randn(shape_of(a), dtype=kw.get('dtype') or torch.float32)
    def __exit__(self, *e):
        torch.rand, torch.randn = self._rand, self._randn


def run_case(M, name, case):
    conf = case['conf']
    M.c = argparse.Namespace(dataset=conf['cfg']['dataset'])
    torch.manual_seed(0)
    net = M.create_model(conf['cfg'], data_size=conf['data_size'], mixtures=conf['mixtures'], contexts=conf['contexts'])
    net.eval()
    sd = net.state_dict()
    synth.fill_state(sd, case.get('wseed', 'w0'))
    if case.get('fresh_actnorm'):
        for k in sd:
            if k.endswith('.initialized'):
                sd[k].fill_(0)
    net.load_state_dict(sd)
    x, ctx = synth.make_inputs(conf, case['B'], case.get('iseed', 'in0'))
    rec = {}
    hooks = []
    for i, m in enumerate(net.sequence_modules):
        def hook(mod, inp, out, i=i):
            z, ldj = out
            rec[f'ldj_{i}'] = ldj.detach().numpy().astype(np.float32)
            zd = z.detach().double()
            rec[f'zsum_{i}'] = np.array([zd.sum().item(), zd.abs().sum().item()])
        hooks.append(m.register_forward_hook(hook))
    tape = synth.NoiseTape(case.get('nseed', 'noise0'))
    with torch.no_grad(), patched_rng(tape):
        z, logp = net(x, ctx)
    for h in hooks:
        h.remove()
    rec['z'] = z.numpy(); rec['logp'] = logp.numpy()
    rec['draws'] = np.array(json.dumps(tape.log))
    rec['n_layers'] = np.array(len(net.sequence_modules))
    rec['layer_types'] = np.array(json.dumps([type(m).__name__ for m in net.sequence_modules]))
    if case.get('fresh_actnorm'):
        post = net.state_dict()
        for k in post:
            if k.endswith('NN_t') or k.endswith('NN_logs'):
                rec['post:' + k] = post[k].numpy()
    rec['keys'] = np.array(json.dumps({k: list(v.shape) for k, v in net.state_dict().items()}))
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', f'{name}.npz'), **rec)
    print(f'{name}: layers={len(net.sequence_modules)} draws={len(tape.log)} logp[0]={logp[0, :3].tolist()}')


if __name__ == '__main__':
    M = import_reference()
    only = sys.argv[1:]
    for name, case in CASES.items():
        if only and name not in only:
            continue
        run_case(M, name, case)
