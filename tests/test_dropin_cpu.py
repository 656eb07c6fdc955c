"""Drop-in boundary on the CPU.  Without the reference: contextflow_b200.builder.create_model, which the GPU tests and bench use, yields
the state_dict table and layer sequence the unmodified reference recorded over its own layers (tests/golden).  With a reference checkout
($CFPP_REFERENCE or baseline/_ref, see tools/refshim.py; skipped otherwise): the reference's own, unmodified model.create_model /
ContextEncoder, executed over THIS package's `layers` namespace, must construct, and must yield exactly the module tree / state_dict of
(a) the reference over its own layers (the golden `keys` tables) and (b) contextflow_b200.builder.create_model."""
import argparse, json, os, subprocess, sys, textwrap
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import refshim  # noqa: E402

REF = refshim.find_reference()

SCRIPT = textwrap.dedent('''
    import sys, types, json, argparse
    sys.path.insert(0, %(root)r)
    sys.dont_write_bytecode = True
    from contextflow_b200.run import install_layers
    L = install_layers()
    REF = %(ref)r
    sys.path.insert(0, REF)
    pkg = types.ModuleType('datasets'); pkg.__path__ = [REF + '/datasets']; pkg.corrupt = None
    sys.modules['datasets'] = pkg
    class _Stub(types.ModuleType):
        __path__ = []
        def __getattr__(self, k):
            if k.startswith('__'): raise AttributeError(k)
            return lambda *a, **kw: None
    for n in ('matplotlib', 'matplotlib.pyplot', 'torchinfo', 'ood_metrics'): sys.modules[n] = _Stub(n)
    import model as M                      # the reference's model.py, unmodified
    assert M.Conv1x1 is L.Conv1x1 and M.FlowSequential is L.FlowSequential, 'model.py did not pick up the replacement layers'
    from contextflow_b200 import builder, synth
    from tests.golden.cases import CASES
    out = {}
    for name, case in CASES.items():
        conf = case['conf']
        M.c = argparse.Namespace(dataset=conf['cfg']['dataset'])
        net = M.create_model(conf['cfg'], data_size=conf['data_size'], mixtures=conf['mixtures'], contexts=conf['contexts'])
        mine = builder.build_named(conf)
        a = {k: list(v.shape) for k, v in net.state_dict().items()}
        b = {k: list(v.shape) for k, v in mine.state_dict().items()}
        ta = [type(m).__name__ for m in net.modules()]; tb = [type(m).__name__ for m in mine.modules()]
        ga = sorted(k for k, p in net.named_parameters() if p.requires_grad); gb = sorted(k for k, p in mine.named_parameters() if p.requires_grad)
        out[name] = dict(keys=a, same_keys=(a == b and list(a) == list(b)), same_tree=(ta == tb), same_trainable=(ga == gb), n_trainable=len(ga))
    print('RESULT' + json.dumps(out))
''')


def test_builder_matches_reference_tables():
    from contextflow_b200 import builder
    from tests.golden.cases import CASES
    from tests.helpers import load_golden
    for name, case in CASES.items():
        g = load_golden(name)
        model = builder.build_named(case['conf'])
        keys = {k: list(v.shape) for k, v in model.state_dict().items()}
        assert keys == g['keys'] and list(keys) == list(g['keys']), f'{name}: state_dict differs from the reference over its own layers'
        assert [type(m).__name__ for m in model.sequence_modules] == g['layer_types'], f'{name}: layer sequence differs'


@pytest.mark.skipif(REF is None, reason='no checkout of the unmodified reference (CFPP_REFERENCE)')
def test_reference_create_model_runs_over_replacement_layers():
    from tests.golden.cases import CASES
    from tests.helpers import load_golden
    r = subprocess.run([sys.executable, '-c', SCRIPT % dict(root=ROOT, ref=REF)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads(r.stdout.split('RESULT', 1)[1])
    for name in CASES:
        g = load_golden(name)
        assert res[name]['keys'] == g['keys'], f'{name}: state_dict differs from the reference over its own layers'
        assert res[name]['same_keys'], f'{name}: builder.create_model state_dict differs'
        assert res[name]['same_tree'], f'{name}: module tree differs'
        assert res[name]['same_trainable'], f'{name}: requires_grad pattern differs (freeze_parameters semantics)'
