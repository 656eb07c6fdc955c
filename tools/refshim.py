"""Locating and importing the UNMODIFIED reference (gudovskiy/contextflow) for baselines and boundary tests.  Measurement / test
infrastructure only: nothing under contextflow_b200/ imports this.

Search order: $CFPP_REFERENCE (the `contextflow` package directory of an upstream checkout), <repo>/baseline/_ref/contextflow (the
offline install made by tools/install_reference.py, git-ignored).  A directory counts only when it holds the whole package
(`model.py` AND `layers/`): the reference's setup.py lists `packages=['contextflow']` without sub-packages, so a bare pip install
lacks layers/, utils/ and datasets/ and cannot run.

`import_reference(ref, replacement=False)` applies the import shim of SURVEY App. B (datasets/__init__ skipped because it needs
skimage; matplotlib / torchinfo / ood_metrics stubbed) and returns the reference's `model` module.  With replacement=True this
repo's layers are registered as `layers` first (contextflow_b200.run.install_layers), i.e. exactly what
`python -m contextflow_b200.run model.py` does, so model.py / experiment_*.py execute over the CUDA path."""
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CANDIDATES = [os.environ.get('CFPP_REFERENCE'), os.path.join(ROOT, 'baseline', '_ref', 'contextflow')]


def find_reference():
    for c in CANDIDATES:
        if c and os.path.isfile(os.path.join(c, 'model.py')) and os.path.isdir(os.path.join(c, 'layers')):
            return c
    return None


class _Stub(types.ModuleType):
    __path__ = []

    def __getattr__(self, k):
        if k.startswith('__'):
            raise AttributeError(k)
        return lambda *a, **kw: None


def import_reference(ref=None, replacement=False):
    ref = ref or find_reference()
    if ref is None:
        raise FileNotFoundError('no complete reference checkout (model.py + layers/) under ' + ', '.join(c for c in CANDIDATES if c))
    sys.dont_write_bytecode = True
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    if replacement:
        from contextflow_b200.run import install_layers
        install_layers()
    sys.path.insert(0, ref)
    pkg = types.ModuleType('datasets'); pkg.__path__ = [os.path.join(ref, 'datasets')]; pkg.corrupt = None
    sys.modules['datasets'] = pkg
    for n in ('matplotlib', 'matplotlib.pyplot', 'torchinfo', 'ood_metrics', 'wandb'):
        if n not in sys.modules:
            try:
                __import__(n)
            except Exception:
                sys.modules[n] = _Stub(n)
    import model as M                                   # the reference's model.py, unmodified
    return M


def create_model(M, conf):
    """The reference's create_model for one of synth.CONFIGS-style dicts (global `c.dataset` is read at model.py:113,125)."""
    import argparse
    M.c = argparse.Namespace(dataset=conf['cfg']['dataset'])
    return M.create_model(conf['cfg'], data_size=conf['data_size'], mixtures=conf['mixtures'], contexts=conf['contexts'])
