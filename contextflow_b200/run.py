"""Launcher: run the reference's UNMODIFIED model.py over this package's layers.

    cd <reference>/contextflow && python -m contextflow_b200.run [--multi-gpu] model.py --gpu 0 --dataset smap --action-type test ...

model.py does `from layers import *` and `from layers.rtdl.nn._embeddings import *` (model.py:14-15) and is started from
the reference directory, whose own `layers/` package would win on sys.path.  The replacement is therefore registered in
sys.modules under those names BEFORE model.py executes; datasets/, utils/, config.py, experiment_*.py keep coming from
the reference.

The launcher also installs the fused AdamW (contextflow_b200/optim.py) and turns on CUDA graphs for model.log_prob: scoring calls and
the training loop's calls (CFPP_CUDA_GRAPHS=1, CFPP_CUDA_GRAPHS_TRAIN=1 unless already set), so the unchanged loop runs a training step
as two graph launches plus its own loss and optimizer step.
"""
import os
import runpy
import sys


def install_layers():
    """Register contextflow_b200.layers as the top-level `layers` package (and its rtdl sub-namespace)."""
    import contextflow_b200.layers as L
    import contextflow_b200.layers.rtdl as R
    import contextflow_b200.layers.rtdl.nn as RN
    import contextflow_b200.layers.rtdl.nn._embeddings as RE
    sys.modules['layers'] = L
    sys.modules['layers.rtdl'] = R
    sys.modules['layers.rtdl.nn'] = RN
    sys.modules['layers.rtdl.nn._embeddings'] = RE
    for name, mod in list(sys.modules.items()):
        if name.startswith('contextflow_b200.layers.'):
            sys.modules.setdefault('layers.' + name[len('contextflow_b200.layers.'):], mod)
    return L


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if argv and argv[0] == '--multi-gpu':                     # score large inference batches on every visible GPU from this one process
        os.environ['CFPP_MULTI_GPU'] = '1'                    # (contextflow_b200/multigpu.py; model.py itself stays unchanged)
        argv = argv[1:]
    if not argv:
        raise SystemExit(__doc__)
    script = os.path.abspath(argv[0])
    # inference calls of model.log_prob (eval_epoch, experiment_ad.py:262 / experiment_cl.py:185) replay a captured CUDA graph per input
    # shape; training calls (autograd on, train_epoch) replay a forward and a backward graph per input shape while the loop keeps its own
    # loss, backward() and optimizer step.  CFPP_CUDA_GRAPHS=0 keeps scoring eager, CFPP_CUDA_GRAPHS_TRAIN=0 keeps training eager.
    os.environ.setdefault('CFPP_CUDA_GRAPHS', '1')
    os.environ.setdefault('CFPP_CUDA_GRAPHS_TRAIN', '1')
    install_layers()
    if os.environ.get('CFPP_FUSED_ADAMW', '1') != '0':          # model.py:289 `optim.AdamW(...)` then builds the one-kernel optimizer
        from contextflow_b200 import optim as _optim
        _optim.install()
    sys.argv = [script] + argv[1:]
    sys.path.insert(0, os.path.dirname(script))
    os.chdir(os.path.dirname(script))
    runpy.run_path(script, run_name='__main__')


if __name__ == '__main__':
    main()
