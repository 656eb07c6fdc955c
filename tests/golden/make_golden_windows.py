"""Generate tests/golden/windows.npz with the UNMODIFIED reference's get_windows (datasets/mtad_data_preprocess.py:58-74) followed by the
transpose / float32 cast of sliding_window_dataset (datasets/mtad_dataloader.py:106-110), on hash-derived float64 series.
    CFPP_REFERENCE=<upstream checkout>/contextflow python tests/golden/make_golden_windows.py"""
import sys, types, os
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from contextflow_b200 import synth  # noqa: E402
REF = os.environ.get('CFPP_REFERENCE', '')
SPECS = {'smap': (41, 25, 8, 1), 'msl': (30, 55, 8, 3), 'tiny': (5, 3, 8, 1)}      # rows, D, window, stride

if __name__ == '__main__':
    if not os.path.isdir(os.path.join(REF, 'datasets')):
        sys.exit('set CFPP_REFERENCE to the upstream contextflow package directory')
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    pkg = types.ModuleType('datasets'); pkg.__path__ = [REF + '/datasets']; sys.modules['datasets'] = pkg
    from datasets.mtad_data_preprocess import get_windows
    rec = {}
    for name, (rows, D, L, stride) in SPECS.items():
        ts = synth.uniform(f'win:{name}', (rows, D), 0.0, 1.0, torch.float64).numpy()
        w, _ = get_windows(ts, window_size=L, stride=stride)
        X = np.transpose(np.array(w), axes=(0, 2, 1))                      # mtad_dataloader.py:106
        rec[f'{name}:x'] = torch.tensor(X, dtype=torch.float).unsqueeze(-1).numpy()   # :110
        rec[f'{name}:spec'] = np.array([rows, D, L, stride])
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', 'windows.npz'), **rec)
