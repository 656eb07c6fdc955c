"""The drop-in boundary end to end on the GPU (SURVEY §8b; VERDICT r1 next-7): the reference's UNMODIFIED experiment loops
(experiment_ad.py:184-291, experiment_cl.py:107-215: eval_epoch, train_epoch with the AdamW model.py:289 builds, save / load of a
generalist checkpoint into a specialist with strict=False) run over this repo's layers and over the reference's own torch layers on
the same GPU; every reported number must agree.  Needs a complete reference checkout ($CFPP_REFERENCE, or baseline/_ref made by
tools/install_reference.py): skipped otherwise."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import refshim  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(refshim.find_reference() is None, reason='no complete reference checkout ($CFPP_REFERENCE or baseline/_ref)')]


def _arm(arm, kind, tmp_path):
    out = str(tmp_path / f'{arm}_{kind}.json')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'boundary_arm.py'), arm, kind, out], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, f'{arm}/{kind} failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}'
    return json.load(open(out))


def _close(a, b, rtol, what):
    assert abs(a - b) <= rtol * max(abs(a), abs(b)) + 1e-6, f'{what}: {a} (this repo) vs {b} (reference)'


@pytest.mark.parametrize('kind', ['ad', 'cl'])
def test_unmodified_experiment_loops_match_reference(kind, tmp_path):
    mine = _arm('replacement', kind, tmp_path)
    ref = _arm('reference', kind, tmp_path)
    assert mine['launches'] > 0 and mine['graphs'] >= 2           # inference went through graph replays (two eval batch shapes)
    assert mine['spec_trainable'] == ref['spec_trainable']          # freeze_parameters pattern after the strict=False load
    for key in ('gen_eval0', 'spec_eval0'):                        # same weights, same noise: inference parity through eval_epoch
        _close(mine[key]['loss'], ref[key]['loss'], 1e-4, f'{kind} {key} loss')
        n = len(ref[key]['scores'])
        bad = [i for i in range(n) if abs(mine[key]['scores'][i] - ref[key]['scores'][i]) > 1e-4 * abs(ref[key]['scores'][i]) + 1e-4]
        assert not bad, f'{kind} {key}: {len(bad)} of {n} scores differ, first {bad[:3]}'
        if kind == 'cl':
            _close(mine[key]['log_px'], ref[key]['log_px'], 1e-4, f'{kind} {key} log_px')
    for key in ('gen_train', 'spec_train'):                        # three AdamW steps through the backward kernels
        _close(mine[key], ref[key], 1e-3, f'{kind} {key} mean loss')
    for key in ('gen_eval1', 'spec_eval1'):                        # after training: the updated weights were picked up (graphs re-captured)
        _close(mine[key]['loss'], ref[key]['loss'], 2e-3, f'{kind} {key} loss')
    _close(mine['param_abs_sum'], ref['param_abs_sum'], 1e-4, f'{kind} parameters after training')
