"""CPU test of the launcher's environment: `python -m contextflow_b200.run model.py` turns on CUDA graphs for scoring and training calls
of log_prob unless the caller chose otherwise."""
import json
import sys

import pytest

from contextflow_b200 import run

KEYS = ('CFPP_CUDA_GRAPHS', 'CFPP_CUDA_GRAPHS_TRAIN')


def _launch(tmp_path, monkeypatch):
    script = tmp_path / 'train.py'
    script.write_text('import json, os\n'
                      f'json.dump({{k: os.environ.get(k) for k in {KEYS!r}}}, open("env.json", "w"))\n')
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(sys, 'argv', list(sys.argv))
    monkeypatch.setattr(sys, 'path', list(sys.path))
    monkeypatch.setenv('CFPP_FUSED_ADAMW', '0')                   # keep torch.optim.AdamW as it is for the rest of the session
    run.main([str(script)])
    return json.loads((tmp_path / 'env.json').read_text())


def test_launcher_turns_training_graphs_on(tmp_path, monkeypatch):
    for k in KEYS:
        monkeypatch.delenv(k, raising=False)
    assert _launch(tmp_path, monkeypatch) == {'CFPP_CUDA_GRAPHS': '1', 'CFPP_CUDA_GRAPHS_TRAIN': '1'}


@pytest.mark.parametrize('preset', ['0', '1'])
def test_launcher_keeps_a_preset_choice(tmp_path, monkeypatch, preset):
    monkeypatch.delenv('CFPP_CUDA_GRAPHS', raising=False)
    monkeypatch.setenv('CFPP_CUDA_GRAPHS_TRAIN', preset)
    assert _launch(tmp_path, monkeypatch) == {'CFPP_CUDA_GRAPHS': '1', 'CFPP_CUDA_GRAPHS_TRAIN': preset}
