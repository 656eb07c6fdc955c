"""CPU tests of the host-side logic that needs no kernel launch: the fused log_prob plan's segmentation of the BASELINE stacks, the
reference arm of bench.py, and the C-ABI descriptors the Python layer builds."""
import json
import os
import subprocess
import sys

import pytest
import torch

from contextflow_b200 import builder, synth
from contextflow_b200.layers._fastpath import FastLogProb, _ConvAct, _Coup, _Generic, _Prologue

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _segments(name):
    model = builder.build_named(synth.CONFIGS[name])
    return model, FastLogProb(model).segs


def test_fused_plan_segments_cfg2():
    model, segs = _segments('cfg2')
    kinds = [type(s).__name__ for s in segs]
    assert kinds[0] == '_Prologue' and len(segs[0].mods) == 5                      # Dequant, Norm, Norm, Logit, Augment (model.py:97-100,121-123)
    assert kinds.count('_ConvAct') == 12 and kinds.count('_Coup') == 12            # 3 levels x 4 steps (SURVEY §8 stack table)
    assert sum(len(s.mods) for s in segs) == len(model.sequence_modules)            # every layer belongs to exactly one segment, in order
    flat = [m for s in segs for m in s.mods]
    assert all(a is b for a, b in zip(flat, model.sequence_modules))
    # context pre-pass: one CN job per contextual Conv1x1 / ActNorm / Coupling, the Conv1x1 ones flagged lower-triangular
    # (the Conv1x1 ones are absent when the persistent Conv1x1 + context-network kernel has a plan for the level: its CN runs in-kernel)
    jobs = [j for s in segs if isinstance(s, (_ConvAct, _Coup)) for j in s.cn_jobs()]
    assert len(jobs) == 24
    assert sorted({tril for _, _, tril, _, _ in jobs}) == [0]


def test_fused_plan_segments_cfg2_two_kernel_conv1x1(monkeypatch):
    monkeypatch.setenv('CFPP_C1X1_CTX', '0')                                        # the two-kernel route: CN pre-pass + per-sample-matrix kernel
    _, segs = _segments('cfg2')
    jobs = [j for s in segs if isinstance(s, (_ConvAct, _Coup)) for j in s.cn_jobs()]
    assert len(jobs) == 36
    assert sorted({tril for _, _, tril, _, _ in jobs}) == [0, 16, 32, 64]


@pytest.mark.parametrize('name,n_conv,n_coup,prologue', [('cfg1', 4, 4, True), ('cfg3', 12, 12, False), ('cfg4', 8, 8, False)])
def test_fused_plan_segments_other_stacks(name, n_conv, n_coup, prologue):
    model, segs = _segments(name)
    kinds = [type(s).__name__ for s in segs]
    assert (kinds[0] == '_Prologue') == prologue
    assert kinds.count('_ConvAct') == n_conv and kinds.count('_Coup') == n_coup
    assert sum(len(s.mods) for s in segs) == len(model.sequence_modules)


def test_fused_plan_is_not_used_on_cpu_tensors():
    model, _ = _segments('cfg1')
    x, ctx = synth.make_inputs(synth.CONFIGS['cfg1'], 2, 'h0')
    with torch.no_grad():
        assert not FastLogProb(model).usable(x, ctx)                                 # CPU tensors: the plan (and every kernel) is CUDA only
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        with torch.no_grad():
            model.log_prob(x, ctx)


def test_dump_outputs_samples_the_same_rows_within_budget(tmp_path, monkeypatch):
    import numpy as np
    import bench
    monkeypatch.setattr(bench, 'DUMP_BYTES', 4000)
    big, small = torch.arange(3000.0).reshape(1500, 2), torch.ones(10, 1)          # 12040 bytes together
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'big': big, 'small': small})
    a, b = np.load(tmp_path / 'a' / 'big.npy'), np.load(tmp_path / 'b' / 'big.npy')
    s = np.load(tmp_path / 'a' / 'small.npy')
    assert a.dtype == s.dtype == np.float32 and np.array_equal(a, b)
    assert a.nbytes + s.nbytes <= 4000 and a.shape[1] == 2 and s.shape == (3, 1)
    assert np.all(np.diff(a[:, 0]) > 0) and np.all(a[:, 1] == a[:, 0] + 1)        # whole rows, in batch order
    bench.dump_outputs(str(tmp_path / 'c'), {'small': small})                        # under the budget: every row
    assert np.array_equal(np.load(tmp_path / 'c' / 'small.npy'), small.numpy())


@pytest.mark.parametrize('force_port', ['1', '0'])
def test_reference_arm_prints_one_json_line(force_port):
    """--impl reference: the unmodified reference when a complete checkout exists ($CFPP_REFERENCE or baseline/_ref), else the port."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'cfg4', '--batch', '64',
                          '--steps', '1', '--warmup', '1'], capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, CFPP_BENCH_FORCE_PORT=force_port))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'flow_log_prob_samples_per_sec' and d['value'] > 0
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import refshim
    want = 'port' if force_port == '1' or refshim.find_reference() is None else 'reference'
    assert d['cpu_baseline']['kind'] == want and d['cpu_baseline']['cores'] >= 1
    assert d['config']['batch_per_gpu'] == 131072                   # the reference arm reports this repo's arm's config; the bounded sample is described apart
    assert '64-sample' in d['cpu_baseline']['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
