"""Single-process N-GPU log_prob (contextflow_b200/multigpu.py): needs at least two visible GPUs; skipped otherwise."""
import pytest
import torch

from contextflow_b200 import builder, synth

pytestmark = pytest.mark.gpu


def _model(name, **over):
    conf = synth.variant(name, **over)
    model = builder.build_named(conf)
    sd = model.state_dict(); synth.fill_state(sd, 'mg'); model.load_state_dict(sd)
    return conf, model.to('cuda:0').eval()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
# even channel counts: no Augment noise, so the time-series stacks are deterministic (cfg1 draws dequantisation noise)
@pytest.mark.parametrize('name,B,over', [('cfg1', 1500, {}), ('cfg4', 4100, dict(data_size=(24, 8, 1))),
                                         ('cfg4', 1030, dict(data_size=(24, 8, 1), coupling='conv', num_blocks=1, block_size=2))])
def test_replicated_log_prob_equals_single_device(name, B, over):
    """Deterministic stacks (no dequantisation noise on the time-series path; MNIST noise is per device, so cfg1 is compared through
    its noise-free statistics): rows come back in batch order and equal the one-device result."""
    conf, model = _model(name, **over)
    x, ctx = synth.make_inputs(conf, B, 'mg')
    x, ctx = x.to('cuda:0'), ctx.to('cuda:0')
    with torch.no_grad():
        ref = model.log_prob(x, ctx)
        model.enable_multi_gpu(min_rows=256)
        got = model.log_prob(x, ctx)
        torch.cuda.synchronize()
    assert got.shape == ref.shape and got.device == ref.device
    if conf['image']:
        # the dequantisation noise is redrawn per call (and per device): rows move by tens of nats on a log-prob of thousands, the batch
        # statistics do not (row order is pinned by the deterministic time-series stacks)
        assert (got - ref).abs().max().item() < 5e-2 * ref.abs().max().item()
        assert abs(got.mean().item() - ref.mean().item()) < 2e-3 * abs(ref.mean().item())
    else:
        assert torch.allclose(got, ref, rtol=1e-5, atol=1e-4), (got - ref).abs().max().item()
    n_used = min(torch.cuda.device_count(), B // 256)
    assert len(model.__dict__['_replicated']._replicas) == n_used - 1


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_replicas_follow_weight_updates():
    conf, model = _model('cfg4', data_size=(24, 8, 1))
    x, ctx = synth.make_inputs(conf, 2048, 'mg2')
    x, ctx = x.to('cuda:0'), ctx.to('cuda:0')
    model.enable_multi_gpu(min_rows=256)
    with torch.no_grad():
        a = model.log_prob(x, ctx)
        for p in model.parameters():
            if p.dim() == 1:
                p.add_(0.01)
        b = model.log_prob(x, ctx)
        model.enable_multi_gpu(False)
        ref = model.log_prob(x, ctx)
    assert not torch.allclose(a, b)
    assert torch.allclose(b, ref, rtol=1e-5, atol=1e-4)
