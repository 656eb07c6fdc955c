"""Parity after the weights have moved.  Every other parity test scores a model that was just built; here the CUDA model takes optimizer
steps first (torch.optim.AdamW, the fused AdamW of contextflow_b200/optim.py eagerly or captured by GraphedTrainStep) and is then compared
with the oracle at the weights it holds at that moment.  Many values derived from the weights (log|det NN| and NN^-1 of Conv1x1, the
mixture tables, the masked MAF weights, the packs of the fused plan, the signature of a captured log_prob graph, the weights of the
multi-GPU replicas) are cached on the tensors' version counters, so an update that does not bump them leaves stale values behind."""
import copy

import numpy as np
import pytest
import torch

from contextflow_b200 import rng, synth
from contextflow_b200.graphed import GraphedTrainStep
from contextflow_b200.optim import FusedAdamW, _TorchAdamW
from oracle import flow_oracle as O
from tests.golden.cases import CASES, TRAINING_CASES
from tests.helpers import L_ATOL, L_RTOL, Z_ATOL, Z_RTOL, assert_close, case_inputs, golden_state, load_golden
from tests.test_gpu_multigpu import _model as multigpu_model
from tests.test_gpu_parity import FUSED_EXPECTED
from tests.test_gpu_training import REF_FACTOR, build_cuda_model, device_loss, labels, reference_loss
from tests.test_oracle_golden_training import load_train

pytestmark = pytest.mark.gpu

LR = 1e-2          # Adam moves every entry by ~lr per step whatever the gradient scale: a stale derived value misses the gates by far
STEPS = 3
OPTIMIZERS = {'torch_adamw': _TorchAdamW, 'fused_adamw': FusedAdamW}


def oracle_state(name, case, model):
    """The oracle's state at the weights the CUDA model holds now (the fp64 truth never follows Adam's own trajectory)."""
    stack, state = golden_state(load_golden(name), case)
    sd = model.state_dict()
    assert set(sd) == set(state)
    for k in state:
        state[k] = sd[k].detach().cpu().clone()
    return stack, state


def oracle_losses(name, case, model, spec, names, x, ctx, gt, tape):
    """(fp64 loss, {dtype: {name: gradient}}, fp32 log-probs) of autograd over the oracle at the model's current weights."""
    stack, state = oracle_state(name, case, model)
    for k in names:
        state[k].requires_grad_(True)
    w = None if spec['weight'] is None else torch.tensor(spec['weight'])
    grads, logps, cost = {}, {}, None
    for dt in (torch.float32, torch.float64):
        for k in names:
            state[k].grad = None
        _, logps[dt] = O.forward(stack, state, x, ctx, synth.NoiseTape(tape), dt)
        cost, _, _ = O.training_loss(logps[dt], gt, case['conf']['data_size'], spec['alpha'], spec['criterion'], None if w is None else w.to(dt))
        cost.backward()
        grads[dt] = {k: state[k].grad.double().clone() for k in names}
    return cost.item(), grads, logps[torch.float32].detach()


def loss_gate(want):
    return 1e-5 + 1e-4 * abs(want)                                  # assert_close(loss, want, 1e-4, 1e-5)


@pytest.mark.parametrize('opt', sorted(OPTIMIZERS))
@pytest.mark.parametrize('name,B', [('cfg1', 37), ('cifar_gen', 21), ('msl_conv_gen', 50), ('cfg4', 50), ('mnist_maf', 9), ('msl_maf', 14),
                                    ('cifar_vardeq', 7), ('mnist_onehot_uniform', 21), ('atm_argmax2', 11)])
def test_gradients_follow_optimizer_steps(name, B, opt):
    """Loss and every gradient of the CUDA training step against autograd over the oracle, before each of STEPS optimizer steps and
    after the last one, with the gate of test_gradients_match_oracle_autograd_fresh_inputs; then the inference log_prob at the trained
    weights (the no-grad path reads caches the training path does not, e.g. the fused plan's CN packs of the context specialists)."""
    case = dict(CASES[name], B=B, iseed='wu_in', nseed='wu_noise')
    spec = TRAINING_CASES[name]
    model = build_cuda_model(case).train()
    names = list(load_train(name)['names'])
    x, ctx = case_inputs(case)
    gt = labels(name + 'wu', B, case['conf']['mixtures'])
    optimizer = OPTIMIZERS[opt]([p for p in model.parameters() if p.requires_grad], lr=LR)
    with torch.no_grad(), rng.use_source(synth.NoiseTape('wu_noise')):
        model.log_prob(x.cuda(), ctx.cuda())                        # the inference caches start filled at the initial weights
    first = None
    for step in range(STEPS + 1):
        want, grads, want_logp = oracle_losses(name, case, model, spec, names, x, ctx, gt, 'wu_noise')
        first = want if first is None else first
        optimizer.zero_grad(set_to_none=True)
        with rng.use_source(synth.NoiseTape('wu_noise')):
            cost, _, _ = reference_loss(model, x.cuda(), ctx.cuda(), gt.cuda(), case['conf']['data_size'], spec)
        cost.backward()
        assert_close(cost.item(), want, 1e-4, 1e-5, f'{name} {opt}: loss after {step} optimizer steps')
        named = dict(model.named_parameters())
        for k in names:
            truth = grads[torch.float64][k]; got = named[k].grad.cpu().double()
            scale = truth.abs().max().item() + 1e-12
            err = (got - truth).abs().max().item()
            ref_err = (grads[torch.float32][k] - truth).abs().max().item()
            assert err <= 2e-4 * scale + REF_FACTOR() * ref_err + 1e-7, \
                f'{name} {opt}: grad {k} after {step} optimizer steps: max abs err {err:.3e}, fp32 reference err {ref_err:.3e}, scale {scale:.3e}'
        if step < STEPS:
            optimizer.step()
    model.eval()
    with torch.no_grad(), rng.use_source(synth.NoiseTape('wu_noise')):
        logp = model.log_prob(x.cuda(), ctx.cuda())
    assert_close(logp.cpu().numpy(), want_logp.numpy(), L_RTOL, L_ATOL, f'{name} {opt}: log_prob after {STEPS} optimizer steps')
    # the steps moved the loss far beyond its gate: a derived value left at the initial weights could not have passed the checks above
    assert abs(want - first) > 100 * loss_gate(want), f'{name} {opt}: the loss moved by {abs(want - first):.3e} only'


def _train(model, trainer, case, spec, B):
    """STEPS optimizer steps on seeded batches, the way the launcher's train_epoch runs them."""
    loss_fn = device_loss(case['conf']['data_size'], spec)
    params = [p for p in model.parameters() if p.requires_grad]
    batches = []
    for i in range(STEPS):
        x, c = case_inputs(dict(case, B=B, iseed=f'wu_train{i}'))
        batches.append((x.cuda(), None if c is None else c.cuda(), labels(f'wu_train{i}', B, case['conf']['mixtures']).cuda()))
    model.train()
    if trainer == 'graphed':
        step = GraphedTrainStep(model, loss_fn, *batches[0]).attach_optimizer(FusedAdamW(params, lr=LR))
        for i, batch in enumerate(batches):
            torch.manual_seed(200 + i)
            step(*batch); step.step()
    else:
        opt = OPTIMIZERS[trainer](params, lr=LR)
        for i, batch in enumerate(batches):
            torch.manual_seed(200 + i)
            opt.zero_grad(set_to_none=True)
            loss_fn(model, *batch).backward()
            opt.step()
    torch.cuda.synchronize()
    model.eval()


@pytest.mark.parametrize('trainer', ['torch_adamw', 'fused_adamw', 'graphed'])
@pytest.mark.parametrize('name,B_train', [('cfg2', 7), ('cfg1', 32), ('mnist_maf', 9), ('cfg4', 50)])
def test_scoring_after_training_matches_oracle(name, B_train, trainer):
    """eval -> train -> eval: every cache the first evaluation filled (fused-plan packs, mixture tables, log|det|, the captured log_prob
    graph, the inverse's operands) must follow the weights the optimizer wrote."""
    case = CASES[name]
    spec = TRAINING_CASES['cifar_vardeq' if name == 'cfg2' else name]       # cfg2 (the bench workload) has cifar_vardeq's loss
    model = build_cuda_model(case).eval()
    B = 37
    x0, c0 = case_inputs(dict(case, B=B, iseed='wu_eval0'))
    x0, c0 = x0.cuda(), c0.cuda()
    out_size = golden_state(load_golden(name), case)[0]['out_size']
    with torch.no_grad():
        with rng.use_source(synth.NoiseTape('wu_eval0')):
            model(x0, c0)
        with rng.use_source(synth.NoiseTape('wu_eval0')):
            model.log_prob(x0, c0)
        if name in FUSED_EXPECTED:
            assert model._fastpath.usable(x0, c0)
        model.enable_cuda_graphs()
        model.log_prob(x0, c0)                                      # captured at the shape scored after training
        if name == 'cfg4':
            model.reverse(synth.NoiseTape('wu_z0').randn((B,) + tuple(out_size)).cuda(), c0)

    _train(model, trainer, case, spec, B_train)

    x, ctx = case_inputs(dict(case, B=B, iseed='wu_eval1'))
    xc, cc = x.cuda(), ctx.cuda()
    stack, state = oracle_state(name, case, model)
    _, want = O.forward(stack, state, x, ctx, synth.NoiseTape('wu_eval1'), torch.float32)
    with torch.no_grad():
        with rng.use_source(synth.NoiseTape('wu_eval1')):
            layers = model(xc, cc)[1]
        with rng.use_source(synth.NoiseTape('wu_eval1')):
            fused = model.log_prob(xc, cc)
        torch.manual_seed(7); replay = model.log_prob(xc, cc)
        torch.manual_seed(7); eager = model.log_prob_eager(xc, cc)
    assert len(model._graphed._entries) == 1
    assert_close(layers.cpu().numpy(), want.numpy(), L_RTOL, L_ATOL, f'{name} {trainer}: layer-by-layer logp after training')
    assert_close(fused.cpu().numpy(), want.numpy(), L_RTOL, L_ATOL, f'{name} {trainer}: log_prob after training')
    assert torch.equal(replay, eager), f'{name} {trainer}: graph replay differs from the eager call, max abs {(replay - eager).abs().max().item():.3e}'
    if name == 'cfg4':
        z = synth.NoiseTape('wu_z1').randn((B,) + tuple(out_size))
        ref = O.reverse(stack, state, z, ctx, synth.NoiseTape('u'), torch.float32)
        with torch.no_grad():
            got = model.reverse(z.cuda(), cc)
        assert_close(got.cpu().numpy(), ref.numpy(), Z_RTOL, Z_ATOL * max(1.0, float(ref.abs().max())), f'{name} {trainer}: reverse after training')


@pytest.fixture
def host_dequant():
    prev = rng._dequant_on_host
    rng.set_dequant_mode('host')
    try:
        yield
    finally:
        rng.set_dequant_mode('host' if prev else 'device')


def test_graphed_train_step_host_dequant_matches_eager(host_dequant):
    """Dequantisation noise drawn on the CPU generator (the reference's uniform.py:32): the captured training step refills its noise
    buffer from the CPU generator before every replay, so under the same seed it trains exactly as the eager step does."""
    name, B = 'cfg1', 32
    case = dict(CASES[name], B=B)
    spec = TRAINING_CASES[name]
    m_eager = build_cuda_model(case).train()
    m_graph = copy.deepcopy(m_eager)
    batches = [case_inputs(dict(case, iseed=f'wu_host{i}')) for i in range(STEPS)]
    gts = [labels(f'wu_host{i}', B, case['conf']['mixtures']).cuda() for i in range(STEPS)]
    loss_fn = device_loss(case['conf']['data_size'], spec)
    opt_e = _TorchAdamW([p for p in m_eager.parameters() if p.requires_grad], lr=1e-3)
    opt_g = _TorchAdamW([p for p in m_graph.parameters() if p.requires_grad], lr=1e-3)
    step = GraphedTrainStep(m_graph, loss_fn, batches[0][0].cuda(), batches[0][1].cuda(), gts[0])
    for i, ((x, c), gt) in enumerate(zip(batches, gts)):
        xc, cc = x.cuda(), c.cuda()
        torch.manual_seed(300 + i)
        opt_e.zero_grad(set_to_none=True)
        le = loss_fn(m_eager, xc, cc, gt); le.backward(); opt_e.step()
        torch.manual_seed(300 + i)
        lg = step(xc, cc, gt); opt_g.step()
        assert le.item() == lg.item(), f'step {i}: loss {le.item()} (eager) vs {lg.item()} (graph replay)'
        for (k, pe), (_, pg) in zip(m_eager.named_parameters(), m_graph.named_parameters()):
            assert torch.equal(pe, pg), f'step {i}: parameter {k} differs after the optimizer step'


# ---- single-process multi-GPU scoring (contextflow_b200/multigpu.py) -------------------------------------------------------------------
def _mg_model():
    """Deterministic time-series stack (even channel count: no Augment noise), as in test_gpu_multigpu.py."""
    conf, model = multigpu_model('cfg4', data_size=(24, 8, 1))
    model.enable_multi_gpu(min_rows=256)
    return conf, model


def _fused_step(model, tag):
    params = [p for p in model.parameters() if p.requires_grad]
    for i, p in enumerate(params):
        p.grad = synth.normal(f'{tag}{i}', tuple(p.shape)).to(p.device)
    FusedAdamW(params, lr=LR).step()


def _non_contiguous(t):
    return torch.stack([t, t], -1)[..., 0]                          # same values, every stride doubled


def test_non_contiguous_inputs_score_like_contiguous_inputs():
    conf, model = multigpu_model('cfg4', data_size=(24, 8, 1))
    x, ctx = synth.make_inputs(conf, 600, 'wu_nc')
    x, ctx = x.to('cuda:0'), ctx.to('cuda:0')
    xn, cn = _non_contiguous(x), _non_contiguous(ctx)
    assert not xn.is_contiguous() and not cn.is_contiguous()
    with torch.no_grad():
        assert torch.equal(model.log_prob(xn, cn), model.log_prob(x, ctx))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_replicas_follow_a_fused_optimizer_step():
    conf, model = _mg_model()
    x, ctx = synth.make_inputs(conf, 2048, 'wu_mg')
    x, ctx = x.to('cuda:0'), ctx.to('cuda:0')
    with torch.no_grad():
        before = model.log_prob(x, ctx)                             # builds and fills the replicas
    _fused_step(model, 'wu_mg_g')
    with torch.no_grad():
        got = model.log_prob(x, ctx)
        ref = model._log_prob_single(x, ctx)
        torch.cuda.synchronize()
    assert not torch.allclose(before, ref)
    assert torch.allclose(got, ref, rtol=1e-5, atol=1e-4), (got - ref).abs().max().item()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_replicated_log_prob_takes_non_contiguous_inputs():
    conf, model = _mg_model()
    x, ctx = synth.make_inputs(conf, 2048, 'wu_mgnc')
    x, ctx = x.to('cuda:0'), ctx.to('cuda:0')
    with torch.no_grad():
        ref = model._log_prob_single(x, ctx)
        got = model.log_prob(_non_contiguous(x), _non_contiguous(ctx))
        torch.cuda.synchronize()
    assert len(model.__dict__['_replicated']._replicas) >= 1
    assert torch.allclose(got, ref, rtol=1e-5, atol=1e-4), (got - ref).abs().max().item()


@pytest.mark.skipif(torch.cuda.device_count() < 3, reason='needs three GPUs')
def test_every_replica_follows_a_weight_update_across_batch_sizes():
    """A weight update, then a batch that uses two GPUs, then one that uses all of them: the replicas the first call left alone must
    still be refreshed by the second."""
    n = torch.cuda.device_count()
    conf, model = _mg_model()
    xs, cs = synth.make_inputs(conf, 512, 'wu_mg2')
    xa, ca = synth.make_inputs(conf, 256 * n, 'wu_mgn')
    xs, cs, xa, ca = xs.to('cuda:0'), cs.to('cuda:0'), xa.to('cuda:0'), ca.to('cuda:0')
    with torch.no_grad():
        model.log_prob(xa, ca)                                      # every replica built at the initial weights
        for p in model.parameters():
            if p.dim() == 1:
                p.add_(0.01)
        small = model.log_prob(xs, cs)
        full = model.log_prob(xa, ca)
        ref_small, ref_full = model._log_prob_single(xs, cs), model._log_prob_single(xa, ca)
        torch.cuda.synchronize()
    assert len(model.__dict__['_replicated']._replicas) == n - 1
    assert torch.allclose(small, ref_small, rtol=1e-5, atol=1e-4), (small - ref_small).abs().max().item()
    assert torch.allclose(full, ref_full, rtol=1e-5, atol=1e-4), (full - ref_full).abs().max().item()
