"""Training of StudentMixtureDistribution (`--dist tdist`, reference layers/distributions/student.py:44-111) through its CUDA kernels:
the prior alone against float64 autograd over O.student_mixture_log_prob, and whole flows whose base density or split priors are Student-t
mixtures, against the oracle's flow composed with the same density, through optimizer steps and CUDA-graph replay."""
import copy
import math
import os

import numpy as np
import pytest
import torch

from contextflow_b200 import layers as L, rng, synth
from contextflow_b200.layers.splitprior import SplitPrior
from contextflow_b200.optim import FusedAdamW, _TorchAdamW
from oracle import flow_oracle as O
from tests.golden.cases import CASES, TRAINING_CASES
from tests.helpers import GOLD, L_ATOL, L_RTOL, assert_close, case_inputs, golden_state, load_golden
from tests.test_gpu_graphed_training import FULL, SIZES, _batches, _compare_runs, _run
from tests.test_gpu_training import build_cuda_model, reference_loss
from tests.test_oracle_golden_training import labels, load_train

pytestmark = pytest.mark.gpu

TRAINED = ('mG', 'sG', 'wG', 'mS', 'sS', 'wS')
GRAD_GATE = 2e-4                    # of the gradient's largest entry
LOGP_RTOL, LOGP_ATOL = 2e-5, 1e-3   # test_gpu_ops.py::test_student_mixture_matches_oracle
OPTIMIZERS = {'torch_adamw': _TorchAdamW, 'fused_adamw': FusedAdamW}
LR, STEPS = 1e-2, 3
# Whole flows: factor on the float32 oracle's own error in the gradient gate (REF_FACTOR of test_gpu_training.py is 4).  At the prior
# itself the kernels' errors against float64 are those of torch float32 autograd over the oracle (measured on a B200 at 6x16x16, M = 10:
# dx 7.3e-4 against 8.5e-4, every parameter gradient within 1.6x); both come from the float32 log-densities, ~1e-3 absolute over 1536
# elements, through the responsibilities.  The bias gradients of the conditioner that feeds cifar_gen's Student split prior are signed
# sums of that input gradient over the batch and the pixels, and there the float32 oracle's error swings between steps: 2.9e-8 in one
# step where the kernels' is 4.9e-7 (scale 4.7e-4), 6.1e-8 against 1.9e-7 in the step before.
FLOW_REF_FACTOR = 16.0


@pytest.fixture
def student_oracle(monkeypatch):
    """O.forward with every mixture that has Student-t parameters in the state evaluated by O.student_mixture_log_prob."""
    gmm = O.gmm_log_prob

    def log_prob(P, state, lay, x, ctx, noise, dt):
        k = lay['key']
        if f'{k}.mS' in state:
            return O.student_mixture_log_prob({n: P(f'{k}.{n}') for n in TRAINED + ('vS',)}, x)
        return gmm(P, state, lay, x, ctx, noise, dt)
    monkeypatch.setattr(O, 'gmm_log_prob', log_prob)


def _student(size, M, seed):
    dist = L.StudentMixtureDistribution(tuple(size), mixtures=M)
    sd = dist.state_dict(); synth.fill_state(sd, seed); dist.load_state_dict(sd)
    return dist.cuda()


def _reference(dist, x, g):
    """float64 autograd over the oracle on the GPU, in batch chunks: (logp, dx, {name: gradient})."""
    P = {k: getattr(dist, k).detach().double().requires_grad_(k != 'vS') for k in TRAINED + ('vS',)}
    chunk = max(1, 2 ** 26 // (dist.M * dist.K * x[0].numel()))
    logps, dxs = [], []
    for i in range(0, x.shape[0], chunk):
        xc = x[i:i + chunk].double().requires_grad_(True)
        lp = O.student_mixture_log_prob(P, xc)
        lp.backward(g[i:i + chunk].double())
        logps.append(lp.detach()); dxs.append(xc.grad)
    assert P['vS'].grad is None
    return torch.cat(logps), torch.cat(dxs), {k: P[k].grad for k in TRAINED}


def _forward_backward(dist, x, g):
    for k in TRAINED:
        getattr(dist, k).grad = None
    xg = x.clone().requires_grad_(True)
    logp = dist.log_prob(xg)
    logp.backward(g)
    return logp.detach(), xg.grad, {k: getattr(dist, k).grad for k in TRAINED}


def _check(dist, x, g, what):
    want_logp, want_dx, want = _reference(dist, x, g)
    logp, dx, got = _forward_backward(dist, x, g)
    assert_close(logp.cpu().numpy(), want_logp.float().cpu().numpy(), LOGP_RTOL, LOGP_ATOL, f'{what}: logp')
    for k, truth, have in [('x', want_dx, dx)] + [(k, want[k], got[k]) for k in TRAINED]:
        scale = truth.abs().max().item() + 1e-30
        err = (have.double() - truth).abs().max().item()
        assert err <= GRAD_GATE * scale, f'{what}: d{k} max abs err {err:.3e}, largest entry {scale:.3e}'
    assert dist.vS.grad is None
    if dist.M == 1:                                                 # softmax over one mixture: the weights have no gradient at all
        assert torch.count_nonzero(got['wG']).item() == 0 and torch.count_nonzero(got['wS']).item() == 0
    return got


def _upstream(B, M, tag):
    g = synth.normal(tag, (B, M))
    g[::3] = 0.0                                                    # rows that receive no gradient
    return g.cuda()


def _inputs(B, size, tag, scale=2.0):
    gen = torch.Generator(device='cuda').manual_seed(sum(map(ord, tag)))
    return (torch.rand((B,) + tuple(size), device='cuda', generator=gen) * 2.0 - 1.0) * scale


@pytest.mark.parametrize('B,M,size', [(9, 2, (8, 16, 16)), (300, 10, (4, 3, 2)), (1, 1, (1, 1, 1)), (8192, 10, (32, 8, 8)), (1000, 1, (26, 8, 1))])
def test_gradients_match_float64_autograd(B, M, size):
    dist = _student(size, M, f'stut{B}')
    _check(dist, _inputs(B, size, f'stutx{B}'), _upstream(B, M, f'stutg{B}'), f'B={B} M={M} {size}')


def test_reference_fixture_parameters():
    from tests.golden.make_golden_extras import STUDENT
    g = dict(np.load(os.path.join(GOLD, 'extras.npz')))
    dist = _student(STUDENT['size'], STUDENT['mixtures'], 'student')
    x = torch.from_numpy(g['stu_x']).cuda()
    _check(dist, x, _upstream(x.shape[0], STUDENT['mixtures'], 'stufix'), 'extras.npz parameters')


@pytest.mark.parametrize('M', [1, 3])
def test_small_scales_and_the_log1p_tail(M):
    """softplus(sS) = 1e-3 with |x - mS| up to 1: |y| up to 1e3, far into log1p's tail, for every df of the linspace(1, 10) init."""
    size = (6, 4, 4)
    dist = _student(size, M, 'stuhard')
    with torch.no_grad():
        dist.sS.fill_(math.log(math.expm1(1e-3)))
        dist.mS.uniform_(-0.05, 0.05)
    assert torch.allclose(torch.nn.functional.softplus(dist.sS), torch.full_like(dist.sS, 1e-3), rtol=1e-3)
    assert torch.equal(dist.vS[0, :, 0, 0, 0].cpu(), torch.linspace(1, 10, 8))
    x = _inputs(64, size, 'stuhardx', scale=1.0)
    _check(dist, x, _upstream(64, M, 'stuhardg'), f'small scales M={M}')


def test_backward_is_deterministic():
    B, M, size = 4096, 10, (32, 8, 8)
    dist = _student(size, M, 'studet')
    x, g = _inputs(B, size, 'studetx'), _upstream(B, M, 'studetg')
    first = _forward_backward(dist, x, g)
    second = _forward_backward(dist, x, g)
    assert torch.equal(first[0], second[0]) and torch.equal(first[1], second[1])
    for k in TRAINED:
        assert torch.equal(first[2][k], second[2][k]), f'd{k} differs between two identical runs'


# ---- whole flows -------------------------------------------------------------------------------------------------------------------
def _with_student_priors(name, model):
    """cfg1: the base density becomes a Student-t mixture of the same size and M.  cifar_gen: every split prior does."""
    M = CASES[name]['conf']['mixtures']
    if name == 'cfg1':
        model.dist = _student(model.dist.size, M, 'stu_base')
    else:
        for i, m in enumerate(model.sequence_modules):
            if isinstance(m, SplitPrior):
                m.dist = _student(m.dist.size, M, f'stu_split{i}')
    return model


def _names(name, model):
    """Parameters the reference's backward reaches: those of the Gaussian-mixture stack minus the replaced priors, plus theirs."""
    keys = dict(model.named_parameters())
    students = [k for k in keys if k.rsplit('.', 1)[-1] in ('mS', 'sS', 'wS')]
    prefixes = {k.rsplit('.', 1)[0] for k in students}
    names = [k for k in load_train(name)['names'] if k in keys and k.rsplit('.', 1)[0] not in prefixes]
    return names + [f'{p}.{n}' for p in sorted(prefixes) for n in TRAINED]


def _oracle(name, case, model, names, x, ctx, gt):
    """(float64 loss, {dtype: {name: gradient}}, float32 log-probs) of autograd over the oracle at the model's current weights."""
    stack = golden_state(load_golden(name), case)[0]
    state = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    for k in names:
        state[k].requires_grad_(True)
    spec = TRAINING_CASES[name]
    w = None if spec['weight'] is None else torch.tensor(spec['weight'])
    grads, logps, cost = {}, {}, None
    for dt in (torch.float32, torch.float64):
        for k in names:
            state[k].grad = None
        _, logps[dt] = O.forward(stack, state, x, ctx, synth.NoiseTape('stu_noise'), dt)
        cost, _, _ = O.training_loss(logps[dt], gt, case['conf']['data_size'], spec['alpha'], spec['criterion'], None if w is None else w.to(dt))
        cost.backward()
        grads[dt] = {k: state[k].grad.double().clone() for k in names}
    return cost.item(), grads, logps[torch.float32].detach()


@pytest.mark.parametrize('opt', sorted(OPTIMIZERS))
@pytest.mark.parametrize('name,B', [('cfg1', 37), ('cifar_gen', 7)])
def test_flow_with_student_priors_trains_like_the_oracle(name, B, opt, student_oracle):
    case = dict(CASES[name], B=B, iseed='stu_in', nseed='stu_noise')
    spec = TRAINING_CASES[name]
    model = _with_student_priors(name, build_cuda_model(case)).train()
    names = _names(name, model)
    x, ctx = case_inputs(case)
    gt = labels(name + 'stu', B, case['conf']['mixtures'])
    optimizer = OPTIMIZERS[opt]([p for p in model.parameters() if p.requires_grad], lr=LR)
    with torch.no_grad(), rng.use_source(synth.NoiseTape('stu_noise')):
        model.log_prob(x.cuda(), ctx.cuda())                        # the scoring table starts filled at the initial weights
    first = None
    named = dict(model.named_parameters())
    for step in range(STEPS + 1):
        want, grads, want_logp = _oracle(name, case, model, names, x, ctx, gt)
        first = want if first is None else first
        optimizer.zero_grad(set_to_none=True)
        with rng.use_source(synth.NoiseTape('stu_noise')):
            cost, _, _ = reference_loss(model, x.cuda(), ctx.cuda(), gt.cuda(), case['conf']['data_size'], spec)
        cost.backward()
        assert_close(cost.item(), want, 1e-4, 1e-5, f'{name} {opt}: loss after {step} optimizer steps')
        for k in names:
            truth = grads[torch.float64][k]; got = named[k].grad.cpu().double()
            scale = truth.abs().max().item() + 1e-12
            err = (got - truth).abs().max().item()
            ref_err = (grads[torch.float32][k] - truth).abs().max().item()
            assert err <= GRAD_GATE * scale + FLOW_REF_FACTOR * ref_err + 1e-7, \
                f'{name} {opt}: grad {k} after {step} optimizer steps: max abs err {err:.3e}, fp32 reference err {ref_err:.3e}, scale {scale:.3e}'
        for k, p in named.items():
            if k.endswith('.vS'):
                assert p.grad is None
        if step < STEPS:
            optimizer.step()
    model.eval()
    with torch.no_grad(), rng.use_source(synth.NoiseTape('stu_noise')):
        logp = model.log_prob(x.cuda(), ctx.cuda())
    assert_close(logp.cpu().numpy(), want_logp.numpy(), L_RTOL, L_ATOL, f'{name} {opt}: log_prob after {STEPS} optimizer steps')
    gate = 1e-5 + 1e-4 * abs(want)
    assert abs(want - first) > 100 * gate, f'{name} {opt}: the loss moved by {abs(want - first):.3e} only'


@pytest.mark.parametrize('opt', sorted(OPTIMIZERS))
@pytest.mark.parametrize('name', ['cfg1', 'cifar_gen'])
def test_training_graphs_match_eager_with_student_priors(name, opt):
    """enable_cuda_graphs(training=True): losses, every .grad and the parameters after each step equal the eager loop's bit for bit,
    over full and ragged batches; the mixture's table is recomputed inside the captured forward after every optimizer step."""
    case = CASES[name]
    m_eager = _with_student_priors(name, build_cuda_model(dict(case, B=FULL))).train()
    x, c = case_inputs(dict(case, B=FULL, iseed='stu_gtr_init'))
    with torch.no_grad():
        m_eager.log_prob(x.cuda(), c.cuda())
    m_graph = copy.deepcopy(m_eager).enable_cuda_graphs(training=True)
    batches = _batches(name, case, SIZES, 'stu_gtr')
    make = OPTIMIZERS[opt]
    want = _run(m_eager, make([p for p in m_eager.parameters() if p.requires_grad], lr=LR), name, case, batches)
    got = _run(m_graph, make([p for p in m_graph.parameters() if p.requires_grad], lr=LR), name, case, batches)
    _compare_runs(want, got, f'{name} {opt} Student-t priors')
    assert len(m_graph._graphed_train._entries) == 2
