"""CUDA-graph replay of log_prob under autograd (graphed.GraphedTrainLogProb) inside the training loop as the reference writes it
(experiment_ad.py:204-213): CPU batch -> .to(device), dim_inv * log_prob, NaN scrub, loss with CPU constants, zero_grad(), backward(),
optimizer.step(), .item().  Every check compares a model with training graphs against an eager copy, bit for bit."""
import copy

import pytest
import torch

from contextflow_b200 import _cabi, rng, synth
from contextflow_b200.graphed import GraphedTrainStep
from contextflow_b200.optim import FusedAdamW, _TorchAdamW
from tests.golden.cases import CASES, TRAINING_CASES
from tests.helpers import case_inputs
from tests.test_gpu_training import build_cuda_model, device_loss, labels, reference_loss

pytestmark = pytest.mark.gpu

OPTIMIZERS = {'torch_adamw': _TorchAdamW, 'fused_adamw': FusedAdamW}
FULL, RAGGED = 24, 13
SIZES = (FULL, FULL, RAGGED, FULL, RAGGED)          # the ragged shape runs eagerly first, then is captured
NO_CONTEXT = {'cfg4'}                               # the generalist trained as model.log_prob(x)


def _spec(name):
    return TRAINING_CASES['cifar_vardeq' if name == 'cfg2' else name]


def _pair(name):
    """(case, eager model, copy with training graphs), both after ActNorm's data-dependent initialisation."""
    case = CASES[name]
    m_eager = build_cuda_model(dict(case, B=FULL)).train()
    x, c = case_inputs(dict(case, B=FULL, iseed='gtr_init'))
    with torch.no_grad():
        m_eager.log_prob(x.cuda(), None if name in NO_CONTEXT else c.cuda())
    return case, m_eager, copy.deepcopy(m_eager).enable_cuda_graphs(training=True)


def _batches(name, case, sizes, tag):
    """CPU batches, as a DataLoader hands them to the loop."""
    out = []
    for i, B in enumerate(sizes):
        x, c = case_inputs(dict(case, B=B, iseed=f'{tag}{i}'))
        out.append((x, None if name in NO_CONTEXT else c, labels(f'{tag}{i}', B, case['conf']['mixtures'])))
    return out


def _loss(model, name, case, batch):
    x, c, gt = batch
    cost, _, _ = reference_loss(model, x.to('cuda'), None if c is None else c.to('cuda'), gt.to('cuda'), case['conf']['data_size'], _spec(name))
    return cost


def _grads(model):
    return {k: None if p.grad is None else p.grad.clone() for k, p in model.named_parameters()}


def _assert_same_grads(want, got, what):
    assert want.keys() == got.keys()
    for k in want:
        if want[k] is None or got[k] is None:
            assert want[k] is None and got[k] is None, f'{what}: .grad of {k} is {want[k] is None} None (eager) vs {got[k] is None} (graphs)'
        else:
            assert torch.equal(want[k], got[k]), f'{what}: .grad of {k} differs, max abs {(want[k] - got[k]).abs().max().item():.3e}'


def _assert_same_params(m_eager, m_graph, what):
    for (k, pe), (_, pg) in zip(m_eager.named_parameters(), m_graph.named_parameters()):
        assert torch.equal(pe, pg), f'{what}: parameter {k} differs'


def _run(model, opt, name, case, batches, seed=11):
    """The reference's loop body over `batches`, one seed for the whole run: [(loss, grads, params after the step)]."""
    torch.manual_seed(seed)
    out = []
    for batch in batches:
        cost = _loss(model, name, case, batch)
        opt.zero_grad()
        cost.backward()
        grads = _grads(model)
        opt.step()
        out.append((cost.item(), grads, [p.detach().clone() for p in model.parameters()]))
    return out


def _compare_runs(want, got, what):
    for i, ((le, ge, pe), (lg, gg, pg)) in enumerate(zip(want, got)):
        assert le == lg, f'{what} step {i}: loss {le} (eager) vs {lg} (graphs)'
        _assert_same_grads(ge, gg, f'{what} step {i}')
        assert all(torch.equal(a, b) for a, b in zip(pe, pg)), f'{what} step {i}: parameters differ after the optimizer step'


def _optimizer(kind, model):
    return OPTIMIZERS[kind]([p for p in model.parameters() if p.requires_grad], lr=1e-3)


@pytest.mark.parametrize('opt', sorted(OPTIMIZERS))
@pytest.mark.parametrize('name', ['cfg1', 'cifar_vardeq', 'cifar_gen', 'atm_argmax2', 'cfg4', 'cifar_conventional', 'mnist_maf'])
def test_training_loop_matches_eager(name, opt):
    case, m_eager, m_graph = _pair(name)
    batches = _batches(name, case, SIZES, 'gtr_loop')
    want = _run(m_eager, _optimizer(opt, m_eager), name, case, batches)
    o_graph = _optimizer(opt, m_graph)
    got = _run(m_graph, o_graph, name, case, batches)
    _compare_runs(want, got, f'{name} {opt}')
    assert len(m_graph._graphed_train._entries) == 2

    # steady state: a full batch replays both graphs, no libcfpp launch from the host, every .grad a view of one fresh buffer
    x, c, gt = batches[0]
    x, c, gt = x.cuda(), None if c is None else c.cuda(), gt.cuda()
    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    cost, _, _ = reference_loss(m_graph, x, c, gt, case['conf']['data_size'], _spec(name))
    o_graph.zero_grad()
    cost.backward()
    assert _cabi.launch_count() == l0
    assert len(m_graph._graphed_train._entries) == 2
    storages = {p.grad.untyped_storage().data_ptr() for p in m_graph.parameters() if p.grad is not None}
    assert len(storages) == 1


@pytest.fixture
def host_dequant():
    prev = rng._dequant_on_host
    rng.set_dequant_mode('host')
    try:
        yield
    finally:
        rng.set_dequant_mode('host' if prev else 'device')


def test_host_dequantisation_matches_eager(host_dequant):
    """Dequantisation noise from the CPU generator: the replay refills its noise buffer from the CPU generator, so the CPU stream is
    consumed as by the eager loop."""
    case, m_eager, m_graph = _pair('cfg2')
    batches = _batches('cfg2', case, (8, 8, 5, 8, 5), 'gtr_host')
    want = _run(m_eager, _optimizer('torch_adamw', m_eager), 'cfg2', case, batches)
    got = _run(m_graph, _optimizer('torch_adamw', m_graph), 'cfg2', case, batches)
    _compare_runs(want, got, 'cfg2 host dequantisation')
    assert len(m_graph._graphed_train._entries) == 2


def _primed(name='cifar_vardeq'):
    """Both arms after two loss+backward calls at the full shape: the graph arm has captured and replays from then on."""
    case, m_eager, m_graph = _pair(name)
    batch = _batches(name, case, (FULL,), 'gtr_sem')[0]
    for m in (m_eager, m_graph):
        torch.manual_seed(3)
        for _ in range(2):
            _loss(m, name, case, batch).backward()
        m.zero_grad(set_to_none=True)
    assert len(m_graph._graphed_train._entries) == 1
    return name, case, m_eager, m_graph, batch


def _on_both(m_eager, m_graph, fn, seed=21):
    out = []
    for m in (m_eager, m_graph):
        torch.manual_seed(seed)
        out.append(fn(m))
    return out


def test_gradients_accumulate_without_zero_grad():
    name, case, m_eager, m_graph, batch = _primed()

    def fn(m):
        _loss(m, name, case, batch).backward()
        _loss(m, name, case, batch).backward()
        return _grads(m)
    want, got = _on_both(m_eager, m_graph, fn)
    _assert_same_grads(want, got, 'two backwards without zero_grad')


def test_zero_grad_keeps_tensors():
    name, case, m_eager, m_graph, batch = _primed()

    def fn(m):
        _loss(m, name, case, batch).backward()
        m.zero_grad(set_to_none=False)
        _loss(m, name, case, batch).backward()
        return _grads(m)
    want, got = _on_both(m_eager, m_graph, fn)
    _assert_same_grads(want, got, 'zero_grad(set_to_none=False)')


def test_autograd_grad_leaves_dot_grad_alone():
    name, case, m_eager, m_graph, batch = _primed()

    def fn(m):
        params = [p for p in m.parameters() if p.requires_grad]
        for i, p in enumerate(params):
            p.grad = torch.full_like(p, float(i))
        g = torch.autograd.grad(_loss(m, name, case, batch), params, allow_unused=True)
        assert all(torch.equal(p.grad, torch.full_like(p, float(i))) for i, p in enumerate(params))
        return g
    want, got = _on_both(m_eager, m_graph, fn)
    assert len(want) == len(got)
    for a, b in zip(want, got):
        assert (a is None and b is None) or torch.equal(a, b)


def test_two_log_probs_in_one_loss():
    name, case, m_eager, m_graph, batch = _primed()

    def fn(m):
        (_loss(m, name, case, batch) + 0.5 * _loss(m, name, case, batch)).backward()
        return _grads(m)
    want, got = _on_both(m_eager, m_graph, fn)
    _assert_same_grads(want, got, 'two log_prob calls in one loss')


def test_retain_graph_and_overwritten_activations():
    name, case, m_eager, m_graph, batch = _primed()

    def fn(m):
        cost = _loss(m, name, case, batch)
        cost.backward(retain_graph=True)
        cost.backward()
        return _grads(m)
    want, got = _on_both(m_eager, m_graph, fn)
    _assert_same_grads(want, got, 'retain_graph=True, two backwards')
    first = _loss(m_graph, name, case, batch)
    first.backward(retain_graph=True)
    _loss(m_graph, name, case, batch).backward()                 # replays again: the first forward's activations are gone
    with pytest.raises(RuntimeError, match='overwrote the activations'):
        first.backward()


@pytest.mark.parametrize('name', ['cifar_vardeq', 'cfg4'])
def test_input_that_requires_grad_stays_eager(name):
    name, case, m_eager, m_graph, batch = _primed(name)
    entry = next(iter(m_graph._graphed_train._entries.values()))
    replays = entry.generation

    def fn(m):
        x, c, gt = batch
        x = x.cuda().requires_grad_(True)
        cost, _, _ = reference_loss(m, x, None if c is None else c.cuda(), gt.cuda(), case['conf']['data_size'], _spec(name))
        cost.backward()
        return x.grad, _grads(m)
    (xe, ge), (xg, gg) = _on_both(m_eager, m_graph, fn)
    assert entry.generation == replays                          # the call ran eagerly
    assert (xe is None and xg is None) or torch.equal(xe, xg)
    _assert_same_grads(ge, gg, 'x.requires_grad')


@pytest.mark.parametrize('change', ['load_state_dict', 'freeze', 'double_and_back'])
def test_invalidation_matches_eager(change):
    name = 'cifar_vardeq'                                       # contextflow specialist: ActNorm's NN_t / NN_logs are frozen
    case, m_eager, m_graph = _pair(name)
    batches = _batches(name, case, SIZES, 'gtr_inv')
    o_eager, o_graph = _optimizer('fused_adamw', m_eager), _optimizer('fused_adamw', m_graph)
    _compare_runs(_run(m_eager, o_eager, name, case, batches[:2]), _run(m_graph, o_graph, name, case, batches[:2]), f'{change}: before')
    assert any(not p.requires_grad for p in m_graph.parameters())
    for m in (m_eager, m_graph):
        if change == 'load_state_dict':
            sd = m.state_dict()
            synth.fill_state(sd, 'gtr_new')
            m.load_state_dict(sd)
        elif change == 'freeze':
            next(p for k, p in m.named_parameters() if p.requires_grad and 'dist' not in k).requires_grad_(False)
        else:
            m.double(); m.float()
    _assert_same_params(m_eager, m_graph, change)
    _compare_runs(_run(m_eager, o_eager, name, case, batches), _run(m_graph, o_graph, name, case, batches), f'{change}: after')
    assert len(m_graph._graphed_train._entries) == 2


def test_scoring_between_training_steps():
    """no_grad scoring replays its own graph, equal to log_prob_eager; the training graphs do not touch the scoring entries."""
    name, case, m_eager, m_graph, batch = _primed()
    x, c, _ = batch
    xc, cc = x.cuda(), c.cuda()
    opt = _optimizer('fused_adamw', m_graph)
    for i in range(3):
        torch.manual_seed(40 + i)
        _loss(m_graph, name, case, batch).backward()
        opt.step(); opt.zero_grad()
        with torch.no_grad():
            torch.manual_seed(7); replay = m_graph.log_prob(xc, cc)
            torch.manual_seed(7); eager = m_graph.log_prob_eager(xc, cc)
        assert torch.equal(replay, eager), f'step {i}: scoring replay differs from log_prob_eager'
        assert len(m_graph._graphed._entries) == 1
        assert len(m_graph._graphed_train._entries) == 1


@pytest.mark.parametrize('name', ['cfg1', 'cifar_vardeq'])
def test_graphed_train_step_over_a_model_with_training_graphs(name):
    """GraphedTrainStep captures loss and backward itself: a model whose log_prob training graphs are on (and have replayed) gives the
    same GraphedTrainStep result as one without them."""
    case, m_plain, m_graph = _pair(name)
    batches = _batches(name, case, (FULL, FULL, FULL), 'gtr_gts')
    for _ in range(2):                                           # the training graphs capture and replay; no optimizer step
        _loss(m_graph, name, case, batches[0]).backward()
    m_graph.zero_grad(set_to_none=True)
    loss_fn = device_loss(case['conf']['data_size'], _spec(name))
    results = []
    for m in (m_plain, m_graph):
        x, c, gt = (t.cuda() for t in batches[1])
        torch.manual_seed(5)
        step = GraphedTrainStep(m, loss_fn, x, c, gt)
        out = []
        for x, c, gt in batches:
            torch.manual_seed(6)
            out.append((step(x.cuda(), c.cuda(), gt.cuda()).item(), _grads(m)))
        results.append(out)
    for (la, ga), (lb, gb) in zip(*results):
        assert la == lb
        _assert_same_grads(ga, gb, 'GraphedTrainStep')
