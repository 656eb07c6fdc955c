"""The tensor-core Gaussian-mixture kernel (csrc/gmm_tc.cu) behind ops.gmm_tile_logprob, against an fp64 evaluation of the density:
the cfg2 prior levels and other shapes, 0 / 1 / 2 context features, bucket edge cases, strided views, fp32-range parameters and inputs,
the accuracy guard's routing to the exact kernel, and run-to-run determinism."""
import math
import pytest
import torch

from contextflow_b200 import ops, synth
from tests.helpers import L_ATOL, L_RTOL, assert_close

pytestmark = pytest.mark.gpu
dev = 'cuda'


def _oracle(x, mG, sG, wG, ctx=None, tabs=None, chunk=128):
    """fp64 log-prob, on the device in sample chunks.  tabs: the context tables ('b (p m k d)': means then scales)."""
    M, K, D = mG.shape[:3]
    B, MKD = x.shape[0], M * K * D
    out = []
    for b0 in range(0, B, chunk):
        xs = x[b0:b0 + chunk].double().reshape(-1, 1, 1, D, x.shape[2] * x.shape[3])
        mean = mG.double().reshape(1, M, K, D, -1)
        pre = sG.double().reshape(1, M, K, D, -1)
        if tabs is not None:
            c = torch.cat([t[ctx[b0:b0 + chunk, i]] for i, t in enumerate(tabs)], 1).double()
            mean = mean + c[:, :MKD].reshape(-1, M, K, D, 1)
            pre = pre + c[:, MKD:].reshape(-1, M, K, D, 1)
        scale = torch.nn.functional.softplus(pre)
        comp = (-((xs - mean) ** 2) / (2 * scale ** 2) - scale.log() - 0.5 * math.log(2 * math.pi)).sum((-2, -1))
        out.append(torch.logsumexp(comp + torch.log_softmax(wG.double(), -1)[None], -1))
    return torch.cat(out)


def _params(tag, M, K, D, H, W, sigma=None, mean=None):
    mG = synth.uniform(f'{tag}m', (M, K, D, H, W)).to(dev) if mean is None else torch.full((M, K, D, H, W), float(mean), device=dev)
    sG = (1 + 0.3 * synth.uniform(f'{tag}s', (M, K, D, H, W))).to(dev)
    if sigma is not None:
        sG = torch.full_like(sG, math.log(math.expm1(sigma)))
    return mG, sG, synth.uniform(f'{tag}w', (M, K)).to(dev)


def _tables(tag, M, K, D, cards, scale=0.2):
    width = 2 * M * K * D // len(cards)
    return [(synth.uniform(f'{tag}t{i}', (card, width)) * scale).to(dev) for i, card in enumerate(cards)]


def _run(x, mG, sG, wG, ctx=None, cards=(), tabs=None):
    M, K, D = mG.shape[:3]
    if not cards:
        return ops.gmm_tile_logprob(x, ops.gmm_tile_table(mG, sG, wG), M, K)
    n = len(cards)
    tab = ops.gmm_tile_table(mG, sG, wG, tabs[n - 1], 0 if n == 2 else M * K * D)
    return ops.gmm_tile_logprob(x, tab, M, K, ctx, list(cards), tabs[0], 0)


def _ctx(tag, B, cards):
    return torch.stack([synth.randint(f'{tag}c{i}', (B,), card) for i, card in enumerate(cards)], 1).to(dev)


# the three cfg2 prior levels (D x H x W) with M = 10, K = 8, and a wider D at HW = 16
LEVELS = [(8, 16, 16), (16, 8, 8), (64, 4, 4), (48, 4, 4)]


@pytest.mark.parametrize('D,H,W', LEVELS)
@pytest.mark.parametrize('B', [8192, 1000])
@pytest.mark.parametrize('cards', [(), (10,), (15, 5)])
def test_tc_matches_fp64(D, H, W, B, cards):
    M, K = 10, 8
    mG, sG, wG = _params('tc', M, K, D, H, W)
    x = (synth.uniform('tcx', (B, D, H, W)) * 2).to(dev)
    ctx = _ctx('tc', B, cards) if cards else None
    tabs = _tables('tc', M, K, D, cards) if cards else None
    got = _run(x, mG, sG, wG, ctx, cards, tabs)
    assert_close(got.cpu().numpy(), _oracle(x, mG, sG, wG, ctx, tabs).cpu().numpy(), L_RTOL, L_ATOL, f'gmm tc {D}x{H}x{W} B={B} cards={cards}')
    assert torch.equal(got, _run(x, mG, sG, wG, ctx, cards, tabs)), 'two runs differ'


@pytest.mark.parametrize('case', ['one_tuple', 'sparse'])
def test_tc_bucket_edges(case):
    """All samples in one tuple (one bucket of many tiles), and a batch that leaves most of 75 buckets empty."""
    M, K, D, H, W = 10, 8, 16, 8, 8
    cards, B = ((10,), 3000) if case == 'one_tuple' else ((15, 5), 300)
    mG, sG, wG = _params('be', M, K, D, H, W)
    x = (synth.uniform('bex', (B, D, H, W)) * 2).to(dev)
    ctx = torch.full((B, 1), 7, dtype=torch.int64, device=dev) if case == 'one_tuple' else _ctx('be', B, cards)
    tabs = _tables('be', M, K, D, cards)
    assert_close(_run(x, mG, sG, wG, ctx, cards, tabs).cpu().numpy(), _oracle(x, mG, sG, wG, ctx, tabs).cpu().numpy(), L_RTOL, L_ATOL, case)


def test_tc_strided_view():
    """SplitPrior reads x[:, C/2:] in place: rows through the batch stride."""
    M, K, D, H, W, B = 10, 8, 8, 16, 16, 777
    mG, sG, wG = _params('sv', M, K, D, H, W)
    x = (synth.uniform('svx', (B, D, H, W)) * 2).to(dev)
    wide = torch.cat([torch.zeros_like(x), x], 1)
    got = _run(wide[:, D:], mG, sG, wG)
    assert torch.equal(got, _run(x.contiguous(), mG, sG, wG))
    assert_close(got.cpu().numpy(), _oracle(x, mG, sG, wG).cpu().numpy(), L_RTOL, L_ATOL, 'strided view')


def test_tc_fp32_range():
    """sigma = 1e-3 (a = 5e5) and |x| up to 1e3: beyond the fp16 range, inside the tf32 pair's."""
    M, K, D, H, W, B = 8, 8, 16, 8, 8, 640
    mG, sG, wG = _params('fr', M, K, D, H, W, sigma=1e-3, mean=0.0)
    x = ((synth.uniform('frx', (B, D, H, W)) * 2 - 1) * 1e3).to(dev)
    assert_close(_run(x, mG, sG, wG).cpu().numpy(), _oracle(x, mG, sG, wG).cpu().numpy(), L_RTOL, L_ATOL, 'sigma 1e-3, |x| 1e3')


def _guard_mean(E, K, wG, frac):
    """A constant mean m whose guard term 4 * 2^-20 * sum_e a m^2 (sigma = 1: a = 1/2) is `frac` of what the guard allows."""
    lbmax = (torch.log_softmax(wG.double(), -1).max(-1).values - 0.5 * E * math.log(2 * math.pi)).min().item()
    allow = 0.1 * (L_ATOL + L_RTOL * max(0.0, -(lbmax + math.log(K))))
    return math.sqrt(frac * allow / (4 * 2.0 ** -20 * 0.5 * E))


@pytest.mark.parametrize('frac', [0.9, 1e4])
def test_tc_guard(frac):
    """x ~ m: the expansion cancels.  Just inside the guard the tensor-core result passes the gate; far beyond it (where the expansion's
    error would be ~100x the tolerance) every slice is flagged and the exact tile kernel's result passes it."""
    M, K, D, H, W, B = 10, 8, 16, 8, 8, 1024
    E = D * H * W
    wG = synth.uniform('gdw', (M, K)).to(dev)
    m = _guard_mean(E, K, wG, frac)
    mG, sG, _ = _params('gd', M, K, D, H, W, sigma=1.0, mean=m)
    x = (m + synth.uniform('gdx', (B, D, H, W)) * 2 - 1).to(dev)
    want = _oracle(x, mG, sG, wG)
    got = _run(x, mG, sG, wG)
    assert_close(got.cpu().numpy(), want.cpu().numpy(), L_RTOL, L_ATOL, f'guard frac={frac}')
    if frac > 1:   # the exact kernel's per-slice sums: the same numbers as the misaligned-x route, which never takes the tensor cores
        flat = torch.zeros(x.numel() + 1, device=dev); flat[1:] = x.flatten()
        ref = _run(flat[1:].view_as(x), mG, sG, wG)
        assert_close(got.cpu().numpy(), ref.cpu().numpy(), 1e-6, 1e-5, 'beyond the guard: exact kernel')
