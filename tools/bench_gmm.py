"""Micro-benchmark of the mixture log-prob kernels at the cfg2 prior shapes and a wider-D HW16 shape: the tensor-core kernel (gmm_tc, aligned
x) against the exact register-tiled kernel (tile_kernel, reached through a misaligned view of the same x), and the max error of each
against fp64 in units of the log-prob tolerance (atol 1e-3 + rtol 1e-4 |ref|)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from contextflow_b200 import ops

dev = 'cuda'
B = int(os.environ.get('B', 8192))
M, K = 10, 8
cards = [15, 5]


def timeit(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def fp64(x, mG, sG, wG, chunk=256):
    out = []
    for b0 in range(0, x.shape[0], chunk):
        xs = x[b0:b0 + chunk].double()[:, None, None]
        sc = torch.nn.functional.softplus(sG.double())
        comp = (-((xs - mG.double()) ** 2) / (2 * sc ** 2) - sc.log() - 0.9189385332046727).sum((-3, -2, -1))
        out.append(torch.logsumexp(comp + torch.log_softmax(wG.double(), -1), -1))
    return torch.cat(out)


for D, H, W in [(8, 16, 16), (16, 8, 8), (64, 4, 4), (48, 4, 4)]:
    xs = [torch.randn(B, 2 * D, H, W, device=dev) for _ in range(3)]
    mG, sG, wG = torch.randn(M, K, D, H, W, device=dev), torch.ones(M, K, D, H, W, device=dev), torch.randn(M, K, device=dev)
    tabs = [torch.randn(c, M * K * D, device=dev) * 0.1 for c in cards]
    ctx = torch.stack([torch.randint(0, c, (B,), device=dev) for c in cards], 1)
    it = [0]
    def nx():
        it[0] += 1; return xs[it[0] % 3][:, D:]
    tab = ops.gmm_tile_table(mG, sG, wG, tabs[1], 0)
    tab0 = ops.gmm_tile_table(mG, sG, wG)
    t_tile = timeit(lambda: ops.gmm_tile_logprob(nx(), tab, M, K, ctx, cards, tabs[0], 0))
    t_plain = timeit(lambda: ops.gmm_tile_logprob(nx(), tab0, M, K))
    t_old = timeit(lambda: ops.gmm_logprob_ctxtab(nx(), mG, sG, wG, ctx, cards, tabs))
    flat = torch.empty(B * D * H * W + 1, device=dev)
    xm = flat[1:].view(B, D, H, W); xm.copy_(xs[0][:, D:])                     # misaligned rows: the exact tile kernel
    t_exact = timeit(lambda: ops.gmm_tile_logprob(xm, tab0, M, K))
    ref = fp64(xs[0][:, D:], mG, sG, wG)
    tol = 1e-3 + 1e-4 * ref.abs()
    err_tc = ((ops.gmm_tile_logprob(xs[0][:, D:], tab0, M, K).double() - ref).abs() / tol).max().item()
    err_exact = ((ops.gmm_tile_logprob(xm, tab0, M, K).double() - ref).abs() / tol).max().item()
    ev = B * M * K * D * H * W
    print(json.dumps({'D': D, 'HW': H * W, 'tile_ctx_us': round(t_tile, 1), 'tile_plain_us': round(t_plain, 1), 'old_ctxtab_us': round(t_old, 1), 'exact_plain_us': round(t_exact, 1),
                      'err_tol_tc': round(err_tc, 4), 'err_tol_exact': round(err_exact, 4),
                      'tile_ctx_Gevals_s': round(ev / t_tile / 1e3, 1), 'fp32_issue_frac_4op': round(4 * ev / (t_tile * 1e-6) / (148 * 128 * 1.965e9), 3)}))
