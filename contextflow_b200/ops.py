"""Tensor-level wrappers over the C ABI (include/cfpp.h).  torch supplies device memory and the stream; every
computation below is a libcfpp kernel.  CPU tensors are rejected: there is no fallback path."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

from . import _cabi
from ._cabi import check, lib, vp


class OpTimer:
    """Collects (op, cuda start event, cuda end event, work dict) per libcfpp launch on the launching stream (bench.py)."""

    def __init__(self):
        self.records = []

    def summary(self):
        out = {}
        for name, s, e, work in self.records:
            d = out.setdefault(name, dict(ms=0.0, n=0, bytes=0.0, flops=0.0, shapes={}))
            ms = s.elapsed_time(e)
            d['ms'] += ms; d['n'] += 1
            d['bytes'] += work.get('bytes', 0.0); d['flops'] += work.get('flops', 0.0)
            if 'shape' in work:
                sh = d['shapes'].setdefault(work['shape'], dict(ms=0.0, n=0, bytes=0.0, flops=0.0))
                sh['ms'] += ms; sh['n'] += 1; sh['bytes'] += work.get('bytes', 0.0); sh['flops'] += work.get('flops', 0.0)
        return out


_timer = None          # set to an OpTimer to time every launch with CUDA events
_work = {}             # algorithmic work of the next launch (bytes / flops), set by the wrapper that knows the shapes


def set_timer(t):
    global _timer
    _timer = t


_dev = None            # device of the current op's tensors (set by _need_cuda): launches go to ITS current stream under ITS context


def _call(name, args, label=None):
    global _work
    if _dev is not None and _dev.index != torch.cuda.current_device():
        # the reference builds torch.device('cuda:{gpu}') and never calls set_device (model.py:170): launch under the tensors' device
        with torch.cuda.device(_dev):
            return _call_on_device(name, args)
    return _call_on_device(name, args)


def _call_on_device(name, args):
    global _work
    fn = getattr(lib(), 'cfpp_' + name)
    if _timer is None:
        _work = {}
        check(fn(*args), name)
        return
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    rc = fn(*args)
    e.record()
    _timer.records.append((name, s, e, _work)); _work = {}
    check(rc, name)


def _set_work(**kw):
    global _work
    _work = kw


def _stream():
    return vp(torch.cuda.current_stream(_dev).cuda_stream)


def _need_cuda(*ts):
    global _dev
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError('contextflow_b200 kernels run on CUDA tensors only (no CPU fallback); got a CPU tensor')
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f'contextflow_b200: tensor arguments live on different devices ({dev} and {t.device})')
    if dev is not None:
        _dev = dev


def _f32(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise TypeError(f'float32 expected, got {t.dtype}')
    return t if t.is_contiguous() else t.contiguous()


def _p(t: Optional[torch.Tensor]):
    return None if t is None else vp(t.data_ptr())


def _half_view(x: torch.Tensor):
    """Accept (B,C,H,W) tensors that are contiguous or a channel-slice view of a contiguous tensor: returns batch stride."""
    if x.dtype != torch.float32:
        raise TypeError(f'float32 expected, got {x.dtype}')
    B, Cc, H, W = x.shape
    st = x.stride()
    if B == 0 or (st[1] == H * W and st[2] == W and st[3] == 1) or (Cc == 1 and st[2] == W and st[3] == 1):
        return x, (st[0] if B > 1 else Cc * H * W)
    x = x.contiguous()
    return x, Cc * H * W


# ---------------------------------------------------------------------------------------------- index ops
def squeeze(x, p1, p2):
    _need_cuda(x)
    if not x.is_contiguous() and x.dtype == torch.float32 and x.dim() == 4 and p1 == 2 and p2 == 2 and x.shape[3] % 8 == 0:
        st = x.stride()                                          # a leading-channels view of a wider tensor (SplitPrior's z): read it in place
        B, Cc, H, W = x.shape
        if st[3] == 1 and st[2] == W and st[1] == H * W and st[0] % 4 == 0 and st[0] >= Cc * H * W and x.data_ptr() % 16 == 0:
            y = torch.empty((B, Cc * 4, H // 2, W // 2), device=x.device, dtype=x.dtype)
            _set_work(bytes=8.0 * x.numel())
            _call('squeeze_strided_fwd', (_p(x), st[0], _p(y), B, Cc, H, W, p1, p2, _stream()), 'squeeze_fwd')
            return y
    x = _f32(x)
    B, Cc, H, W = x.shape
    y = torch.empty((B, Cc * p1 * p2, H // p1, W // p2), device=x.device, dtype=x.dtype)
    _set_work(bytes=8.0 * x.numel())
    _call('squeeze_fwd', (_p(x), _p(y), B, Cc, H, W, p1, p2, _stream()), 'squeeze_fwd')
    return y


def unsqueeze(y, p1, p2):
    _need_cuda(y); y = _f32(y)
    B, Cs, Hs, Ws = y.shape
    Cc, H, W = Cs // (p1 * p2), Hs * p1, Ws * p2
    x = torch.empty((B, Cc, H, W), device=y.device, dtype=y.dtype)
    _set_work(bytes=8.0 * y.numel())
    _call('squeeze_inv', (_p(y), _p(x), B, Cc, H, W, p1, p2, _stream()), 'squeeze_inv')
    return x


def permute_chw(x):
    _need_cuda(x); x = _f32(x)
    B, Cc, H, W = x.shape
    y = torch.empty((B, H, Cc, W), device=x.device, dtype=x.dtype)
    step = max(1, 65535 // max(W, 1))
    for b0 in range(0, B, step):
        nb = min(step, B - b0)
        _set_work(bytes=8.0 * nb * Cc * H * W)
        _call('permute_fwd', (_p(x[b0:]), _p(y[b0:]), nb, Cc, H, W, _stream()), 'permute_fwd')
    return y


def slice_channels(x, c0, cn):
    _need_cuda(x); x = _f32(x)
    B, Cc, H, W = x.shape
    y = torch.empty((B, cn, H, W), device=x.device, dtype=x.dtype)
    _set_work(bytes=8.0 * y.numel())
    _call('slice_channels', (_p(x), _p(y), B, Cc, H * W, c0, cn, _stream()), 'slice_channels')
    return y


def windows(ts, L, end=None, end0=0, stride=1, count=None):
    """Sliding windows of a device-resident series (n_rows, D) in the model layout (B, D, L, 1): get_windows + the dataset transpose
    (mtad_data_preprocess.py:58-74, mtad_dataloader.py:106-110).  end: int64 (B,) window end rows, or the arithmetic run end0 + b*stride."""
    _need_cuda(ts, end)
    if ts.dtype not in (torch.float32, torch.float64) or ts.dim() != 2:
        raise TypeError('series must be a (rows, D) float32 / float64 tensor')
    ts = ts.contiguous()
    n_rows, D = ts.shape
    if end is not None:
        if end.dtype != torch.int64:
            raise TypeError('window end rows must be int64')
        end = end.contiguous(); B = end.shape[0]
    else:
        B = int(count)
    x = torch.empty((B, D, L, 1), device=ts.device, dtype=torch.float32)
    _set_work(bytes=4.0 * x.numel() * 2)
    _call('windows_fwd', (_p(ts), int(ts.dtype == torch.float64), _p(end), int(end0), int(stride), _p(x), B, n_rows, D, L, _stream()))
    return x


# ---------------------------------------------------------------------------------------------- prologue
def add(x, u):
    _need_cuda(x, u); x = _f32(x); u = _f32(u)
    y = torch.empty_like(x)
    _call('add_fwd', (_p(x), _p(u), _p(y), x.numel(), _stream()), 'add_fwd')
    return y


def normalize(x, scale: float, translation: float):
    _need_cuda(x); x = _f32(x)
    y = torch.empty_like(x)
    _call('normalize_fwd', (_p(x), _p(y), x.numel(), scale, translation, _stream()), 'normalize_fwd')
    return y


def logit(x):
    _need_cuda(x); x = _f32(x)
    B = x.shape[0]
    y = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    _call('logit_fwd', (_p(x), _p(y), _p(ldj), B, x[0].numel() if B else 0, _stream()), 'logit_fwd')
    return y, ldj


def augment(x, eps):
    """cat([x, eps], 1) and ldj = sum(0.5 log 2pi + 0.5 eps^2) (B,).  x may be None (pure noise log-density)."""
    _need_cuda(eps); eps = _f32(eps)
    B, A = eps.shape[0], eps.shape[1]
    HW = eps[0, 0].numel() if B else 1
    Cc = 0 if x is None else x.shape[1]
    if x is not None:
        _need_cuda(x); x = _f32(x)
    y = torch.empty((B, Cc + A) + tuple(eps.shape[2:]), device=eps.device, dtype=eps.dtype)
    ldj = torch.empty(B, device=eps.device, dtype=eps.dtype)
    _call('augment_fwd', (_p(x), _p(eps), _p(y), _p(ldj), B, Cc, A, HW, _stream()), 'augment_fwd')
    return y, ldj


def prologue(x, u, eps, s0, t0, s1, t1, ldj_const):
    _need_cuda(x, u, eps); x = _f32(x); u = _f32(u)
    B, Cc, H, W = x.shape
    A = 0 if eps is None else eps.shape[1]
    if eps is not None:
        eps = _f32(eps)
    y = torch.empty((B, Cc + A, H, W), device=x.device, dtype=x.dtype)
    ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    _set_work(bytes=4.0 * (2 * x.numel() + (0 if eps is None else eps.numel()) + y.numel()))
    _call('prologue_fwd', (_p(x), _p(u), _p(eps), _p(y), _p(ldj), B, Cc, A, H * W, s0, t0, s1, t1, ldj_const, _stream()), 'prologue_fwd')
    return y, ldj


# ---------------------------------------------------------------------------------------------- 1x1 conv / actnorm
def slogdet(A):
    _need_cuda(A); A = _f32(A)
    out = torch.empty(1, device=A.device, dtype=A.dtype)
    _call('slogdet', (_p(A), A.shape[0], _p(out), _stream()), 'slogdet')
    return out


def conv1x1(x, NN, logabsdet, c=None, logp_c=None, contextflow=False, an_t=None, an_logs=None, an_logp_c=None, an_logp_scale=0.0):
    _need_cuda(x, NN); x = _f32(x)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    z = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    if an_t is not None and an_logs is None:                      # one (B, 2D) 'b (p d)' matrix: [t | logs] per sample
        per_sample, an_logs = 2, an_t[:, D:]
    else:
        per_sample = int(an_t is not None and an_t.dim() == 2)
    _set_work(bytes=8.0 * x.numel() + (0 if c is None else 4.0 * c.numel()), flops=2.0 * D * x.numel(), shape=f'D{D}xHW{HW}')
    _call('conv1x1_fwd', (_p(x), _p(z), _p(ldj), _p(_f32(NN)), _p(logabsdet), _p(None if c is None else _f32(c)),
                                 _p(logp_c), int(bool(contextflow)), _p(an_t), _p(an_logs), per_sample, _p(an_logp_c),
                                 float(an_logp_scale), B, D, HW, _stream()), 'conv1x1_fwd')
    return z, ldj


def conv1x1_ctx_supported(B, D, HW, K) -> bool:
    return bool(lib().cfpp_conv1x1_ctx_supported(int(B), int(D), int(HW), int(K)))


def pack_cn_tril(weight, bias, D):
    """Conv1x1.CN (nn.Linear(C, D*D), conv1x1.py:22) restricted to the entries torch.tril keeps, K-major over the packed triangle:
    -> (cnw_tri (K, T), cnb_tri (T)), T = D(D+1)/2, entry t = i(i+1)/2 + j <-> output row i*D + j (one-time weight prep)."""
    ii, jj = torch.tril_indices(D, D, device=weight.device)
    rows = ii * D + jj                                               # row-major lower triangle: i ascending, j <= i ascending
    return weight.detach().to(torch.float32)[rows].t().contiguous(), bias.detach().to(torch.float32)[rows].contiguous()


def conv1x1_ctx(x, e, cnw_tri, cnb_tri, NN, logabsdet, logp_c=None, contextflow=False, an_t=None, an_logs=None, an_logp_c=None, an_logp_scale=0.0):
    """Conv1x1 with its context network and the ActNorm epilogue in one kernel (cfpp_conv1x1_ctx_fwd)."""
    _need_cuda(x, e, cnw_tri); x = _f32(x); e = _f32(e)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    z = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    per_sample = 0
    if an_t is not None:
        if an_logs is None:
            per_sample, an_logs = 2, an_t[:, D:]
        else:
            per_sample = 1
    K, T = cnw_tri.shape
    _set_work(bytes=8.0 * x.numel() + 4.0 * e.numel(), flops=2.0 * D * x.numel() + 2.0 * B * K * T, shape=f'D{D}xHW{HW}')
    _call('conv1x1_ctx_fwd', (_p(x), _p(z), _p(ldj), _p(e), _p(cnw_tri), _p(cnb_tri), _p(_f32(NN)), _p(logabsdet), _p(logp_c),
                              int(bool(contextflow)), _p(an_t), _p(an_logs), per_sample, _p(an_logp_c), float(an_logp_scale),
                              B, D, HW, K, _stream()), 'conv1x1_fwd')
    return z, ldj


def actnorm(x, base_t, base_logs, c=None, logp_c=None, logp_scale=0.0, mode=0):
    _need_cuda(x); x = _f32(x)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    z = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    _set_work(bytes=8.0 * x.numel())
    _call('actnorm_fwd', (_p(x), _p(z), _p(ldj), _p(base_t), _p(base_logs), _p(None if c is None else _f32(c)), _p(logp_c),
                                 float(logp_scale), mode, B, D, HW, _stream()), 'actnorm_fwd')
    return z, ldj


def actnorm_stats(x):
    _need_cuda(x); x = _f32(x)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel()
    mean = torch.empty(D, device=x.device, dtype=x.dtype); logstd = torch.empty_like(mean)
    _call('actnorm_stats', (_p(x), _p(mean), _p(logstd), B, D, HW, _stream()), 'actnorm_stats')
    return mean, logstd


# ---------------------------------------------------------------------------------------------- coupling
def coupling(x, h, add=None, logp_c=None, logp_scale=0.0):
    _need_cuda(x, h); x = _f32(x); h = _f32(h)
    B, Cc = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    z = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    _set_work(bytes=12.0 * x.numel(), shape=f'C{Cc}xHW{HW}')
    _call('coupling_fwd', (_p(x), _p(h), _p(None if add is None else _f32(add)), _p(logp_c), float(logp_scale),
                                  _p(z), _p(ldj), B, Cc, HW, _stream()), 'coupling_fwd')
    return z, ldj


def coupling_inv(z, h, add=None):
    """Coupling.reverse core (coupling.py:68-73): x = cat(z0, (z1 - t) / s)."""
    _need_cuda(z, h); z = _f32(z); h = _f32(h)
    B, Cc = z.shape[0], z.shape[1]
    HW = z[0, 0].numel() if B else 1
    x = torch.empty_like(z)
    _set_work(bytes=12.0 * z.numel())
    _call('coupling_inv', (_p(z), _p(h), _p(None if add is None else _f32(add)), _p(x), B, Cc, HW, _stream()), 'coupling_inv')
    return x


# ---------------------------------------------------------------------------------------------- inverse direction
def actnorm_inv(z, t, logs):
    _need_cuda(z, t, logs); z = _f32(z)
    B, D = z.shape[0], z.shape[1]
    HW = z[0, 0].numel() if B else 1
    x = torch.empty_like(z)
    _set_work(bytes=8.0 * z.numel())
    _call('actnorm_inv', (_p(z), _p(x), _p(_f32(t)), _p(_f32(logs)), B, D, HW, _stream()), 'actnorm_inv')
    return x


def mat_inverse(A):
    """torch.inverse(NN) (conv1x1.py:70): returns (Ainv, singular flag as a device int tensor)."""
    _need_cuda(A); A = _f32(A)
    out = torch.empty_like(A); flag = torch.empty(1, device=A.device, dtype=torch.int32)
    _call('mat_inverse', (_p(A), A.shape[0], _p(out), _p(flag), _stream()), 'mat_inverse')
    return out, flag


def sigmoid(x):
    _need_cuda(x); x = _f32(x)
    y = torch.empty_like(x)
    _call('sigmoid_fwd', (_p(x), _p(y), x.numel(), _stream()), 'sigmoid_fwd')
    return y


def normalize_inv(y, scale: float, translation: float):
    _need_cuda(y); y = _f32(y)
    x = torch.empty_like(y)
    _call('normalize_inv', (_p(y), _p(x), y.numel(), float(scale), float(translation), _stream()), 'normalize_inv')
    return x


def floor(x):
    _need_cuda(x); x = _f32(x)
    y = torch.empty_like(x)
    _call('floor_fwd', (_p(x), _p(y), x.numel(), _stream()), 'floor_fwd')
    return y


def prologue_inv(z, C, s1, t1, s0, t0, do_floor=True, keep_cont=False):
    """Augment / Logit / Normalization x2 / Dequantization reverses in one pass; z is (B, C + A, H, W)."""
    _need_cuda(z); z = _f32(z)
    B, CA, H, W = z.shape
    x = torch.empty((B, C, H, W), device=z.device, dtype=z.dtype)
    cont = torch.empty_like(x) if keep_cont else None
    _set_work(bytes=8.0 * x.numel())
    _call('prologue_inv', (_p(z), _p(x), _p(cont), B, C, CA - C, H * W, float(s1), float(t1), float(s0), float(t0),
                           int(bool(do_floor)), _stream()), 'prologue_inv')
    return (x, cont) if keep_cont else x


def gmm_sample(mG, sG, comp, eps, m=1):
    """x[b] = mG[m, comp[b]] + softplus(sG[m, comp[b]]) * eps[b]  (gaussian.py:163-166 after its draws)."""
    _need_cuda(mG, sG, comp, eps); eps = _f32(eps)
    if comp.dtype != torch.int64:
        raise TypeError('component indices must be int64')
    M, K = mG.shape[0], mG.shape[1]
    B = eps.shape[0]
    n = mG[0, 0].numel()
    x = torch.empty_like(eps)
    _call('gmm_sample', (_p(_f32(mG)), _p(_f32(sG)), _p(comp.contiguous()), _p(eps), _p(x), B, M, K, n, int(m), _stream()), 'gmm_sample')
    return x


# ---------------------------------------------------------------------------------------------- loss / score epilogue
def score_epilogue(logp, dim_inv, gt=None, class_w=None, want=('scaled', 'lse', 'softmax1', 'last', 'argmax')):
    """experiment_ad.py:204-211,262-281 / experiment_cl.py:127-133,185-204 after log_prob, two launches.  Returns a dict with the
    requested per-sample outputs and 'sums' (4,) = [sum logsigmoid(lse), sum logsigmoid(scaled), CE numerator, CE denominator]."""
    _need_cuda(logp); logp = _f32(logp)
    B, M = logp.shape
    dev = logp.device
    out = {}
    if 'scaled' in want: out['scaled'] = torch.empty_like(logp)
    for k in ('lse', 'softmax1', 'last'):
        if k in want: out[k] = torch.empty(B, device=dev, dtype=torch.float32)
    if 'argmax' in want: out['argmax'] = torch.empty(B, device=dev, dtype=torch.int64)
    out['sums'] = torch.empty(4, device=dev, dtype=torch.float32)
    ws = torch.empty(int(lib().cfpp_score_workspace_bytes(B)), device=dev, dtype=torch.uint8)
    if gt is not None:
        _need_cuda(gt)
        if gt.dtype != torch.int64:
            raise TypeError('gt must be int64 class indices')
        gt = gt.contiguous()
    _set_work(bytes=4.0 * logp.numel() * (2 if 'scaled' in want else 1))
    _call('score_epilogue', (_p(logp), float(dim_inv), _p(gt), _p(None if class_w is None else _f32(class_w)),
                             _p(out.get('scaled')), _p(out.get('lse')), _p(out.get('softmax1')), _p(out.get('last')),
                             _p(out.get('argmax')), _p(out['sums']), _p(ws), B, M, _stream()), 'score_epilogue')
    return out


def pack_kmajor(w2d: torch.Tensor, pad_to: int = 16) -> torch.Tensor:
    """(N, K) weight -> K-major (K, NP) with the output dim zero-padded to a multiple of `pad_to` (one-time weight prep)."""
    N, K = w2d.shape
    NP = (N + pad_to - 1) // pad_to * pad_to
    out = torch.zeros((K, NP), device=w2d.device, dtype=torch.float32)
    out[:, :N] = w2d.detach().t().to(torch.float32)
    return out


def pad_vec(v: torch.Tensor, pad_to: int = 16) -> torch.Tensor:
    N = v.shape[0]
    NP = (N + pad_to - 1) // pad_to * pad_to
    out = torch.zeros(NP, device=v.device, dtype=torch.float32)
    out[:N] = v.detach().to(torch.float32)
    return out


def conv_cond(x, cin, packed, H, W, KH, KW, cout, bias1_b=None):
    """packed = (w1t, b1, w2t, b2, w3t, b3) from pack_kmajor/pad_vec; reads the first `cin` channels of x in place."""
    _need_cuda(x)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    w1t, b1, w2t, b2, w3t, b3 = packed
    ch = w2t.shape[0] // (KH * KW)
    h = torch.empty((B, cout, H, W), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * H * W * (cin + cout), flops=2.0 * B * H * W * (cin * ch + ch * ch * KH * KW + ch * cout))
    _call('conv_cond_fwd', (_p(xv), bstride, _p(h), _p(w1t), _p(b1), _p(None if bias1_b is None else _f32(bias1_b)),
                                   _p(w2t), _p(b2), _p(w3t), _p(b3), B, cin, ch, cout, H, W, KH, KW, _stream()), 'conv_cond_fwd')
    return h


CONV_COND_FUSED_MAX_BATCH = 4096     # B200, cfg2: fused 0.682 / 1.207 / 1.811 ms per step at B = 256 / 1024 / 2048 against 0.706 / 1.230 / 1.818 split; 5.73 against 5.66 at 8192


def conv_cond_tc_mode() -> str:
    """'auto' (tensor cores whenever the shape has a plan; below CONV_COND_FUSED_MAX_BATCH samples the conditioner and the coupling transform
    run as ONE kernel, so h never reaches HBM and a launch is saved -- measured faster there; above it the two-kernel route is ~1 % ahead),
    'fused' / 'split' (force either), 'fma' (force the FP32-FMA conditioner) -- env CFPP_CONV_COND."""
    import os
    return os.environ.get('CFPP_CONV_COND', 'auto')


def conv_cond_tc_pack(w1, w2, w3, cin):
    """Repack torch-layout conditioner weights for cfpp_conv_cond_tc_fwd; None when the channel counts have no tensor-core plan."""
    _need_cuda(w1, w2, w3)
    ch, cout, KH, KW = w2.shape[0], w3.shape[0], w2.shape[2], w2.shape[3]
    nbytes = int(lib().cfpp_conv_cond_tc_pack_bytes(cin, ch, cout, KH, KW))
    if nbytes < 0:
        return None
    w1 = _f32(w1.detach().reshape(ch, -1)); w2 = _f32(w2.detach()); w3 = _f32(w3.detach().reshape(cout, -1))
    out = torch.empty(nbytes, device=w2.device, dtype=torch.uint8)
    _call('conv_cond_tc_pack', (_p(w1), w1.shape[1], _p(w2), _p(w3), _p(out), cin, ch, cout, KH, KW, _stream()))
    return out


def conv_cond_tc(x, cin, wpack, b1, b2, b3, ch, H, W, KH, KW, cout, bias1_b=None):
    """Tensor-core conditioner; returns None (nothing launched) when this shape has no plan so the caller can use conv_cond."""
    _need_cuda(x, wpack)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    if not lib().cfpp_conv_cond_tc_supported(B, cin, ch, cout, H, W, KH, KW, bstride) or xv.data_ptr() % 16:
        return None
    h = torch.empty((B, cout, H, W), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * H * W * (cin + cout), flops=2.0 * B * H * W * (cin * ch + ch * ch * KH * KW + ch * cout), shape=f'Ch{ch}x{H}x{W}')
    _call('conv_cond_tc_fwd', (_p(xv), bstride, _p(h), _p(wpack), _p(b1), _p(None if bias1_b is None else _f32(bias1_b)), _p(b2), _p(b3),
                               B, cin, ch, cout, H, W, KH, KW, _stream()))
    return h


def conv_cond_tc_train(x, cin, wpack, b1, b2, b3, ch, H, W, KH, KW, cout, bias1_b=None):
    """Training forward of the tensor-core conditioner: (h, a1, a2) with the post-ReLU activations the backward pass reads, or None
    (nothing launched) when this shape has no plan."""
    _need_cuda(x, wpack)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    if x.dtype != torch.float32 or not lib().cfpp_conv_cond_tc_supported(B, cin, ch, cout, H, W, KH, KW, bstride) or xv.data_ptr() % 16:
        return None
    h = torch.empty((B, cout, H, W), device=x.device, dtype=torch.float32)
    a1 = torch.empty((B, ch, H, W), device=x.device, dtype=torch.float32)
    a2 = torch.empty((B, ch, H, W), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * H * W * (cin + cout + 2 * ch), flops=2.0 * B * H * W * (cin * ch + ch * ch * KH * KW + ch * cout), shape=f'Ch{ch}x{H}x{W}')
    _call('conv_cond_tc_train_fwd', (_p(xv), bstride, _p(h), _p(a1), _p(a2), _p(wpack), _p(b1), _p(None if bias1_b is None else _f32(bias1_b)), _p(b2), _p(b3),
                                     B, cin, ch, cout, H, W, KH, KW, _stream()))
    return h, a1, a2


def conv_cond_tc_coupling(x, wpack, b1, b2, b3, ch, KH, KW, add=None, logp_c=None, logp_scale=0.0, bias1_b=None):
    """Conditioner + affine coupling in one kernel: (z, ldj), or None (nothing launched) when the shape has no fused plan."""
    _need_cuda(x, wpack)
    if x.dtype != torch.float32 or not x.is_contiguous() or x.data_ptr() % 16:
        return None
    B, Cc, H, W = x.shape
    if Cc % 16 or not lib().cfpp_conv_cond_tc_coupling_supported(B, Cc, ch, H, W, KH, KW):
        return None
    z = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=torch.float32)
    cin = Cc // 2
    _set_work(bytes=8.0 * x.numel(), flops=2.0 * B * H * W * (cin * ch + ch * ch * KH * KW + ch * Cc), shape=f'Ch{ch}x{H}x{W}')
    _call('conv_cond_tc_coupling_fwd', (_p(x), _p(z), _p(ldj), _p(wpack), _p(b1), _p(None if bias1_b is None else _f32(bias1_b)), _p(b2), _p(b3),
                                        _p(None if add is None else _f32(add)), _p(logp_c), float(logp_scale), B, Cc, ch, H, W, KH, KW, _stream()))
    return z, ldj


def conv_cond_tc_last_plan():
    out = (_cabi.i32 * 12)()
    lib().cfpp_conv_cond_tc_last_plan(out)
    return dict(zip(('seg', 'S', 'R', 'T1', 'T2', 'nstages', 'smem_bytes', 'ntiles', 'occ', 'row_bytes', 'pipe'), list(out)))


def vit_cond(x, desc: _cabi.VitDesc, cout, extra=None):
    _need_cuda(x)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    h = torch.empty((B, cout, desc.H, desc.W), device=x.device, dtype=torch.float32)
    cextra = 0 if extra is None else extra.shape[1]
    _set_work(bytes=4.0 * B * desc.H * desc.W * (desc.Cin + cout), flops=2.0 * B * desc.n_tok * (desc.patch_dim * desc.T + desc.depth * (desc.T * 192 + 2 * desc.n_tok * 64 + 64 * desc.T + 2 * desc.T * desc.T)))
    _call('vit_cond_fwd', (_p(xv), bstride, _p(None if extra is None else _f32(extra)), cextra, _p(h), C.byref(desc), B, _stream()),
          'vit_cond_fwd')
    return h


def vit_tc_pack(mats):
    """mats: [(weight (out, in) row-major, n_rows, k_cols)] in chunk order -> packed fp16 hi/lo weight stream of cfpp_vit_tc_fwd."""
    _need_cuda(*[m[0] for m in mats])
    chunk = int(lib().cfpp_vit_tc_pack_bytes(0))
    out = torch.empty(chunk * len(mats), device=mats[0][0].device, dtype=torch.uint8)
    keep = []
    for i, (w, n_rows, k_cols) in enumerate(mats):
        w = _f32(w.detach()); keep.append(w)
        _call('vit_tc_pack_chunk', (_p(w), w.stride(0), n_rows, k_cols, vp(out.data_ptr() + i * chunk), _stream()))
    return out


def vit_cond_tc(x, desc: _cabi.VitDesc, wpack, cout, general=False):
    """general=False: cfpp_vit_tc_fwd (T <= 64, residual stream in registers); True: cfpp_vit_tc2_fwd (T <= 192, any token count)."""
    _need_cuda(x, wpack)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    h = torch.empty((B, cout, desc.H, desc.W), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * desc.H * desc.W * (desc.Cin + cout), flops=2.0 * B * desc.n_tok * (desc.patch_dim * desc.T + desc.depth * (desc.T * 192 + 2 * desc.n_tok * 64 + 64 * desc.T + 2 * desc.T * desc.T)))
    _call('vit_tc2_fwd' if general else 'vit_tc_fwd', (_p(xv), bstride, _p(h), C.byref(desc), _p(wpack), B, _stream()), 'vit_cond_tc_fwd')
    return h


# ---------------------------------------------------------------------------------------------- GMM
def gmm_logprob(x, mG, sG, wG, ctx_off=None, logp_c=None, logp_scale=0.0):
    _need_cuda(x, mG)
    M, K, D = mG.shape[0], mG.shape[1], mG.shape[2]
    xv, bstride = _half_view(x)
    B = x.shape[0]
    HW = x.shape[2] * x.shape[3]
    out = torch.empty((B, M), device=x.device, dtype=torch.float32)
    ws = torch.empty(int(lib().cfpp_gmm_workspace_floats(M, K, D, HW)), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * D * HW + 4.0 * B * M, flops=3.0 * B * M * K * D * HW)
    _call('gmm_logprob', (_p(xv), bstride, _p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(None if ctx_off is None else _f32(ctx_off)),
                                 _p(logp_c), float(logp_scale), _p(out), _p(ws), B, M, K, D, HW, _stream()), 'gmm_logprob')
    return out


def gmm_logprob_ctxtab(x, mG, sG, wG, ctx, cards, tables, logp_scale=0.0, keep=None):
    """GMM log-prob with embedding-lookup context offsets (bucketed per-context tables); None if the structure is unsupported.
    keep: a dict the caller holds per parameter version -- the workspace then lives in it and its parameter-only tables are computed once."""
    _need_cuda(x, mG, ctx)
    M, K, D = mG.shape[0], mG.shape[1], mG.shape[2]
    xv, bstride = _half_view(x)
    B, HW, n = x.shape[0], x.shape[2] * x.shape[3], len(cards)
    carr = (_cabi.i32 * n)(*cards)
    need = int(lib().cfpp_gmm_ctxtab_workspace_bytes(B, M, K, D, HW, n, carr))
    if need < 0:
        return None
    out = torch.empty((B, M), device=x.device, dtype=torch.float32)
    ready = 0
    if keep is not None:
        ent = keep.get((B, x.device))
        if ent is None or ent.numel() != need:
            ent = keep[(B, x.device)] = torch.empty(need, device=x.device, dtype=torch.uint8)
        else:
            ready = 1
        ws = ent
    else:
        ws = torch.empty(need, device=x.device, dtype=torch.uint8)
    tabs = [_f32(t) for t in tables]
    tarr = (vp * n)(*[vp(t.data_ptr()) for t in tabs])
    _set_work(bytes=4.0 * B * D * HW + 4.0 * B * M, flops=3.0 * B * M * K * D * HW)
    _call('gmm_logprob_ctxtab_cached', (_p(xv), bstride, _p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(ctx.contiguous()), n, carr, tarr,
                                        tabs[0].shape[1], None, float(logp_scale), _p(out), _p(ws), need, ready, B, M, K, D, HW, _stream()),
          'gmm_logprob_ctxtab')
    return out


def gmm_tile_table(mG, sG, wG, scale_table=None, scale_off=0):
    """(mu, 1/(2 sigma^2)) table of cfpp_gmm_tile_logprob, one per row of scale_table; None when the sizes are unsupported.
    A function of the parameters only: callers cache it per parameter version."""
    _need_cuda(mG, sG, wG, scale_table)
    M, K, D = mG.shape[0], mG.shape[1], mG.shape[2]
    HW = mG.shape[3] * mG.shape[4]
    nv = 1 if scale_table is None else scale_table.shape[0]
    nbytes = int(lib().cfpp_gmm_tile_table_bytes(M, K, D, HW, nv))
    if nbytes < 0:
        return None
    tab = torch.empty(nbytes, device=mG.device, dtype=torch.uint8)
    st = None if scale_table is None else _f32(scale_table)
    _call('gmm_tile_prepare', (_p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(st), 0 if st is None else st.shape[1], int(scale_off), nv,
                               _p(tab), M, K, D, HW, _stream()))
    return tab


def gmm_tile_logprob(x, table, M, K, ctx=None, cards=(), mean_table=None, mean_off=0, logp_c=None, logp_scale=0.0):
    """cards: cardinalities of the 0, 1 or 2 context features; the table must hold cards[-1] scale contexts (1 without context)."""
    _need_cuda(x, table, ctx, mean_table)
    xv, bstride = _half_view(x)
    B, D, HW = x.shape[0], x.shape[1], x.shape[2] * x.shape[3]
    n = len(cards)
    n_keys = 1
    for c in cards:
        n_keys *= int(c)
    out = torch.empty((B, M), device=x.device, dtype=torch.float32)
    need = int(lib().cfpp_gmm_tile_workspace_bytes(B, M, K, D, HW, n_keys))
    if need < 0:
        raise RuntimeError(f'gmm_tile_logprob: {n_keys} context tuples unsupported')
    ws = torch.empty(max(need, 1), device=x.device, dtype=torch.uint8)
    mt = None if mean_table is None else _f32(mean_table)
    carr = (_cabi.i32 * max(n, 1))(*[int(c) for c in cards])
    _set_work(bytes=4.0 * B * D * HW + 4.0 * B * M, flops=3.0 * B * M * K * D * HW, shape=f'D{D}xHW{HW}xK{n_keys}')
    _call('gmm_tile_logprob', (_p(xv), bstride, _p(table), _p(None if ctx is None else ctx.contiguous()), n, carr,
                               _p(mt), 0 if mt is None else mt.shape[1], int(mean_off), _p(logp_c), float(logp_scale),
                               _p(out), _p(ws), need, B, M, K, D, HW, _stream()))
    return out


# ---------------------------------------------------------------------------------------------- context
def embed_lookup(ctx, tables: Sequence[torch.Tensor]):
    _need_cuda(ctx, *tables)
    B, n = ctx.shape
    width = tables[0].shape[1]
    out = torch.empty((B, n * width), device=ctx.device, dtype=torch.float32)
    arr = (vp * n)(*[vp(_f32(t).data_ptr()) for t in tables])
    _call('embed_lookup', (_p(ctx.contiguous()), arr, n, width, _p(out), B, _stream()), 'embed_lookup')
    return out


def ctx_encode(ctx, noise, desc: _cabi.EncDesc, emit_stage=-1):
    _need_cuda(ctx, noise)
    B = ctx.shape[0]
    c = torch.empty((B, desc.C), device=ctx.device, dtype=torch.float32)
    logp = torch.empty(B, device=ctx.device, dtype=torch.float32)
    _call('ctx_encode', (_p(ctx.contiguous()), _p(None if noise is None else _f32(noise)), _p(c), _p(logp), C.byref(desc),
                                emit_stage, B, _stream()), 'ctx_encode')
    return c, logp


def _carve(B, widths, device, align=64):
    """(B, w_i) fp32 matrices carved out of one allocation, each starting on a 256-byte boundary (consumers use 128-bit loads)."""
    sizes = [(B * w + align - 1) // align * align for w in widths]
    flat = torch.empty(sum(sizes), device=device, dtype=torch.float32)
    outs, off = [], 0
    for w, sz in zip(widths, sizes):
        outs.append(flat[off: off + B * w].view(B, w)); off += sz
    return outs


def ctx_encode_batch(ctx, descs_dev, noises, widths, flow_width=0):
    """n encoders over one context batch in a single launch; returns ([c_i (B, width_i)], [logp_i (B,)]).
    flow_width = C when every encoder carries the inner flow at that width (the tiled kernel is used where it exists)."""
    _need_cuda(ctx, descs_dev)
    B, n = ctx.shape[0], len(widths)
    logp_all = torch.empty((n, B), device=ctx.device, dtype=torch.float32)
    cs = _carve(B, widths, ctx.device)
    arr = lambda ts: (vp * n)(*[vp(0 if t is None else t.data_ptr()) for t in ts])
    noises = [None if t is None else _f32(t) for t in noises]
    if flow_width and lib().cfpp_ctx_encode_flow_supported(int(flow_width)):
        _call('ctx_encode_batch_flow', (_p(ctx.contiguous()), _p(descs_dev), n, int(flow_width), arr(noises), arr(cs), arr(list(logp_all)), B, _stream()))
    else:
        _call('ctx_encode_batch', (_p(ctx.contiguous()), _p(descs_dev), n, arr(noises), arr(cs), arr(list(logp_all)), B, _stream()))
    return cs, list(logp_all)


def linear(x, wt, b=None, relu=False, n_out=None):
    """y = act(x @ wt + b); wt is K-major (K, N) (possibly column-padded: pass n_out to trim)."""
    _need_cuda(x, wt); x = _f32(x)
    B, K = x.shape
    N = wt.shape[1]
    y = torch.empty((B, N), device=x.device, dtype=torch.float32)
    _call('linear_fwd', (_p(x), _p(wt), _p(b), _p(y), B, K, N, int(relu), _stream()), 'linear_fwd')
    return y if n_out is None or n_out == N else y[:, :n_out]


def cn_job(layers, tril_dim=0):
    """Descriptor of one CN chain: layers = [(wt K-major (K, N), bias (N) or None), ...] (1..3 entries, ReLU between).
    Returns (CnJob, keep-alive list)."""
    j = _cabi.CnJob()
    j.n_layers, j.K, j.tril_dim = len(layers), layers[0][0].shape[0], tril_dim
    keep = []
    for l, (wt, b) in enumerate(layers):
        wt = _f32(wt); keep.append(wt)
        j.w[l], j.N[l] = vp(wt.data_ptr()), wt.shape[1]
        if b is not None:
            b = _f32(b); keep.append(b); j.b[l] = vp(b.data_ptr())
    return j, keep


def cn_batch(jobs, ins):
    """All CN context networks of a forward in one launch: jobs[i] (cn_job descriptors) applied to ins[i] (B, K_i)."""
    _need_cuda(*ins)
    n, B = len(jobs), ins[0].shape[0]
    widths = [int(j.N[j.n_layers - 1]) for j in jobs]
    outs = _carve(B, widths, ins[0].device)
    ins = [_f32(t) for t in ins]
    for i0 in range(0, n, _cabi.MAX_CN_JOBS):
        m = min(_cabi.MAX_CN_JOBS, n - i0)
        jarr = (_cabi.CnJob * m)(*jobs[i0: i0 + m])
        iarr = (vp * m)(*[vp(t.data_ptr()) for t in ins[i0: i0 + m]])
        oarr = (vp * m)(*[vp(t.data_ptr()) for t in outs[i0: i0 + m]])
        _call('cn_batch', (jarr, m, iarr, oarr, B, _stream()))
    return outs


def ldj_accumulate(logdet, ldj):
    _need_cuda(logdet, ldj)
    B, M = logdet.shape
    cols = 1 if ldj.dim() == 1 else ldj.shape[1]
    _call('ldj_accumulate', (_p(logdet), _p(_f32(ldj)), B, M, cols, _stream()), 'ldj_accumulate')
    return logdet


LDJ_SUM_MAX = 64


def ldj_sum(terms, B, M, device, last=None):
    """logdet (B,M) = ((0 + t_0) + t_1) + ... [then last + logdet], in order, one launch per 64 terms."""
    _need_cuda(*terms)
    out = torch.empty((B, M), device=device, dtype=torch.float32)
    terms = [_f32(t) for t in terms]
    first = None
    for k0 in range(0, max(len(terms), 1), LDJ_SUM_MAX):
        chunk = terms[k0: k0 + LDJ_SUM_MAX]
        n = len(chunk)
        final = k0 + LDJ_SUM_MAX >= len(terms)
        parr = (vp * max(n, 1))(*[vp(t.data_ptr()) for t in chunk])
        carr = (_cabi.i32 * max(n, 1))(*[1 if t.dim() == 1 else t.shape[1] for t in chunk])
        _call('ldj_sum', (_p(out), _p(first), _p(last if final else None), parr, carr, n, B, M, _stream()))
        first = out
    return out


# ---------------------------------------------------------------------------------------------- training direction (SURVEY §8f-1)
def coupling_bwd(x, h, dz, dldj=None, add=None):
    _need_cuda(x, h, dz); x = _f32(x); h = _f32(h); dz = _f32(dz)
    B, Cc = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    dx = torch.empty_like(x); dh = torch.empty_like(h)
    _set_work(bytes=20.0 * x.numel())
    _call('coupling_bwd', (_p(x), _p(h), _p(None if add is None else _f32(add)), _p(dz), _p(None if dldj is None else _f32(dldj)), _p(dx), _p(dh),
                           B, Cc, HW, _stream()))
    return dx, dh


def actnorm_bwd(x, dz, dldj, t, logs, need_dx=True):
    _need_cuda(x, dz); x = _f32(x); dz = _f32(dz)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel()
    dx = torch.empty_like(x) if need_dx else None
    dt = torch.empty(D, device=x.device, dtype=torch.float32); dlogs = torch.empty_like(dt)
    ws = torch.empty(int(lib().cfpp_actnorm_bwd_workspace_floats(B, D)), device=x.device, dtype=torch.float32)
    _set_work(bytes=(12.0 if need_dx else 8.0) * x.numel())
    _call('actnorm_bwd', (_p(x), _p(dz), _p(None if dldj is None else _f32(dldj)), _p(_f32(t)), _p(_f32(logs)), _p(dx), _p(dt), _p(dlogs),
                          _p(ws), B, D, HW, _stream()))
    return dx, dt, dlogs


def relu(x):
    _need_cuda(x); x = _f32(x)
    y = torch.empty_like(x)
    _set_work(bytes=8.0 * x.numel())
    _call('relu_fwd', (_p(x), _p(y), x.numel(), _stream()))
    return y


def maf_coupling(x, h, add=None, logp_c=None, logp_scale=0.0):
    """MaskedCoupling elementwise part (ar.py:35-57): h (B, 2C, H, W) without the identity; add (B, 2C) = CN(c) of a --contextflow
    specialist, ldj += logp_scale * logp_c."""
    _need_cuda(x, h, add, logp_c); x = _f32(x); h = _f32(h)
    B, Cc = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    z = torch.empty_like(x); ldj = torch.empty(B, device=x.device, dtype=x.dtype)
    _set_work(bytes=16.0 * x.numel())
    _call('maf_coupling_ctx_fwd', (_p(x), _p(h), _p(None if add is None else _f32(add)), _p(None if logp_c is None else _f32(logp_c)), float(logp_scale),
                                   _p(z), _p(ldj), B, Cc, HW, _stream()))
    return z, ldj


def relu_mask_(g, act):
    """g[i] = 0 where act[i] <= 0, in place (ReLU backward on the saved post-activation)."""
    _need_cuda(g, act)
    _call('relu_mask', (_p(g), _p(_f32(act)), g.numel(), _stream()))
    return g


def maf_coupling_bwd(x, h, dz, dldj=None):
    _need_cuda(x, h, dz); x = _f32(x); h = _f32(h); dz = _f32(dz)
    B, Cc = x.shape[0], x.shape[1]
    HW = x[0, 0].numel() if B else 1
    dx = torch.empty_like(x); dh = torch.empty_like(h)
    _set_work(bytes=24.0 * x.numel())
    _call('maf_coupling_bwd', (_p(x), _p(h), _p(dz), _p(None if dldj is None else _f32(dldj)), _p(dx), _p(dh), B, Cc, HW, _stream()))
    return dx, dh


def conv2d_fwd(x, cin, w, b, relu, relu_in=False):
    """out = [relu](conv([relu_in](x[:, :cin])) + b), 'same' reflect padding; x may be wider than cin channels (read through its batch stride)."""
    _need_cuda(x, w)
    xv, bstride = _half_view(x[:, :cin])
    B, H, W = x.shape[0], x.shape[2], x.shape[3]
    cout, KH, KW = w.shape[0], w.shape[2], w.shape[3]
    out = torch.empty((B, cout, H, W), device=x.device, dtype=torch.float32)
    _set_work(flops=2.0 * B * cout * cin * KH * KW * H * W)
    _call('conv2d_fwd', (_p(xv), bstride, _p(_f32(w)), _p(None if b is None else _f32(b)), _p(out), B, cin, cout, H, W, KH, KW,
                         int(bool(relu)) | (2 if relu_in else 0), _stream()))
    return out


def conv2d_bwd_data(dout, w, act=None, out=None, accumulate=False):
    """Gradient w.r.t. the convolution's input; `out` (B, >=Cin, H, W) may be a wider tensor whose first Cin channels receive (+)= it."""
    _need_cuda(dout, w); dout = _f32(dout)
    B, cout, H, W = dout.shape
    cin, KH, KW = w.shape[1], w.shape[2], w.shape[3]
    if out is None:
        out = torch.empty((B, cin, H, W), device=dout.device, dtype=torch.float32)
    ov, ostride = _half_view(out[:, :cin])
    assert ov.data_ptr() == out.data_ptr(), 'conv2d_bwd_data: output view must alias the given tensor'
    av, astride = (None, 0) if act is None else _half_view(act[:, :cin])
    _set_work(flops=2.0 * B * cout * cin * KH * KW * H * W)
    _call('conv2d_bwd_data', (_p(dout), _p(_f32(w)), _p(av), astride, _p(ov), ostride, int(bool(accumulate)), B, cin, cout, H, W, KH, KW, _stream()))
    return out


def conv2d_bwd_weight(x, cin, dout, wshape, bias=True):
    _need_cuda(x, dout); dout = _f32(dout)
    xv, bstride = _half_view(x[:, :cin])
    B, cout, H, W = dout.shape
    KH, KW = wshape[2], wshape[3]
    dW = torch.empty(tuple(wshape), device=dout.device, dtype=torch.float32)
    db = torch.empty(cout, device=dout.device, dtype=torch.float32) if bias else None
    _set_work(flops=2.0 * B * cout * cin * KH * KW * H * W)
    ws = torch.empty(max(1, int(lib().cfpp_conv2d_bwd_weight_workspace_floats(B, cin, cout, KH, KW))), device=dout.device, dtype=torch.float32)
    _call('conv2d_bwd_weight', (_p(xv), bstride, _p(dout), _p(dW), _p(db), _p(ws), B, cin, cout, H, W, KH, KW, _stream()))
    return dW, db


def logdet_grad_(dNN, inv, dldj, HW):
    _need_cuda(dNN, inv, dldj)
    _call('logdet_grad', (_p(dNN), _p(_f32(inv)), _p(_f32(dldj)), dldj.shape[0], dNN.shape[0], int(HW), _stream()))
    return dNN


def rowsum(g):
    _need_cuda(g); g = _f32(g)
    B, M = g.shape
    out = torch.empty(B, device=g.device, dtype=torch.float32)
    _call('rowsum', (_p(g), _p(out), B, M, _stream()))
    return out


def gmm_train_prep(sG, wG):
    _need_cuda(sG, wG)
    M, K = wG.shape
    n = sG[0, 0].numel()
    inv_var = torch.empty((M, K, n), device=sG.device, dtype=torch.float32)
    cst = torch.empty((M, K), device=sG.device, dtype=torch.float32)
    _call('gmm_train_prep', (_p(_f32(sG)), _p(_f32(wG)), _p(inv_var), _p(cst), M, K, n, _stream()))
    return inv_var, cst


def gmm_train_fwd(x, mG, inv_var, cst):
    _need_cuda(x, mG)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    M, K, n = inv_var.shape
    logp = torch.empty((B, M), device=x.device, dtype=torch.float32)
    resp = torch.empty((B, M, K), device=x.device, dtype=torch.float32)
    _set_work(flops=3.0 * B * M * K * n)
    _call('gmm_train_fwd', (_p(xv), bstride, _p(_f32(mG)), _p(inv_var), _p(cst), _p(logp), _p(resp), B, M, K, n, _stream()))
    return logp, resp


def place_channels(src, dst, c0):
    """dst[:, c0:c0+Cn] = src (the adjoint of slice_channels)."""
    _need_cuda(src, dst); src = _f32(src)
    B, Cn, H, W = src.shape
    assert dst.is_contiguous() and dst.dtype == torch.float32
    _call('place_channels', (_p(src), _p(dst), B, dst.shape[1], H * W, int(c0), Cn, _stream()))
    return dst


def gmm_train_bwd(x, mG, sG, wG, inv_var, resp, g, need_dx=True, dx_out=None):
    """dx_out: optional (B, D, H, W) channel-slice view of a wider contiguous tensor that receives dx in place."""
    _need_cuda(x, mG, g); g = _f32(g)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    M, K, n = inv_var.shape
    if dx_out is not None:
        dv, dstride = _half_view(dx_out)
        assert dv.data_ptr() == dx_out.data_ptr(), 'gmm_train_bwd: dx_out must be a channel slice of a contiguous tensor'
        dx = dx_out
    else:
        dstride = n
        dx = torch.empty((B,) + tuple(x.shape[1:]), device=x.device, dtype=torch.float32) if need_dx else None
    dmG = torch.empty_like(mG, memory_format=torch.contiguous_format); dsG = torch.empty_like(dmG); dwG = torch.empty((M, K), device=x.device, dtype=torch.float32)
    ws = torch.empty(int(lib().cfpp_gmm_train_bwd_workspace_floats(B, M, K, n)), device=x.device, dtype=torch.float32)
    _set_work(flops=8.0 * B * M * K * n)
    _call('gmm_train_bwd', (_p(xv), bstride, _p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(inv_var), _p(resp), _p(g), _p(dx), dstride,
                            _p(dmG), _p(dsG), _p(dwG), _p(ws), B, M, K, n, _stream()))
    return dx, dmG, dsG, dwG


# ---------------------------------------------------------------------------------------------- ViT conditioner, training direction
def patchify(x, c, p1, p2):
    """(B, >=c, H, W) -> token rows (B * n_tok, p1*p2*c)  (simple_vit.py:102)."""
    _need_cuda(x)
    xv, bstride = _half_view(x[:, :c])
    B, H, W = x.shape[0], x.shape[2], x.shape[3]
    tok = torch.empty((B * (H // p1) * (W // p2), p1 * p2 * c), device=x.device, dtype=torch.float32)
    _call('patchify_fwd', (_p(xv), bstride, _p(tok), B, c, H, W, p1, p2, _stream()))
    return tok


def patchify_inv(tok, c, H, W, p1, p2, out=None, accumulate=False):
    """Token rows -> (B, c, H, W); with `out` (B, >=c, H, W) the first c channels receive (+)= it."""
    _need_cuda(tok); tok = _f32(tok)
    B = tok.shape[0] // ((H // p1) * (W // p2))
    if out is None:
        out = torch.empty((B, c, H, W), device=tok.device, dtype=torch.float32)
    ov, ostride = _half_view(out[:, :c])
    assert ov.data_ptr() == out.data_ptr()
    _call('patchify_inv', (_p(tok), _p(ov), ostride, int(bool(accumulate)), B, c, H, W, p1, p2, _stream()))
    return out


def layernorm_fwd(x, gamma, beta):
    _need_cuda(x); x = _f32(x)
    R, F = x.shape
    y = torch.empty_like(x); mean = torch.empty(R, device=x.device, dtype=torch.float32); rstd = torch.empty_like(mean)
    _set_work(bytes=8.0 * x.numel())
    _call('layernorm_fwd', (_p(x), _p(_f32(gamma)), _p(_f32(beta)), _p(y), _p(mean), _p(rstd), R, F, _stream()))
    return y, mean, rstd


def layernorm_bwd(x, dy, gamma, mean, rstd):
    _need_cuda(x, dy); x = _f32(x); dy = _f32(dy)
    R, F = x.shape
    dx = torch.empty_like(x); dg = torch.empty(F, device=x.device, dtype=torch.float32); db = torch.empty_like(dg)
    ws = torch.empty(int(lib().cfpp_layernorm_bwd_workspace_floats(R, F)), device=x.device, dtype=torch.float32)
    _set_work(bytes=12.0 * x.numel())
    _call('layernorm_bwd', (_p(x), _p(dy), _p(_f32(gamma)), _p(mean), _p(rstd), _p(dx), _p(dg), _p(db), _p(ws), R, F, _stream()))
    return dx, dg, db


def rows_linear(x, w, b=None):
    _need_cuda(x, w); x = _f32(x)
    R, I = x.shape
    J = w.shape[0]
    y = torch.empty((R, J), device=x.device, dtype=torch.float32)
    _set_work(flops=2.0 * R * I * J)
    _call('rows_linear_fwd', (_p(x), _p(_f32(w)), _p(None if b is None else _f32(b)), _p(y), R, I, J, _stream()))
    return y


def rows_linear_bwd_data(dy, w):
    _need_cuda(dy, w); dy = _f32(dy)
    R, J = dy.shape
    I = w.shape[1]
    dx = torch.empty((R, I), device=dy.device, dtype=torch.float32)
    _set_work(flops=2.0 * R * I * J)
    _call('rows_linear_bwd_data', (_p(dy), _p(_f32(w)), _p(dx), 0, R, I, J, _stream()))
    return dx


def rows_linear_bwd_weight(x, dy, bias=True):
    _need_cuda(x, dy); x = _f32(x); dy = _f32(dy)
    R, I = x.shape
    J = dy.shape[1]
    dW = torch.empty((J, I), device=x.device, dtype=torch.float32)
    db = torch.empty(J, device=x.device, dtype=torch.float32) if bias else None
    ws = torch.empty(int(lib().cfpp_rows_linear_bwd_weight_workspace_floats(R, I, J)), device=x.device, dtype=torch.float32)
    _set_work(flops=2.0 * R * I * J)
    _call('rows_linear_bwd_weight', (_p(x), _p(dy), _p(dW), _p(db), _p(ws), R, I, J, _stream()))
    return dW, db


def gelu_fwd(x):
    _need_cuda(x); x = _f32(x)
    y = torch.empty_like(x)
    _call('gelu_fwd', (_p(x), _p(y), x.numel(), _stream()))
    return y


def gelu_bwd(x, dy):
    _need_cuda(x, dy); x = _f32(x); dy = _f32(dy)
    dx = torch.empty_like(x)
    _call('gelu_bwd', (_p(x), _p(dy), _p(dx), x.numel(), _stream()))
    return dx


def add_pos_(x, pos, n_tok):
    _need_cuda(x, pos)
    _call('add_pos', (_p(x), _p(_f32(pos)), x.shape[0], n_tok, x.shape[1], _stream()))
    return x


def attention_fwd(qkv, B, n_tok):
    _need_cuda(qkv); qkv = _f32(qkv)
    O = torch.empty((B * n_tok, 64), device=qkv.device, dtype=torch.float32)
    P = torch.empty((B, n_tok, n_tok), device=qkv.device, dtype=torch.float32)
    _set_work(flops=4.0 * B * n_tok * n_tok * 64)
    _call('attention_fwd', (_p(qkv), _p(O), _p(P), B, n_tok, _stream()))
    return O, P


def attention_bwd(qkv, P, dO, B, n_tok):
    _need_cuda(qkv, P, dO); dO = _f32(dO)
    dqkv = torch.empty_like(qkv)
    _set_work(flops=8.0 * B * n_tok * n_tok * 64)
    _call('attention_bwd', (_p(qkv), _p(P), _p(dO), _p(dqkv), B, n_tok, _stream()))
    return dqkv


# ---------------------------------------------------------------------------------------------- specialist layers, training direction
def conv1x1_ctx_bwd(x, dz, cmat, NN, contextflow, dldj=None, need_dx=True):
    _need_cuda(x, dz, cmat); x = _f32(x); dz = _f32(dz); cmat = _f32(cmat)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel()
    dx = torch.empty_like(x) if need_dx else None
    dc = torch.empty_like(cmat)
    _set_work(flops=4.0 * B * D * D * HW)
    _call('conv1x1_ctx_bwd', (_p(x), _p(dz), _p(cmat), _p(None if NN is None else _f32(NN)), int(bool(contextflow)),
                              _p(None if dldj is None else _f32(dldj)), _p(dx), _p(dc), B, D, HW, _stream()))
    return dx, dc


def actnorm_ctx_bwd(x, dz, cm, base_t, base_logs, dldj=None, need_dx=True):
    _need_cuda(x, dz, cm); x = _f32(x); dz = _f32(dz); cm = _f32(cm)
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel()
    dx = torch.empty_like(x) if need_dx else None
    dc = torch.empty_like(cm)
    _set_work(bytes=(12.0 if need_dx else 8.0) * x.numel())
    _call('actnorm_ctx_bwd', (_p(x), _p(dz), _p(cm), _p(base_t), _p(base_logs), _p(None if dldj is None else _f32(dldj)), _p(dx), _p(dc),
                              B, D, HW, _stream()))
    return dx, dc


def gmm_ctx_train_fwd(x, mG, sG, wG, c):
    _need_cuda(x, mG, c); c = _f32(c)
    xv, bstride = _half_view(x)
    B, D, HW = x.shape[0], x.shape[1], x.shape[2] * x.shape[3]
    M, K = wG.shape
    logp = torch.empty((B, M), device=x.device, dtype=torch.float32)
    resp = torch.empty((B, M, K), device=x.device, dtype=torch.float32)
    _set_work(flops=8.0 * B * M * K * D * HW)
    _call('gmm_ctx_train_fwd', (_p(xv), bstride, _p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(c), _p(logp), _p(resp), B, M, K, D, HW, _stream()))
    return logp, resp


def gmm_ctx_train_bwd(x, mG, sG, c, resp, g, need_dx=True, dx_out=None):
    _need_cuda(x, mG, c, g); c = _f32(c); g = _f32(g)
    xv, bstride = _half_view(x)
    B, D, HW = x.shape[0], x.shape[1], x.shape[2] * x.shape[3]
    M, K = resp.shape[1], resp.shape[2]
    if dx_out is not None:
        dv, dstride = _half_view(dx_out)
        assert dv.data_ptr() == dx_out.data_ptr()
        dx = dx_out
    else:
        dstride = D * HW
        dx = torch.empty((B, D) + tuple(x.shape[2:]), device=x.device, dtype=torch.float32) if need_dx else None
    dc = torch.empty_like(c)
    _set_work(flops=24.0 * B * M * K * D * HW)
    _call('gmm_ctx_train_bwd', (_p(xv), bstride, _p(_f32(mG)), _p(_f32(sG)), _p(c), _p(resp), _p(g), _p(dx), dstride, _p(dc), B, M, K, D, HW, _stream()))
    return dx, dc


# One training step scatters into the embedding tables of every context-conditioned layer (39 layers x 2 features in BASELINE cfg2) and each
# call sorted the SAME context column again: 624 radix-sort launches, 5.3 of 106 ms per step (profiles/r2bb_launches_train_cfg2_summary.txt).
# The sort of a column is kept for the rest of the step, keyed by the context tensor's storage, version counter and layout; FlowSequential.forward
# empties the cache whenever a forward pass starts under autograd (begin_training_step), so a CUDA-graph capture pass -- which begins with its own
# forward -- never reuses tensors sorted outside the capture, and an in-place update of the context (version bump) misses the cache.
_CTX_SORT = {}


def begin_training_step():
    _CTX_SORT.clear()


def _sorted_context(ctx, i, card):
    key = (ctx.data_ptr(), ctx._version, tuple(ctx.shape), tuple(ctx.stride()), ctx.dtype, ctx.device, i, torch.cuda.is_current_stream_capturing())
    hit = _CTX_SORT.get(key)
    if hit is None:
        col = ctx[:, i].contiguous()
        srt, perm = torch.sort(col, stable=True)
        hit = _CTX_SORT[key] = (srt, perm.contiguous(), {})
    srt, perm, offs = hit
    if card not in offs:
        # bucket boundaries without a host synchronisation (torch.bincount sizes its output from the data): capturable in a CUDA graph
        offs[card] = torch.searchsorted(srt, torch.arange(card + 1, device=ctx.device, dtype=srt.dtype)).contiguous()
    return perm, offs[card]


def embed_scatter(dc, ctx, tables):
    """Gradients of the embedding tables from dc (B, n_ctx * width): per feature a stable sort of the batch by context value (torch,
    index preparation only; once per step and feature) and one deterministic bucket-sum kernel."""
    _need_cuda(dc, ctx); dc = _f32(dc)
    width = tables[0].shape[1]
    out = []
    for i, t in enumerate(tables):
        card = t.shape[0]
        perm, offsets = _sorted_context(ctx, i, card)
        dt = torch.empty((card, width), device=dc.device, dtype=torch.float32)
        _call('embed_scatter', (_p(dc), dc.shape[1], i * width, _p(perm), _p(offsets), _p(dt), card, width, _stream()))
        out.append(dt)
    return out


def cond_gauss_fwd(c, eps):
    _need_cuda(c, eps); c = _f32(c); eps = _f32(eps)
    B, C_ = eps.shape
    x = torch.empty_like(eps); logq = torch.empty(B, device=eps.device, dtype=torch.float32)
    _call('cond_gauss_fwd', (_p(c), _p(eps), _p(x), _p(logq), B, C_, _stream()))
    return x, logq


def cond_gauss_bwd(c, eps, dx, dlogq):
    _need_cuda(c, eps)
    B, C_ = eps.shape
    dc = torch.empty_like(c)
    _call('cond_gauss_bwd', (_p(c), _p(eps), _p(None if dx is None else _f32(dx)), _p(None if dlogq is None else _f32(dlogq)), _p(dc), B, C_, _stream()))
    return dc


def vardeq_fwd(u, qu, xcat, qbins, ldj_const, mode=0):
    """mode 0 vardeq, 1 argmax (xcat = +-1 signs), 2 probsample."""
    _need_cuda(u, qu, xcat, qbins); u = _f32(u); qu = _f32(qu)
    B, C_ = u.shape
    z = torch.empty_like(u); ldj = torch.empty(B, device=u.device, dtype=torch.float32)
    _call('vardeq_fwd', (_p(u), _p(qu), _p(None if xcat is None else xcat.contiguous()), _p(None if qbins is None else _f32(qbins)), float(ldj_const),
                         int(mode), _p(z), _p(ldj), B, C_, _stream()))
    return z, ldj


def vardeq_bwd(u, xcat, qbins, dz, dldj, mode=0):
    _need_cuda(u, xcat, qbins)
    B, C_ = u.shape
    du = torch.empty_like(u); dqu = torch.empty(B, device=u.device, dtype=torch.float32)
    _call('vardeq_bwd', (_p(u), _p(None if xcat is None else xcat.contiguous()), _p(None if qbins is None else _f32(qbins)), int(mode),
                         _p(None if dz is None else _f32(dz)), _p(None if dldj is None else _f32(dldj)), _p(du), _p(dqu), B, C_, _stream()))
    return du, dqu


# ---------------------------------------------------------------------------------------------- rows beside the headline path (SURVEY §8f)
_ACT_KIND = dict(sigmoid=0, softplus=1)


def activation_fwd(x, kind, temperature=None):
    """Standalone Sigmoid / Softplus flow layer (activations.py:228-264) on (..., D): (z, ldj over the last axis)."""
    _need_cuda(x, temperature); x = _f32(x)
    D = x.shape[-1]
    rows = x.numel() // D if D else 0
    z = torch.empty_like(x); ldj = torch.empty(x.shape[:-1], device=x.device, dtype=torch.float32)
    _set_work(bytes=8.0 * x.numel())
    _call('activation_fwd', (_p(x), _p(z), _p(ldj), _p(temperature), rows, D, _ACT_KIND[kind], _stream()))
    return z, ldj


def activation_inv(z, kind, eps, temperature=None):
    _need_cuda(z, temperature); z = _f32(z)
    x = torch.empty_like(z)
    _set_work(bytes=8.0 * z.numel())
    _call('activation_inv', (_p(z), _p(x), _p(temperature), z.numel(), float(eps), _ACT_KIND[kind], _stream()))
    return x


def activation_bwd(x, dz, dldj, kind, temperature=None):
    _need_cuda(x, dz, dldj, temperature); x = _f32(x)
    D = x.shape[-1]
    dx = torch.empty_like(x)
    _call('activation_bwd', (_p(x), _p(None if dz is None else _f32(dz)), _p(None if dldj is None else _f32(dldj)), _p(dx), _p(temperature),
                             x.numel() // D if D else 0, D, _ACT_KIND[kind], _stream()))
    return dx


def student_table(mG, sG, wG, mS, sS, wS, vS):
    """Per-element constants of StudentMixtureDistribution (student.py:76-82) for student_logprob; rebuild when parameters change."""
    _need_cuda(mG, sG, wG, mS, sS, wS, vS)
    M, K = wG.shape
    n = mG[0, 0].numel()
    tab = torch.empty(int(lib().cfpp_student_table_floats(M, K, n)), device=mG.device, dtype=torch.float32)
    _call('student_prep', (_p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(_f32(mS)), _p(_f32(sS)), _p(_f32(wS)), _p(_f32(vS)), _p(tab), M, K, n, _stream()))
    return tab


def student_logprob(x, table, M, K):
    _need_cuda(x, table); x = _f32(x)
    B = x.shape[0]
    n = x[0].numel() if B else 1
    logp = torch.empty((B, M), device=x.device, dtype=torch.float32)
    _set_work(flops=12.0 * B * M * K * n)
    _call('student_logprob', (_p(x), _p(table), _p(logp), B, M, K, n, _stream()))
    return logp


def student_train_fwd(x, table, M, K):
    """student_logprob under autograd: also the responsibilities resp (B, M, 2, K) of the Gaussian (0) and Student-t (1) components.
    x (B, D, H, W) may be a channel slice of a contiguous tensor (SplitPrior)."""
    _need_cuda(x, table)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    n = x[0].numel() if B else 1
    logp = torch.empty((B, M), device=x.device, dtype=torch.float32)
    resp = torch.empty((B, M, 2, K), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * n + 4.0 * B * M * (1 + 2 * K), flops=12.0 * B * M * K * n)
    _call('student_train_fwd', (_p(xv), bstride, _p(table), _p(logp), _p(resp), B, M, K, n, _stream()))
    return logp, resp


def student_train_bwd(x, table, sG, wG, sS, wS, resp, g, need_dx=True, need_params=True, dx_out=None):
    """-> dx, (dmG, dsG, dwG, dmS, dsS, dwS) or None.  dx_out: optional (B, D, H, W) channel-slice view of a wider contiguous tensor that
    receives dx in place."""
    _need_cuda(x, table, g); g = _f32(g)
    xv, bstride = _half_view(x)
    B = x.shape[0]
    M, K = resp.shape[1], resp.shape[3]
    n = x[0].numel()
    if dx_out is not None:
        dv, dstride = _half_view(dx_out)
        assert dv.data_ptr() == dx_out.data_ptr(), 'student_train_bwd: dx_out must be a channel slice of a contiguous tensor'
        dx = dx_out
    else:
        dstride = n
        dx = torch.empty((B,) + tuple(x.shape[1:]), device=x.device, dtype=torch.float32) if need_dx else None
    grads = None
    if need_params:
        grads = tuple(torch.empty(p.shape, device=x.device, dtype=torch.float32) for p in (sG, sG, wG, sS, sS, wS))
    ws = torch.empty(int(lib().cfpp_student_train_bwd_workspace_floats(B, M, K, n)), device=x.device, dtype=torch.float32)
    _set_work(bytes=4.0 * B * n * ((2 if need_dx else 0) + (1 if need_params else 0)), flops=(24.0 if need_params else 12.0) * B * M * K * n)
    gp = [None] * 6 if grads is None else [_p(t) for t in grads]
    _call('student_train_bwd', (_p(xv), bstride, _p(table), _p(_f32(sG)), _p(_f32(wG)), _p(_f32(sS)), _p(_f32(wS)), _p(_f32(resp)), _p(g),
                                _p(dx), dstride, *gp, _p(ws), B, M, K, n, _stream()))
    return dx, grads


def bias_rows_relu_(a, bias):
    """a (B, C, H, W) <- relu(a + bias[b, c]) in place (conventional coupling's first convolution, coupling.py:47)."""
    _need_cuda(a, bias)
    B, Cc = a.shape[0], a.shape[1]
    _call('bias_rows_relu', (_p(a), _p(_f32(bias)), B, Cc, a[0, 0].numel() if B else 1, _stream()))
    return a


def gmm_ctx_param_bwd(x, mG, sG, wG, c, resp, g):
    """Gradients of the mixture's own parameters beside per-sample context offsets (gaussian.py:131-155, contextflow = False)."""
    _need_cuda(x, mG, c, g); c = _f32(c); g = _f32(g)
    xv, bstride = _half_view(x)
    B, D, HW = x.shape[0], x.shape[1], x.shape[2] * x.shape[3]
    M, K = resp.shape[1], resp.shape[2]
    dmG = torch.empty_like(mG, dtype=torch.float32); dsG = torch.empty_like(sG, dtype=torch.float32); dwG = torch.empty_like(wG, dtype=torch.float32)
    _set_work(flops=24.0 * B * M * K * D * HW)
    _call('gmm_ctx_param_bwd', (_p(xv), bstride, _p(_f32(mG)), _p(_f32(sG)), _p(_f32(wG)), _p(c), _p(_f32(resp)), _p(g), _p(dmG), _p(dsG), _p(dwG),
                                B, M, K, D, HW, _stream()))
    return dmG, dsG, dwG
