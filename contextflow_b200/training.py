"""Training direction of the context-free (generalist) conv stack (SURVEY §8f-1): torch.autograd.Function wrappers whose forward AND
backward are libcfpp kernels, so that the reference's own training loop (experiment_ad.py:204-213: loss from `model.log_prob`,
`cost_sum.backward()`, the torch optimizer model.py:289 builds) runs unchanged over these layers.

What is covered: Conv1x1, ActNorm, Coupling (conv conditioner), Squeeze, the mixture base and the (B,M) log-det accumulation without a
context_net -- the cfg1 stack.  Context-conditioned (specialist) layers, the ViT conditioner and split priors still raise
NotImplementedError under autograd (next scope row).  Gradients match torch autograd over the reference's op sequence to 1e-4
relative (tests/test_gpu_training.py)."""
from __future__ import annotations

import torch
from torch.autograd import Function

from . import ops


def wants_grad(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _zeros_like_if_none(g, ref_shape, device):
    return torch.zeros(ref_shape, device=device, dtype=torch.float32) if g is None else g


class SqueezeFn(Function):
    @staticmethod
    def forward(ctx, x, p1, p2):
        ctx.p = (p1, p2)
        return ops.squeeze(x, p1, p2)

    @staticmethod
    def backward(ctx, dy):
        return ops.unsqueeze(dy.contiguous(), *ctx.p), None, None


class UnSqueezeFn(Function):
    @staticmethod
    def forward(ctx, y, p1, p2):
        ctx.p = (p1, p2)
        return ops.unsqueeze(y, p1, p2)

    @staticmethod
    def backward(ctx, dx):
        return ops.squeeze(dx.contiguous(), *ctx.p), None, None


class PermuteFn(Function):
    """PermuteAxes((0,2,1,3)) (permute_axes.py:13-14): the swap is its own inverse."""

    @staticmethod
    def forward(ctx, x):
        return ops.permute_chw(x)

    @staticmethod
    def backward(ctx, dy):
        return ops.permute_chw(dy.contiguous())


class Conv1x1Fn(Function):
    """z = NN x per pixel, ldj = HW log|det NN| (conv1x1.py:52-55)."""

    @staticmethod
    def forward(ctx, x, NN, layer):
        z, ldj = ops.conv1x1(x, NN.detach(), layer.logabsdet())
        ctx.save_for_backward(x, NN)
        ctx.layer = layer
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, NN = ctx.saved_tensors
        B, D, H, W = x.shape
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        w4 = NN.detach().reshape(D, D, 1, 1)
        dNN = None
        if ctx.needs_input_grad[1]:
            dNN, _ = ops.conv2d_bwd_weight(x, D, dz, (D, D, 1, 1), bias=False)
            dNN = dNN.view(D, D)
            if dldj is not None:
                ops.logdet_grad_(dNN, ctx.layer.inverse_matrix(check=False), dldj.contiguous(), H * W)
        dx = ops.conv2d_bwd_data(dz, w4) if ctx.needs_input_grad[0] else None
        return dx, dNN, None


class ActNormFn(Function):
    """z = (x - t) exp(-logs), ldj = sum logs (actnorm.py:50-60, context-free)."""

    @staticmethod
    def forward(ctx, x, t, logs):
        z, ldj = ops.actnorm(x, t.detach(), logs.detach())
        ctx.save_for_backward(x, t, logs)
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, t, logs = ctx.saved_tensors
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dt, dlogs = ops.actnorm_bwd(x, dz, None if dldj is None else dldj.contiguous(), t.detach(), logs.detach(),
                                        need_dx=ctx.needs_input_grad[0])
        return dx, dt, dlogs


def _conditioner_fwd(x, Ch, w1, b1, w2, b2, w3, b3):
    """(a1, a2, h) of the 3-conv conditioner on x[:, :Ch] (coupling.py:26-29).  float32 shapes with a tensor-core plan run the inference
    conditioner kernel with its post-ReLU activations written out for the backward pass (cfpp_conv_cond_tc_train_fwd: fp16 hi / scaled-lo
    pairs, fp32 faithful); everything else -- and CFPP_TRAIN_TC=0 -- runs three FP32 convolution launches."""
    import os
    if (x.dtype == torch.float32 and w2.dim() == 4 and os.environ.get('CFPP_TRAIN_TC', '1') != '0'
            and w1.dtype == torch.float32 and w1.shape[1] == Ch and w1.numel() == w1.shape[0] * Ch):
        ch, cout, KH, KW = w2.shape[0], w3.shape[0], w2.shape[2], w2.shape[3]
        pack = ops.conv_cond_tc_pack(w1.detach(), w2.detach(), w3.detach(), Ch)
        if pack is not None:
            out = ops.conv_cond_tc_train(x, Ch, pack, b1.detach().float().contiguous(), b2.detach().float().contiguous(), b3.detach().float().contiguous(),
                                         ch, x.shape[2], x.shape[3], KH, KW, cout)
            if out is not None:
                h, a1, a2 = out
                return a1, a2, h
    a1 = ops.conv2d_fwd(x, Ch, w1.detach(), b1.detach(), relu=True)
    a2 = ops.conv2d_fwd(a1, a1.shape[1], w2.detach(), b2.detach(), relu=True)
    h = ops.conv2d_fwd(a2, a2.shape[1], w3.detach(), b3.detach(), relu=False)
    return a1, a2, h


class CouplingConvFn(Function):
    """Coupling with the 3-conv conditioner (coupling.py:26-29,39-66), context-free.  Training forward = three conv launches with the
    post-ReLU activations saved + the coupling kernel; backward = coupling_bwd, then the conditioner's weight / data gradients, the
    last one accumulated onto dx's pass-through half."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, w3, b3):
        Ch = x.shape[1] // 2
        a1, a2, h = _conditioner_fwd(x, Ch, w1, b1, w2, b2, w3, b3)
        z, ldj = ops.coupling(x, h)
        ctx.save_for_backward(x, a1, a2, h, w1, w2, w3)
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, a1, a2, h, w1, w2, w3 = ctx.saved_tensors
        Ch = x.shape[1] // 2
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dh = ops.coupling_bwd(x, h, dz, None if dldj is None else dldj.contiguous())
        dw3, db3 = ops.conv2d_bwd_weight(a2, a2.shape[1], dh, w3.shape)
        da2 = ops.conv2d_bwd_data(dh, w3.detach(), act=a2)
        dw2, db2 = ops.conv2d_bwd_weight(a1, a1.shape[1], da2, w2.shape)
        da1 = ops.conv2d_bwd_data(da2, w2.detach(), act=a1)
        dw1, db1 = ops.conv2d_bwd_weight(x, Ch, da1, w1.shape)
        ops.conv2d_bwd_data(da1, w1.detach(), out=dx, accumulate=True)       # dx[:, :Ch] += W1^T da1
        return (dx if ctx.needs_input_grad[0] else None), dw1, db1, dw2, db2, dw3, db3


class MaskedCouplingFn(Function):
    """MaskedCoupling (`--coupling maf`, ar.py:35-57) over MaskedResidualBlock2d (masked_conv_2d.py:81-98), context-free.  The weights the
    Function receives are already mask-multiplied in place (the reference's `weight.data *= mask` on every forward, :21-23); exactly like
    autograd in the reference, the weight gradients are the dense ones (the mask is applied to the data, not inside the graph)."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, w3, b3):
        r0 = ops.relu(x)
        a1 = ops.conv2d_fwd(r0, r0.shape[1], w1.detach(), b1.detach(), relu=True)
        a2 = ops.conv2d_fwd(a1, a1.shape[1], w2.detach(), b2.detach(), relu=True)
        h = ops.conv2d_fwd(a2, a2.shape[1], w3.detach(), b3.detach(), relu=False)
        z, ldj = ops.maf_coupling(x, h)
        ctx.save_for_backward(x, r0, a1, a2, h, w1, w2, w3)
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, r0, a1, a2, h, w1, w2, w3 = ctx.saved_tensors
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dh = ops.maf_coupling_bwd(x, h, dz, None if dldj is None else dldj.contiguous())
        dw3, db3 = ops.conv2d_bwd_weight(a2, a2.shape[1], dh, w3.shape)
        da2 = ops.conv2d_bwd_data(dh, w3.detach(), act=a2)
        dw2, db2 = ops.conv2d_bwd_weight(a1, a1.shape[1], da2, w2.shape)
        da1 = ops.conv2d_bwd_data(da2, w2.detach(), act=a1)
        dw1, db1 = ops.conv2d_bwd_weight(r0, r0.shape[1], da1, w1.shape)
        ops.conv2d_bwd_data(da1, w1.detach(), act=x, out=dx, accumulate=True)      # through relu(x): masked by x > 0
        return (dx if ctx.needs_input_grad[0] else None), dw1, db1, dw2, db2, dw3, db3


class GmmFn(Function):
    """GaussianMixtureDistribution.log_prob (gaussian.py:142-161), context-free."""

    @staticmethod
    def forward(ctx, x, mG, sG, wG, layer):
        inv_var, cst = layer._tables.get('train', [sG, wG], lambda: ops.gmm_train_prep(sG.detach(), wG.detach()))
        logp, resp = ops.gmm_train_fwd(x, mG.detach(), inv_var, cst)
        ctx.save_for_backward(x, mG, sG, wG, inv_var, resp)
        return logp

    @staticmethod
    def backward(ctx, g):
        x, mG, sG, wG, inv_var, resp = ctx.saved_tensors
        dx, dmG, dsG, dwG = ops.gmm_train_bwd(x, mG.detach(), sG.detach(), wG.detach(), inv_var, resp, g.contiguous(),
                                              need_dx=ctx.needs_input_grad[0])
        return dx, dmG, dsG, dwG, None


class SplitPriorFn(Function):
    """SplitPrior.forward (splitprior.py:12-15) with a context-free mixture: x -> (x[:, :C/2], log_prob(x[:, C/2:]))."""

    @staticmethod
    def forward(ctx, x, mG, sG, wG, layer):
        half = x.shape[1] // 2
        inv_var, cst = layer._tables.get('train', [sG, wG], lambda: ops.gmm_train_prep(sG.detach(), wG.detach()))
        logp, resp = ops.gmm_train_fwd(x[:, half:], mG.detach(), inv_var, cst)
        ctx.save_for_backward(x, mG, sG, wG, inv_var, resp)
        return ops.slice_channels(x, 0, half), logp

    @staticmethod
    def backward(ctx, dx0, g):
        x, mG, sG, wG, inv_var, resp = ctx.saved_tensors
        half = x.shape[1] // 2
        g = torch.zeros((x.shape[0], mG.shape[0]), device=x.device) if g is None else g.contiguous()
        need_dx = ctx.needs_input_grad[0]
        dx = torch.empty_like(x) if need_dx else None
        if need_dx:
            ops.place_channels(_zeros_like_if_none(dx0, (x.shape[0], half) + tuple(x.shape[2:]), x.device).contiguous(), dx, 0)
        _, dmG, dsG, dwG = ops.gmm_train_bwd(x[:, half:], mG.detach(), sG.detach(), wG.detach(), inv_var, resp, g, need_dx=need_dx,
                                             dx_out=dx[:, half:] if need_dx else None)
        return dx, dmG, dsG, dwG, None


class StudentMixtureFn(Function):
    """StudentMixtureDistribution.log_prob (student.py:76-98); the degrees of freedom vS stay frozen, as in the reference (student.py:59).
    `split` > 0: the SplitPrior form -- x is the full tensor, the mixture scores x[:, split:] and the Function also returns x[:, :split]
    (splitprior.py:12-15)."""

    @staticmethod
    def forward(ctx, x, dist, split, mG, sG, wG, mS, sS, wS):
        src = [mG, sG, wG, mS, sS, wS, dist.vS]
        table = dist._tables.get('student', src, lambda: ops.student_table(*[p.detach() for p in src]))
        logp, resp = ops.student_train_fwd(x[:, split:] if split else x, table, dist.M, dist.K)
        ctx.save_for_backward(x, table, resp, sG, wG, sS, wS)
        ctx.M, ctx.split = dist.M, split
        if split:
            return ops.slice_channels(x, 0, split), logp
        return logp

    @staticmethod
    def backward(ctx, *grads):
        x, table, resp, sG, wG, sS, wS = ctx.saved_tensors
        split = ctx.split
        dx0, g = grads if split else (None, grads[0])
        g = torch.zeros((x.shape[0], ctx.M), device=x.device) if g is None else g.contiguous()
        need_dx = ctx.needs_input_grad[0]
        need_params = any(ctx.needs_input_grad[3:])
        dx = None
        if split and need_dx:
            dx = torch.empty_like(x)
            ops.place_channels(_zeros_like_if_none(dx0, (x.shape[0], split) + tuple(x.shape[2:]), x.device).contiguous(), dx, 0)
        dxs, pg = ops.student_train_bwd(x[:, split:] if split else x, table, sG.detach(), wG.detach(), sS.detach(), wS.detach(), resp, g,
                                        need_dx=need_dx, need_params=need_params, dx_out=dx[:, split:] if dx is not None else None)
        if not split:
            dx = dxs
        pg = pg if pg is not None else (None,) * 6
        return (dx, None, None, *[d if need else None for d, need in zip(pg, ctx.needs_input_grad[3:])])


class LdjSumFn(Function):
    """logprob + ((0 + ldj_0) + ldj_1) + ...  (flowsequential.py:20-27); a (B,) / (B,1) term receives the row sum of the gradient."""

    @staticmethod
    def forward(ctx, last, M, *terms):
        B = last.shape[0]
        ctx.shapes = [tuple(t.shape) for t in terms]
        ctx.M = M
        return ops.ldj_sum([t.detach() for t in terms], B, M, last.device, last=last.detach())

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        rs = None
        grads = []
        for i, shp in enumerate(ctx.shapes):
            if not ctx.needs_input_grad[2 + i]:
                grads.append(None)
            elif len(shp) == 2 and shp[1] == ctx.M and ctx.M > 1:
                grads.append(g)
            else:
                if rs is None:
                    rs = ops.rowsum(g)
                grads.append(rs.view(shp))
        return (g, None, *grads)


class CouplingVitFn(Function):
    """TransCoupling with the SimpleViT conditioner (coupling.py:100-148, simple_vit.py:30-127), context-free.  The training forward is
    the reference's module stack op by op on token rows (LayerNorm, Linear, single-head attention, GELU, residuals) with the
    activations saved; the backward walks it in reverse.  Parameter order = SimpleViT._sources()."""

    @staticmethod
    def forward(ctx, x, add, logp_c, vit, *params):
        # add (B, C) / logp_c (B): the context term CN(c) and the encoder's log-density of a specialist (coupling.py:126-133; note logp_c
        # is NOT scaled by H*W in TransCoupling); None for a generalist.  --contextflow adds CN(c) to h; a conventional specialist
        # (vit.geom['Cin'] = C/2 + C input channels) concatenates CN(c), broadcast over the pixels, to x0 (coupling.py:129).
        g = vit.geom
        c, p1, p2, T, n, depth = g['Cin'], g['p1'], g['p2'], g['T'], g['n_tok'], g['depth']
        B, C, H, W = x.shape
        P = [p.detach() for p in params]
        ln0w, ln0b, pew, peb, ln1w, ln1b, lnfw, lnfb = P[:8]
        concat = add is not None and c > C // 2
        if concat:
            xin = torch.cat([x.detach()[:, :C // 2], add.detach()[:, :, None, None].expand(B, add.shape[1], H, W)], dim=1).contiguous()
            tok = ops.patchify(xin, c, p1, p2)
            add = None
        else:
            tok = ops.patchify(x, c, p1, p2)
        y0, m0, r0 = ops.layernorm_fwd(tok, ln0w, ln0b)
        e = ops.rows_linear(y0, pew, peb)
        X, m1, r1 = ops.layernorm_fwd(e, ln1w, ln1b)
        pos = getattr(vit, '_pos_dev', None)                 # the sincos table on the device, uploaded once (not per step: no H2D in a captured step)
        if pos is None or pos.device != x.device:
            pos = vit._pos_dev = vit.pos_embedding.to(x.device, torch.float32).contiguous()
        ops.add_pos_(X, pos, n)
        saved = [tok, m0, r0, y0, e, m1, r1]
        for l in range(depth):
            anw, anb, qkvw, outw, f0w, f0b, f1w, f1b, f3w, f3b = P[8 + 10 * l: 18 + 10 * l]
            y, ma, ra = ops.layernorm_fwd(X, anw, anb)
            qkv = ops.rows_linear(y, qkvw)
            O, Pm = ops.attention_fwd(qkv, B, n)
            X1 = ops.add(ops.rows_linear(O, outw), X)
            y2, mf, rf = ops.layernorm_fwd(X1, f0w, f0b)
            hpre = ops.rows_linear(y2, f1w, f1b)
            gact = ops.gelu_fwd(hpre)
            X2 = ops.add(ops.rows_linear(gact, f3w, f3b), X1)
            saved += [X, ma, ra, y, qkv, Pm, O, X1, mf, rf, y2, hpre, gact]
            X = X2
        Xf, mz, rz = ops.layernorm_fwd(X, lnfw, lnfb)
        cc = T // (p1 * p2)
        h = ops.patchify_inv(Xf, cc, H, W, p1, p2)
        z, ldj = ops.coupling(x, h, add=add, logp_c=logp_c, logp_scale=1.0)
        saved += [X, mz, rz, x, h]
        ctx.save_for_backward(*saved, *params)
        ctx.add, ctx.concat = add, concat
        ctx.meta = (c, p1, p2, T, n, depth, B, H, W, cc, len(saved))
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        c, p1, p2, T, n, depth, B, H, W, cc, ns = ctx.meta
        S = ctx.saved_tensors[:ns]
        P = [p.detach() for p in ctx.saved_tensors[ns:]]
        ln0w, ln0b, pew, peb, ln1w, ln1b, lnfw, lnfb = P[:8]
        Xlast, mz, rz, x, h = S[-5:]
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dh = ops.coupling_bwd(x, h, dz, None if dldj is None else dldj.contiguous(), add=ctx.add)
        dadd = ops.rowsum(dh.view(B * dh.shape[1], -1)).view(B, dh.shape[1]) if ctx.add is not None else None
        grads = [None] * len(P)
        ng = ctx.needs_input_grad

        def wgrad(idx, xin, dy, bias=True):              # frozen ViT parameters (--contextflow specialists): no weight gradient launches
            if not ng[4 + idx]:
                return None, None
            return ops.rows_linear_bwd_weight(xin, dy, bias=bias)
        dXf = ops.patchify(dh, cc, p1, p2)
        dX, grads[6], grads[7] = ops.layernorm_bwd(Xlast, dXf, lnfw, mz, rz)
        for l in reversed(range(depth)):
            X, ma, ra, y, qkv, Pm, O, X1, mf, rf, y2, hpre, gact = S[7 + 13 * l: 20 + 13 * l]
            o = 8 + 10 * l
            anw, anb, qkvw, outw, f0w, f0b, f1w, f1b, f3w, f3b = P[o: o + 10]
            grads[o + 8], grads[o + 9] = wgrad(o + 8, gact, dX)
            dhpre = ops.gelu_bwd(hpre, ops.rows_linear_bwd_data(dX, f3w))
            grads[o + 6], grads[o + 7] = wgrad(o + 6, y2, dhpre)
            d1, grads[o + 4], grads[o + 5] = ops.layernorm_bwd(X1, ops.rows_linear_bwd_data(dhpre, f1w), f0w, mf, rf)
            dX1 = ops.add(dX, d1)
            grads[o + 3], _ = wgrad(o + 3, O, dX1, bias=False)
            dqkv = ops.attention_bwd(qkv, Pm, ops.rows_linear_bwd_data(dX1, outw), B, n)
            grads[o + 2], _ = wgrad(o + 2, y, dqkv, bias=False)
            d0, grads[o], grads[o + 1] = ops.layernorm_bwd(X, ops.rows_linear_bwd_data(dqkv, qkvw), anw, ma, ra)
            dX = ops.add(dX1, d0)
        tok, m0, r0, y0, e, m1, r1 = S[:7]
        de, grads[4], grads[5] = ops.layernorm_bwd(e, dX, ln1w, m1, r1)
        grads[2], grads[3] = wgrad(2, y0, de)
        dtok, grads[0], grads[1] = ops.layernorm_bwd(tok, ops.rows_linear_bwd_data(de, pew), ln0w, m0, r0)
        if ctx.concat:                                                             # input gradient of cat(x0, CN(c)): x0 part onto dx, the rest summed over pixels
            Ch = x.shape[1] // 2
            dxin = ops.patchify_inv(dtok, c, H, W, p1, p2)
            ops.place_channels(ops.add(ops.slice_channels(dx, 0, Ch), ops.slice_channels(dxin, 0, Ch)), dx, 0)
            dadd = ops.rowsum(ops.slice_channels(dxin, Ch, c - Ch).view(B * (c - Ch), -1)).view(B, c - Ch)
        else:
            ops.patchify_inv(dtok, c, H, W, p1, p2, out=dx, accumulate=True)      # dx[:, :c] += the conditioner's input gradient
        grads = [gr if ng[4 + i] else None for i, gr in enumerate(grads)]          # frozen ViT parameters (--contextflow) take none
        dlogp = dldj if (ng[2] and dldj is not None) else None                                      # TransCoupling: logp_c unscaled (coupling.py:126)
        return (dx if ng[0] else None, dadd, dlogp, None, *grads)


# ---------------------------------------------------------------------------------------------- specialist (--contextflow) layers
def encoder_is_constant(context_net) -> bool:
    """True when the layer's context encoder has no trainable parameter (onehot / eye embeddings with the uniform surjection -- the
    reference's default `--enc-emb onehot --enc-type uniform`): its output (c, logp_c) is then a constant of the graph.  Encoders with
    inner flows (vardeq, argmax, probsample) or trainable embeddings have no backward kernels yet."""
    return not any(p.requires_grad for p in context_net.parameters())


def require_constant_encoder(context_net):
    if not encoder_is_constant(context_net):
        raise NotImplementedError('training through a context encoder with trainable parameters (vardeq / argmax / probsample flows, embed '
                                  'tables) has no backward kernel yet; onehot|eye + uniform encoders train (DESIGN.md §8 f-1)')


class LinearRowsFn(Function):
    """nn.Linear on (B, K) rows: the CN of Conv1x1 / ActNorm (conv1x1.py:22, actnorm.py:21)."""

    @staticmethod
    def forward(ctx, c, W, b):
        ctx.save_for_backward(c, W)
        return ops.rows_linear(c, W.detach(), b.detach())

    @staticmethod
    def backward(ctx, dy):
        c, W = ctx.saved_tensors
        dy = dy.contiguous()
        dW, db = ops.rows_linear_bwd_weight(c, dy)
        dc = ops.rows_linear_bwd_data(dy, W.detach()) if ctx.needs_input_grad[0] else None
        return dc, dW, db


class Mlp3RowsFn(Function):
    """Linear-ReLU-Linear-ReLU-Linear on (B, K) rows: the CN of the couplings (coupling.py:37,121)."""

    @staticmethod
    def forward(ctx, c, w1, b1, w2, b2, w3, b3):
        h1 = ops.relu(ops.rows_linear(c, w1.detach(), b1.detach()))
        h2 = ops.relu(ops.rows_linear(h1, w2.detach(), b2.detach()))
        ctx.save_for_backward(c, h1, h2, w1, w2, w3)
        return ops.rows_linear(h2, w3.detach(), b3.detach())

    @staticmethod
    def backward(ctx, dout):
        c, h1, h2, w1, w2, w3 = ctx.saved_tensors
        dout = dout.contiguous()
        dw3, db3 = ops.rows_linear_bwd_weight(h2, dout)
        dh2 = ops.relu_mask_(ops.rows_linear_bwd_data(dout, w3.detach()), h2)
        dw2, db2 = ops.rows_linear_bwd_weight(h1, dh2)
        dh1 = ops.relu_mask_(ops.rows_linear_bwd_data(dh2, w2.detach()), h1)
        dw1, db1 = ops.rows_linear_bwd_weight(c, dh1)
        dc = ops.rows_linear_bwd_data(dh1, w1.detach()) if ctx.needs_input_grad[0] else None
        return dc, dw1, db1, dw2, db2, dw3, db3


class Conv1x1CtxFn(Function):
    """Conv1x1 with a per-sample context matrix (conv1x1.py:31-50); `cmat` = CN(c) (B, D*D); NN is frozen under --contextflow."""

    @staticmethod
    def forward(ctx, x, cmat, logp_c, layer):
        z, ldj = ops.conv1x1(x, layer.NN.detach(), layer.logabsdet(), cmat, logp_c, layer.contextflow)
        ctx.save_for_backward(x, cmat)
        ctx.layer = layer
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, cmat = ctx.saved_tensors
        lay = ctx.layer
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dc = ops.conv1x1_ctx_bwd(x, dz, cmat, lay.NN.detach() if lay.contextflow else None, lay.contextflow,
                                     None if dldj is None else dldj.contiguous(), need_dx=ctx.needs_input_grad[0])
        HW = x.shape[2] * x.shape[3]
        dlogp = dldj * float(HW) if (ctx.needs_input_grad[2] and dldj is not None) else None      # ldj += HW * logp_c (conv1x1.py:50)
        return dx, dc, dlogp, None


class ActNormCtxFn(Function):
    """ActNorm with per-sample context shift / log-scale (actnorm.py:42-58); `cm` = CN(c) (B, 2D)."""

    @staticmethod
    def forward(ctx, x, cm, logp_c, layer):
        HW = x.shape[2] * x.shape[3]
        if layer.contextflow:
            z, ldj = ops.actnorm(x, layer.NN_t.detach(), layer.NN_logs.detach(), cm, logp_c, float(HW), mode=1)
        else:
            z, ldj = ops.actnorm(x, None, None, cm, logp_c, float(HW), mode=2)
        ctx.save_for_backward(x, cm)
        ctx.layer = layer
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, cm = ctx.saved_tensors
        lay = ctx.layer
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        bt, bl = (lay.NN_t.detach(), lay.NN_logs.detach()) if lay.contextflow else (None, None)
        dx, dc = ops.actnorm_ctx_bwd(x, dz, cm, bt, bl, None if dldj is None else dldj.contiguous(), need_dx=ctx.needs_input_grad[0])
        HW = x.shape[2] * x.shape[3]
        dlogp = dldj * float(HW) if (ctx.needs_input_grad[2] and dldj is not None) else None      # ldj += HW * logp_c (actnorm.py:44,60)
        return dx, dc, dlogp, None


class CouplingCtxConvFn(Function):
    """Coupling with the conv conditioner and the ADDITIVE context term of --contextflow (coupling.py:45): h = NN(x0) + CN(c).  NN is
    frozen in that mode (its weight gradients are skipped unless they require grad); `add` = CN(c) (B, C)."""

    @staticmethod
    def forward(ctx, x, add, logp_c, w1, b1, w2, b2, w3, b3):
        Ch = x.shape[1] // 2
        HW = x.shape[2] * x.shape[3]
        a1, a2, h = _conditioner_fwd(x, Ch, w1, b1, w2, b2, w3, b3)
        z, ldj = ops.coupling(x, h, add=add, logp_c=logp_c, logp_scale=float(HW))
        ctx.save_for_backward(x, add, a1, a2, h, w1, w2, w3)
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, add, a1, a2, h, w1, w2, w3 = ctx.saved_tensors
        B, C = x.shape[0], x.shape[1]
        Ch = C // 2
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dh = ops.coupling_bwd(x, h, dz, None if dldj is None else dldj.contiguous(), add=add)
        dadd = ops.rowsum(dh.view(B * C, -1)).view(B, C)
        ng = ctx.needs_input_grad
        dw3 = db3 = dw2 = db2 = dw1 = db1 = None
        if ng[7] or ng[8]:
            dw3, db3 = ops.conv2d_bwd_weight(a2, a2.shape[1], dh, w3.shape)
        da2 = ops.conv2d_bwd_data(dh, w3.detach(), act=a2)
        if ng[5] or ng[6]:
            dw2, db2 = ops.conv2d_bwd_weight(a1, a1.shape[1], da2, w2.shape)
        da1 = ops.conv2d_bwd_data(da2, w2.detach(), act=a1)
        if ng[3] or ng[4]:
            dw1, db1 = ops.conv2d_bwd_weight(x, Ch, da1, w1.shape)
        ops.conv2d_bwd_data(da1, w1.detach(), out=dx, accumulate=True)
        HW = x.shape[2] * x.shape[3]
        dlogp = dldj * float(HW) if (ng[2] and dldj is not None) else None                          # ldj += HW * logp_c (coupling.py:43)
        return (dx if ng[0] else None), dadd, dlogp, dw1, db1, dw2, db2, dw3, db3


class CouplingConcatConvFn(Function):
    """Coupling with the conv conditioner over the CONCATENATED context of a conventional specialist (coupling.py:47):
    h = NN(cat(x0, CN(c) broadcast)).  The first convolution is 1x1, so it equals W1[:, :D] x0 plus the per-sample bias
    b1 + W1[:, D:] CN(c); every weight trains (contextflow = False).  `cn` = CN(c) (B, O)."""

    @staticmethod
    def forward(ctx, x, cn, logp_c, w1, b1, w2, b2, w3, b3):
        Ch = x.shape[1] // 2
        HW = x.shape[2] * x.shape[3]
        w1d = w1.detach().reshape(w1.shape[0], -1)
        w1a, w1b = w1d[:, :Ch].contiguous(), w1d[:, Ch:].contiguous()
        bias1 = ops.rows_linear(cn.detach(), w1b, b1.detach())                                   # (B, H): b1 + W1[:, D:] CN(c)
        a1 = ops.bias_rows_relu_(ops.conv2d_fwd(x, Ch, w1a.view(-1, Ch, 1, 1), None, relu=False), bias1)
        a2 = ops.conv2d_fwd(a1, a1.shape[1], w2.detach(), b2.detach(), relu=True)
        h = ops.conv2d_fwd(a2, a2.shape[1], w3.detach(), b3.detach(), relu=False)
        z, ldj = ops.coupling(x, h, logp_c=logp_c, logp_scale=float(HW))
        ctx.save_for_backward(x, cn, a1, a2, h, w1a, w1b, w2, w3)
        ctx.w1_shape = tuple(w1.shape)
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        x, cn, a1, a2, h, w1a, w1b, w2, w3 = ctx.saved_tensors
        B, C = x.shape[0], x.shape[1]
        Ch, Hd = C // 2, a1.shape[1]
        dz = _zeros_like_if_none(dz, x.shape, x.device).contiguous()
        dx, dh = ops.coupling_bwd(x, h, dz, None if dldj is None else dldj.contiguous())
        dw3, db3 = ops.conv2d_bwd_weight(a2, a2.shape[1], dh, w3.shape)
        da2 = ops.conv2d_bwd_data(dh, w3.detach(), act=a2)
        dw2, db2 = ops.conv2d_bwd_weight(a1, a1.shape[1], da2, w2.shape)
        da1 = ops.conv2d_bwd_data(da2, w2.detach(), act=a1)
        dw1a, _ = ops.conv2d_bwd_weight(x, Ch, da1, (Hd, Ch, 1, 1), bias=False)
        dbias = ops.rowsum(da1.view(B * Hd, -1)).view(B, Hd)                                    # gradient of the per-sample bias
        dw1b, db1 = ops.rows_linear_bwd_weight(cn, dbias)                                       # W1[:, D:] and b1
        dcn = ops.rows_linear_bwd_data(dbias, w1b) if ctx.needs_input_grad[1] else None
        dw1 = torch.cat([dw1a.view(Hd, Ch), dw1b], dim=1).view(ctx.w1_shape)
        ops.conv2d_bwd_data(da1, w1a.view(Hd, Ch, 1, 1), out=dx, accumulate=True)                # dx[:, :Ch] += W1[:, :D]^T da1
        HW = x.shape[2] * x.shape[3]
        dlogp = dldj * float(HW) if (ctx.needs_input_grad[2] and dldj is not None) else None      # ldj += HW * logp_c (coupling.py:43)
        return (dx if ctx.needs_input_grad[0] else None), dcn, dlogp, dw1, db1, dw2, db2, dw3, db3


def _lookup_tables(dist):
    """The embedding tables of a mixture's context_net when it is the embed + eyesample lookup create_model gives every prior
    (model.py:157,162); None otherwise."""
    from .layers._encoder_desc import EncoderBatch
    fused = dist._plan.fused_for(dist.context_net)
    if fused is None or not EncoderBatch.is_lookup(fused):
        return None
    return fused.emb.tables()


class GmmCtxFn(Function):
    """GaussianMixtureDistribution.log_prob with context offsets from an embedding lookup (gaussian.py:146-155).  The tables always
    train; mG, sG, wG are frozen under --contextflow and train beside the tables in a conventional specialist (gaussian.py:137-141).
    `split` > 0: the SplitPrior form -- x is the full tensor, the mixture scores x[:, split:] and the Function also returns
    x[:, :split] (splitprior.py:12-15)."""

    @staticmethod
    def forward(ctx, x, context, dist, split, mG, sG, wG, *tables):
        c = ops.embed_lookup(context, [t.detach() for t in tables])
        xs = x[:, split:] if split else x
        logp, resp = ops.gmm_ctx_train_fwd(xs, mG.detach(), sG.detach(), wG.detach(), c)
        ctx.save_for_backward(x, context, c, resp, mG, sG, wG, *tables)
        ctx.dist, ctx.split = dist, split
        if split:
            return ops.slice_channels(x, 0, split), logp
        return logp

    @staticmethod
    def backward(ctx, *grads):
        x, context, c, resp, mG, sG, wG = ctx.saved_tensors[:7]
        tables = ctx.saved_tensors[7:]
        dist, split = ctx.dist, ctx.split
        mG, sG, wG = mG.detach(), sG.detach(), wG.detach()
        dx0, g = (grads if split else (None, grads[0]))
        g = torch.zeros((x.shape[0], dist.M), device=x.device) if g is None else g.contiguous()
        need_dx = ctx.needs_input_grad[0]
        if split:
            dx = torch.empty_like(x) if need_dx else None
            if need_dx:
                ops.place_channels(_zeros_like_if_none(dx0, (x.shape[0], split) + tuple(x.shape[2:]), x.device).contiguous(), dx, 0)
            _, dc = ops.gmm_ctx_train_bwd(x[:, split:], mG, sG, c, resp, g, need_dx=need_dx, dx_out=dx[:, split:] if need_dx else None)
        else:
            dx, dc = ops.gmm_ctx_train_bwd(x, mG, sG, c, resp, g, need_dx=need_dx)
        dtables = ops.embed_scatter(dc, context, tables)
        dmG = dsG = dwG = None
        if any(ctx.needs_input_grad[4:7]):                       # conventional specialist: the mixture itself trains too
            dmG, dsG, dwG = ops.gmm_ctx_param_bwd(x[:, split:] if split else x, mG, sG, wG, c, resp, g)
        return (dx, None, None, None, dmG, dsG, dwG, *dtables)


# ---------------------------------------------------------------------------------------------- encoders with trainable parameters
class EmbedLookupFn(Function):
    """CatEmbeddings.forward (rtdl/nn/_embeddings.py:265-283): concatenated table rows; backward = deterministic bucket sums."""

    @staticmethod
    def forward(ctx, context, *tables):
        ctx.save_for_backward(context, *tables)
        return ops.embed_lookup(context, [t.detach() for t in tables])

    @staticmethod
    def backward(ctx, dc):
        context, tables = ctx.saved_tensors[0], ctx.saved_tensors[1:]
        return (None, *ops.embed_scatter(dc.contiguous(), context, tables))


class CondGaussFn(Function):
    """ConditionalGaussianDistribution.sample given its parameters c = [mean | log_scale] and the draw eps (gaussian.py:263-270)."""

    @staticmethod
    def forward(ctx, c, eps):
        ctx.save_for_backward(c, eps)
        return ops.cond_gauss_fwd(c, eps)

    @staticmethod
    def backward(ctx, dx, dlogq):
        c, eps = ctx.saved_tensors
        return ops.cond_gauss_bwd(c, eps, None if dx is None else dx.contiguous(), None if dlogq is None else dlogq.contiguous()), None


class VardeqFn(Function):
    """The epilogue of VariationalCatDequantization.forward (dequantize.py:107-116)."""

    @staticmethod
    def forward(ctx, u, qu, xcat, qbins, ldj_const, mode):
        ctx.save_for_backward(u)
        ctx.aux = (xcat, qbins, mode)
        return ops.vardeq_fwd(u, qu, xcat, qbins, ldj_const, mode)

    @staticmethod
    def backward(ctx, dz, dldj):
        (u,) = ctx.saved_tensors
        xcat, qbins, mode = ctx.aux
        du, dqu = ops.vardeq_bwd(u, xcat, qbins, None if dz is None else dz.contiguous(), None if dldj is None else dldj.contiguous(), mode)
        return du, dqu, None, None, None, None


def encode(owner, context):
    """(c, logp_c) of a layer's context encoder under autograd.  Parameter-free encoders (onehot|eye + uniform) are constants of the graph
    and keep the fused kernel; the variational dequantiser (BASELINE cfg2) runs its module tree -- embedding lookup, conditional-Gaussian
    draw, the inner flow on the FC / ActNormFC / CouplingFC training kernels, the dequantisation epilogue -- in the reference's order
    (model.py:30-90, dequantize.py:107-116, flowsequential.py:60-69), drawing the same noise shapes as the fused path."""
    from . import rng
    from .layers.augment import Augment
    net = owner.context_net
    if encoder_is_constant(net):
        return owner._plan.run(net, context)
    emb, surj = net[0], net[1]
    kind = getattr(surj, 'kind', None)
    if context.dim() != 2:
        raise ValueError('context must be (B, n)')
    trainable_emb = any(p.requires_grad for p in emb.parameters())
    if kind == 'eyesample' and trainable_emb and hasattr(emb, 'tables'):      # embed + eyesample: c is the table lookup itself, ldj = 0
        return EmbedLookupFn.apply(context, *emb.tables()), torch.zeros(context.shape[0], device=context.device)
    # probsample ignores the embedding's values (dequantize.py:152-160 uses x for nothing but the batch size), so a trainable `embed`
    # table in front of it receives no gradient in the reference either
    if kind not in ('vardeq', 'argmax', 'probsample') or (trainable_emb and kind != 'probsample'):
        raise NotImplementedError(f'training through a {kind or type(surj).__name__} context encoder over {type(emb).__name__} has no backward '
                                  'kernel yet (DESIGN.md §8 f-1)')
    with torch.no_grad():
        x, ctx_i = emb(context)
    flow = surj.encoder
    dist = flow.dist
    cemb = EmbedLookupFn.apply(ctx_i, *dist.context_net.tables())
    eps = rng.randn((context.shape[0], dist.D), context.device)
    u, qu = CondGaussFn.apply(cemb, eps)
    for module in flow.sequence_modules:
        if isinstance(module, Augment):
            # the reference itself cannot run this configuration: Augment's (B,1) ldj is subtracted in place from the (B,) log-density
            # (flowsequential.py:66 -> "output with shape [B] doesn't match the broadcast shape [B, B]")
            raise RuntimeError('encoder flows with an Augment step (odd context width) fail in the reference (flowsequential.py:66)')
        u, ldj = module(u, ctx_i)
        qu = qu - ldj                                                   # flowsequential.py:66
    if kind == 'argmax':                                 # dequantize.py:244-256: bits MSB first per feature, one zero column if odd, sign = 2 bit - 1
        nb = surj.num_bits if isinstance(surj.num_bits, (list, tuple)) else [surj.num_bits] * context.shape[1]
        cols = []
        for i, bits in enumerate(nb):                    # integer index preparation (torch integer ops, no arithmetic of the path)
            shifts = torch.arange(bits - 1, -1, -1, device=context.device, dtype=torch.int64)
            cols.append((context[:, i:i + 1] >> shifts) & 1)
        bits_all = torch.cat(cols, 1)
        if bits_all.shape[1] % 2:
            bits_all = torch.cat([bits_all, torch.zeros_like(bits_all[:, :1])], 1)
        return VardeqFn.apply(u, qu, bits_all * 2 - 1, None, 0.0, 1)
    if kind == 'probsample':
        return VardeqFn.apply(u, qu, None, None, 0.0, 2)
    const = getattr(surj, '_ldj_const', None)
    if const is None:
        const = surj._ldj_const = float((surj.ldj_per_dim.detach().float().cpu() * x.shape[1:].numel()).sum())
    return VardeqFn.apply(u, qu, x, surj.qbins, const, 0)
