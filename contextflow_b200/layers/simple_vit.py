"""SimpleViT conditioner (reference layers/simple_vit.py:18-127): parameter container with the reference's module tree /
state_dict names; forward is the fused CUDA kernel (cfpp_vit_cond_fwd)."""
import ctypes

import torch
from torch import nn

from .. import _cabi, ops
from .flowlayer import PackCache

__all__ = ['SimpleViT', 'posemb_sincos_2d']


def pair(t):
    return t if isinstance(t, tuple) else (t, t)


def posemb_sincos_2d(h, w, dim, temperature: int = 10000, dtype=torch.float32):
    assert (dim % 4) == 0, 'feature dimension must be multiple of 4 for sincos emb'
    ys, xs = torch.meshgrid(torch.arange(h), torch.arange(w), indexing='ij')
    omega = 1.0 / (temperature ** (torch.arange(dim // 4) / (dim // 4 - 1)))
    ya = ys.flatten()[:, None] * omega[None, :]
    xa = xs.flatten()[:, None] * omega[None, :]
    return torch.cat((xa.sin(), xa.cos(), ya.sin(), ya.cos()), dim=1).type(dtype)


class FeedForward(nn.Module):
    def __init__(self, dim, hidden_dim):
        super().__init__()
        self.net = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, hidden_dim), nn.GELU(), nn.Linear(hidden_dim, dim))


class Attention(nn.Module):
    def __init__(self, dim, heads=8, dim_head=64):
        super().__init__()
        inner = dim_head * heads
        self.heads, self.scale = heads, dim_head ** -0.5
        self.norm = nn.LayerNorm(dim)
        self.attend = nn.Softmax(dim=-1)
        self.to_qkv = nn.Linear(dim, inner * 3, bias=False)
        self.to_out = nn.Linear(inner, dim, bias=False)


class Transformer(nn.Module):
    def __init__(self, dim, depth, heads, dim_head, mlp_dim):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.layers = nn.ModuleList([nn.ModuleList([Attention(dim, heads=heads, dim_head=dim_head), FeedForward(dim, mlp_dim)])
                                     for _ in range(depth)])


class SimpleViT(nn.Module):
    def __init__(self, *, image_size, patch_size, dim, depth, heads, mlp_dim, channels=3, dim_head=64):
        super().__init__()
        ih, iw = pair(image_size)
        ph, pw = pair(patch_size)
        assert ih % ph == 0 and iw % pw == 0, 'Image dimensions must be divisible by the patch size.'
        if heads != 1 or dim_head != 64 or mlp_dim != dim:
            raise NotImplementedError('the fused kernel covers the TransCoupling configuration: heads=1, dim_head=64, mlp_dim=dim')
        patch_dim = channels * ph * pw
        self.to_patch_embedding = nn.Sequential(nn.Identity(), nn.LayerNorm(patch_dim), nn.Linear(patch_dim, dim), nn.LayerNorm(dim))
        self.geom = dict(H=ih, W=iw, p1=ph, p2=pw, T=dim, depth=depth, Cin=channels, n_tok=(ih // ph) * (iw // pw), patch_dim=patch_dim)
        self.pos_embedding = posemb_sincos_2d(ih // ph, iw // pw, dim)          # plain tensor, not in the state_dict (App. C-6)
        self.transformer = Transformer(dim, depth, heads, dim_head, mlp_dim)
        self._packs = PackCache()

    def _sources(self):
        pe = self.to_patch_embedding
        srcs = [pe[1].weight, pe[1].bias, pe[2].weight, pe[2].bias, pe[3].weight, pe[3].bias,
                self.transformer.norm.weight, self.transformer.norm.bias]
        for attn, ff in self.transformer.layers:
            srcs += [attn.norm.weight, attn.norm.bias, attn.to_qkv.weight, attn.to_out.weight,
                     ff.net[0].weight, ff.net[0].bias, ff.net[1].weight, ff.net[1].bias, ff.net[3].weight, ff.net[3].bias]
        return srcs

    def _build(self):
        g = self.geom
        dev = self.to_patch_embedding[2].weight.device
        pe = self.to_patch_embedding
        f = lambda t: t.detach().float().contiguous()
        blocks = []
        for attn, ff in self.transformer.layers:
            blocks += [f(attn.norm.weight), f(attn.norm.bias), ops.pack_kmajor(attn.to_qkv.weight, 16).flatten(),
                       ops.pack_kmajor(attn.to_out.weight, 16).flatten(), f(ff.net[0].weight), f(ff.net[0].bias),
                       ops.pack_kmajor(ff.net[1].weight, 16).flatten(), ops.pad_vec(ff.net[1].bias, 16),
                       ops.pack_kmajor(ff.net[3].weight, 16).flatten(), ops.pad_vec(ff.net[3].bias, 16)]
        layers = torch.cat(blocks)
        assert layers.numel() == g['depth'] * int(_cabi.lib().cfpp_vit_layer_floats(g['T']))
        keep = dict(ln0_w=f(pe[1].weight), ln0_b=f(pe[1].bias), pe_wt=ops.pack_kmajor(pe[2].weight, 16), pe_b=ops.pad_vec(pe[2].bias, 16),
                    ln1_w=f(pe[3].weight), ln1_b=f(pe[3].bias), pos=self.pos_embedding.to(dev, torch.float32).contiguous(),
                    lnf_w=f(self.transformer.norm.weight), lnf_b=f(self.transformer.norm.bias), layers=layers)
        d = _cabi.VitDesc()
        for k in ('H', 'W', 'p1', 'p2', 'T', 'depth', 'n_tok', 'patch_dim'):
            setattr(d, k, g[k])
        for k, t in keep.items():
            setattr(d, k, ctypes.c_void_p(t.data_ptr()))
        return d, keep

    def descriptor(self, cin):
        d, _ = self._packs.get('vit', self._sources(), self._build)
        d.Cin = cin
        return d

    def _tc_pack(self):
        """(fp16 hi/lo weight stream, general) of the tensor-core kernels, or None when the shape has no plan.  general=False: one
        64 x 64 chunk per matrix (cfpp_vit_tc_fwd, T <= 64 and tokens dividing 32); True: one chunk per (64-row output block, 64-column
        input block), output block outer (cfpp_vit_tc2_fwd)."""
        g = self.geom
        lib = _cabi.lib()
        T, pd = g['T'], g['patch_dim']
        small = bool(lib.cfpp_vit_tc_supported(T, pd, g['n_tok'], 0))
        if not small and not lib.cfpp_vit_tc2_supported(T, pd, g['n_tok'], 0):
            return None

        def blocks(w, n_out, k_in):
            out = []
            for n0 in range(0, n_out, 64):
                for k0 in range(0, k_in, 64):
                    out.append((w[n0: n0 + 64, k0: k0 + 64], min(64, n_out - n0), min(64, k_in - k0)))
            return out

        def build():
            mats = blocks(self.to_patch_embedding[2].weight, T, pd)
            for attn, ff in self.transformer.layers:
                mats += blocks(attn.to_qkv.weight, 192, T) + blocks(attn.to_out.weight, T, 64)
                mats += blocks(ff.net[1].weight, T, T) + blocks(ff.net[3].weight, T, T)
            if not small:
                assert len(mats) == int(lib.cfpp_vit_tc2_chunks(T, pd, g['depth']))
            return ops.vit_tc_pack(mats), not small
        return self._packs.get('tc', self._sources(), build)

    def forward(self, img, extra=None):
        """img (B, channels, H, W) [or (B, channels - extra.shape[1], H, W) plus per-sample constant channels `extra`]."""
        g = self.geom
        cextra = 0 if extra is None else extra.shape[1]
        cout = g['T'] // (g['p1'] * g['p2'])
        if extra is None and img.is_cuda:
            pk = self._tc_pack()
            if pk is not None:
                return ops.vit_cond_tc(img, self.descriptor(g['Cin']), pk[0], cout, general=pk[1])
        return ops.vit_cond(img, self.descriptor(g['Cin'] - cextra), cout, extra)
