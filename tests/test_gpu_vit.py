"""SimpleViT conditioner kernels (reference layers/simple_vit.py:43-127 as used by TransCoupling, coupling.py:100-148) against a float64
restatement in torch."""
import pytest
import torch
import torch.nn.functional as F

from contextflow_b200 import synth
from contextflow_b200.layers.simple_vit import SimpleViT

pytestmark = pytest.mark.gpu
dev = 'cuda'


def _vit(H, W, p1, p2, T, depth, cin, tag):
    m = SimpleViT(image_size=(H, W), patch_size=(p1, p2), dim=T, depth=depth, heads=1, mlp_dim=T, channels=cin)
    sd = m.state_dict()
    synth.fill_state(sd, tag)
    m.load_state_dict(sd)
    return m.to(dev).eval()


def _ref64(m, img):
    g = m.geom
    T, p1, p2 = g['T'], g['p1'], g['p2']
    x = img.double()
    B, C, H, W = x.shape
    h, w = H // p1, W // p2
    x = x.reshape(B, C, h, p1, w, p2).permute(0, 2, 4, 3, 5, 1).reshape(B, h * w, p1 * p2 * C)      # b c (h p1) (w p2) -> b (h w) (p1 p2 c)
    pe = m.to_patch_embedding
    D = lambda t: t.detach().double()
    x = F.layer_norm(x, (x.shape[-1],), D(pe[1].weight), D(pe[1].bias))
    x = x @ D(pe[2].weight).T + D(pe[2].bias)
    x = F.layer_norm(x, (T,), D(pe[3].weight), D(pe[3].bias))
    x = x + m.pos_embedding.double().to(x.device)
    for attn, ff in m.transformer.layers:
        y = F.layer_norm(x, (T,), D(attn.norm.weight), D(attn.norm.bias))
        q, k, v = (y @ D(attn.to_qkv.weight).T).chunk(3, -1)
        a = torch.softmax(q @ k.transpose(-1, -2) * 0.125, -1)
        x = x + (a @ v) @ D(attn.to_out.weight).T
        y = F.layer_norm(x, (T,), D(ff.net[0].weight), D(ff.net[0].bias))
        y = F.gelu(y @ D(ff.net[1].weight).T + D(ff.net[1].bias))
        x = x + y @ D(ff.net[3].weight).T + D(ff.net[3].bias)
    x = F.layer_norm(x, (T,), D(m.transformer.norm.weight), D(m.transformer.norm.bias))
    cout = T // (p1 * p2)
    return x.reshape(B, h, w, p1, p2, cout).permute(0, 5, 1, 3, 2, 4).reshape(B, cout, H, W)


# (H, W, p1, p2, T, depth, Cin): the six cfg3 (ATM) conditioners, the SMD one, two small ATM ones, shapes that exercise two operand
# panels with a token count that does not divide the tile, and the widest tile (T = 192, one 128-token sample)
GEOMS = [(18, 1, 2, 1, 152, 6, 38), (36, 1, 2, 1, 152, 6, 38), (72, 1, 2, 1, 152, 6, 38), (76, 1, 2, 1, 36, 6, 9), (76, 1, 2, 1, 72, 6, 18),
         (76, 1, 2, 1, 144, 6, 36), (8, 1, 2, 1, 76, 6, 19), (12, 1, 2, 1, 16, 6, 4), (10, 2, 2, 2, 128, 2, 16), (14, 6, 2, 2, 64, 1, 8),
         (100, 1, 1, 1, 64, 2, 8), (128, 1, 2, 1, 96, 1, 6), (256, 1, 2, 1, 192, 2, 40)]


@pytest.mark.parametrize('geom', GEOMS)
@pytest.mark.parametrize('B', [1, 7, 301])
def test_vit_general_kernels_match_fp64(geom, B):
    H, W, p1, p2, T, depth, cin = geom
    tag = f'vit{H}.{W}.{T}.{cin}'
    m = _vit(H, W, p1, p2, T, depth, cin, tag)
    x = (synth.uniform(tag + f'x{B}', (B, cin, H, W)) * 2.0 - 1.0).to(dev)
    want = _ref64(m, x)
    scale = max(1.0, float(want.abs().max()))
    with torch.no_grad():
        got = m(x)
    torch.cuda.synchronize()
    err = (got.double() - want).abs().max().item()
    assert err <= 2e-5 * scale, f'{geom} B={B}: max abs err {err:.3e} (scale {scale:.3f})'


def test_vit_strided_half_view(monkeypatch):
    """TransCoupling hands the conditioner x[:, :C/2] of a (B, C, H, W) tensor: the kernel reads it through the batch stride."""
    H, W, p1, p2, T, depth, cin = 36, 1, 2, 1, 152, 2, 38
    m = _vit(H, W, p1, p2, T, depth, cin, 'vit_half')
    full = (synth.uniform('vit_half_x', (33, 2 * cin, H, W)) * 2.0 - 1.0).to(dev)
    want = _ref64(m, full[:, :cin])
    with torch.no_grad():
        got = m(full[:, :cin])
    assert (got.double() - want).abs().max().item() <= 2e-5 * max(1.0, float(want.abs().max()))
