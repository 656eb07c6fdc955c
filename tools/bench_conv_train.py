"""Micro-benchmark of the training-direction convolution family at the cfg2 shapes (run under gpurun): per shape the time of
conv2d_fwd / conv2d_bwd_data / conv2d_bwd_weight with the specialised routes on (default) and off (CFPP_BWD_DATA3=0, CFPP_CONV_ROWS=0)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from contextflow_b200 import ops

B = int(os.environ.get('B', 8192))
dev = 'cuda'


REPS, WARM = int(os.environ.get('REPS', 10)), int(os.environ.get('WARM', 3))
ONLY = os.environ.get('ONLY', '')              # e.g. ONLY=k3: the 3x3 shapes only
VARIANTS = [v for v in os.environ.get('VARIANTS', 'new,old').split(',') if v]
ENV = {'new': {}, 'old': {'CFPP_BWD_DATA3': '0', 'CFPP_CONV_ROWS': '0'}}


def timeit(fn, n=REPS):
    for _ in range(WARM): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


SHAPES = [  # (Cin, Cout, H, W, K)  conditioner C1 / C2 / C3 per level, then the encoder-flow FC / CouplingFC layers
    (8, 32, 16, 16, 1), (32, 32, 16, 16, 3), (32, 16, 16, 16, 1),
    (16, 64, 8, 8, 1), (64, 64, 8, 8, 3), (64, 32, 8, 8, 1),
    (32, 128, 4, 4, 1), (128, 128, 4, 4, 3), (128, 64, 4, 4, 1),
    (20, 20, 1, 1, 1), (10, 40, 1, 1, 1), (40, 40, 1, 1, 1), (40, 20, 1, 1, 1),
]
for cin, cout, H, W, K in SHAPES:
    x = torch.randn(B, cin, H, W, device=dev); w = torch.randn(cout, cin, K, K, device=dev) * 0.1; b = torch.randn(cout, device=dev)
    g = torch.randn(B, cout, H, W, device=dev)
    row = {'shape': f'{cin}->{cout} {H}x{W} k{K}'}
    if ONLY and ONLY not in row['shape']:
        continue
    for tag in VARIANTS:
        env = ENV[tag]
        os.environ.update(env)
        if not ONLY:
            row[f'fwd_{tag}_us'] = round(timeit(lambda: ops.conv2d_fwd(x, cin, w, b, relu=True)), 1)
        row[f'bwd_data_{tag}_us'] = round(timeit(lambda: ops.conv2d_bwd_data(g, w, act=x)), 1)
        if tag == 'new' and not ONLY:
            row['bwd_weight_us'] = round(timeit(lambda: ops.conv2d_bwd_weight(x, cin, g, tuple(w.shape))), 1)
        for k in env: del os.environ[k]
    fl = 2.0 * B * cin * cout * K * K * H * W
    row[f'bwd_data_{VARIANTS[0]}_TFLOPps'] = round(fl / row[f'bwd_data_{VARIANTS[0]}_us'] / 1e6, 2)
    print(json.dumps(row), flush=True)
