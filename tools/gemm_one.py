"""Launch one GEMM shape a few times (for ncu).  Usage: python tools/gemm_one.py M N K tile epi res f32 [fold]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vln_imagine_b200 import ops  # noqa: E402

M, N, K = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
tile = sys.argv[4] if len(sys.argv) > 4 else 'auto'
epi = int(sys.argv[5]) if len(sys.argv) > 5 else 0
res = int(sys.argv[6]) if len(sys.argv) > 6 else 0
f32 = int(sys.argv[7]) if len(sys.argv) > 7 else 0
tile = None if tile == 'auto' else int(tile.rstrip('p')) | (ops.TILE_PAIR if tile.endswith('p') else 0)
ops.ensure_init(torch.zeros(1, device='cuda'))
x = torch.randn(M, K, device='cuda').bfloat16()
w = (torch.randn(N, K, device='cuda') * 0.05).bfloat16()
b = torch.randn(N, device='cuda')
r = torch.randn(M, N, device='cuda') if res else None
out = torch.empty(M, N, dtype=torch.float32 if f32 else torch.bfloat16, device='cuda')
fold = int(sys.argv[8]) if len(sys.argv) > 8 else 0
ln = None
if fold:
    from vln_imagine_b200 import _lib
    stats = torch.zeros(K // 32, M, 2, device='cuda')
    stats[:, :, 1] = 32.0
    ln = (_lib.LN_FOLD, w.float().sum(1), stats, 1e-12)
for _ in range(5):
    ops.gemm(x, w, b, residual=r, epilogue=epi, out=out, ln=ln, tile=tile)
torch.cuda.synchronize()
print('ok')
