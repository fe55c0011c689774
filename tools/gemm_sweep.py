"""Time every GEMM shape of the DUET cfg-2 / HAMT cfg-3 step in isolation, for each tile width the kernel offers.
Usage: python tools/gemm_sweep.py [bn ...]   (default: auto 64 128 256)"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vln_imagine_b200 import ops  # noqa: E402

ops.ensure_init(torch.zeros(1, device='cuda'))
# (name, M, N, K, groups(row ends) or None, epilogue, residual, out fp32)
SHAPES = [
    ('pano.img_linear', 2304, 768, 768, None, 0, False, True),
    ('pano.qkv', 2304, 2304, 768, None, 0, False, False),
    ('pano.o', 2304, 768, 768, None, 0, True, True),
    ('pano.ffn1', 2304, 3072, 768, None, 1, False, False),
    ('pano.ffn2', 2304, 768, 3072, None, 0, True, True),
    ('nav.kv', 5440, 3072, 768, None, 0, False, False),
    ('nav.q', 4416, 768, 768, [2048, 4416], 0, False, False),
    ('nav.o', 4416, 768, 768, [2048, 4416], 0, True, True),
    ('nav.qkv', 4416, 2304, 768, [2048, 4416], 0, False, False),
    ('nav.ffn1', 4416, 3072, 768, [2048, 4416], 1, False, False),
    ('nav.ffn2', 4416, 768, 3072, [2048, 4416], 0, True, True),
    ('nav.head', 4416, 768, 768, [2048, 4416], 2, False, True),
    ('hamt.x_qkv', 9024, 2304, 768, None, 0, False, False),
    ('hamt.ffn1', 9024, 3072, 768, [5632, 9024], 1, False, False),
    ('hamt.ffn2', 9024, 768, 3072, [5632, 9024], 0, True, True),
    ('lang.ffn1', 5120, 3072, 768, None, 1, False, False),
]
tiles = sys.argv[1:] or ['auto', '96', '128', '192', '256', '128p', '192p', '256p']
rows = []
REP = 20
for name, M, N, K, ends, epi, res, f32 in SHAPES:
    ng = 1 if ends is None else len(ends)
    x = torch.randn(M, K, device='cuda').bfloat16()
    w = (torch.randn(ng * N, K, device='cuda') * 0.05).bfloat16()
    b = torch.randn(ng * N, device='cuda')
    r = torch.randn(M, N, device='cuda') if res else None
    out = torch.empty(M, N, dtype=torch.float32 if f32 else torch.bfloat16, device='cuda')
    rec = {'name': name, 'M': M, 'N': N, 'K': K, 'gflop': round(2.0 * M * N * K / 1e9, 2)}
    for tile in tiles:
        tv = None
        if tile != 'auto':
            if N % int(tile.rstrip('p')):
                continue
            tv = int(tile.rstrip('p')) | (ops.TILE_PAIR if tile.endswith('p') else 0)
        for _ in range(3):
            ops.gemm(x, w, b, residual=r, epilogue=epi, out=out, group_row_end=ends, tile=tv)
        torch.cuda.synchronize()
        torch.cuda._sleep(3_000_000)                   # let the host run ahead so launches queue back to back
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(REP):
            ops.gemm(x, w, b, residual=r, epilogue=epi, out=out, group_row_end=ends, tile=tv)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / REP
        rec[tile] = '%.1fus %.0fTF' % (t * 1e3, rec['gflop'] / t)
    # yardstick only (never on the product path): cuBLAS on the same shape, no epilogue
    xs = x if ends is None else x[:ends[0]]
    wt = w[:N].t()
    for _ in range(3):
        torch.matmul(x, wt)
    torch.cuda.synchronize()
    torch.cuda._sleep(3_000_000)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REP):
        torch.matmul(x, wt)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / REP
    rec['cublas_plain'] = '%.1fus %.0fTF' % (t * 1e3, rec['gflop'] / t)
    rows.append(rec)
    print(json.dumps(rec), flush=True)
