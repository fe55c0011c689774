"""Time the GEMM variants of one cross-modal layer at the cfg-2 shapes (M = 4416 rows, two weight groups) in isolation:
plain epilogues against the LayerNorm-folding ones (statistics + dual output, VI_LN_FOLD, VI_LN_RESIDUAL), bf16 and fp16.
CUDA events around N back-to-back launches (PDL overlaps consecutive launches as in a graph replay)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vln_imagine_b200 import _lib, ops  # noqa: E402

dev = torch.device('cuda')
ops.ensure_init(torch.zeros(1, device=dev))
M, ends = 4416, [2048, 4416]
fmt = torch.float16 if '--f16' in sys.argv else torch.bfloat16
reps = 40


def timeit(fn):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    torch.cuda._sleep(2_000_000)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


g = torch.Generator().manual_seed(0)
R = lambda *s: torch.randn(*s, generator=g).to(dev)   # noqa: E731
x16 = R(M, 768).to(fmt)
h16 = R(M, 3072).to(fmt)
res = R(M, 768)
stats = torch.zeros(24, M, 2, device=dev)
stats[:, :, 1] = 32.0
stats_o = torch.empty(24, M, 2, device=dev)
z32 = torch.empty(M, 768, device=dev)
z16 = torch.empty(M, 768, device=dev, dtype=fmt)
gam = torch.ones(2 * 768, device=dev)
out = {}
for name, N, K, xin in (('proj768', 768, 768, x16), ('qkv2304', 2304, 768, x16), ('ffn1_3072', 3072, 768, x16), ('ffn2_k3072', 768, 3072, h16)):
    w = (R(2 * N, K) * 0.05).to(fmt)
    b = R(2 * N) * 0.1
    s = w.float().sum(1)
    rec = {}
    tiles = [0] if '--tiles' not in sys.argv else [64, 96, 128, 192, 256, 128 | 0x1000, 192 | 0x1000, 256 | 0x1000]
    for tile in tiles:
        if tile and N % (tile & 0xFFF):
            continue
        tt = tile or None                                  # 0: the measured table / cost model
        t = {}
        if N == 768:
            t['f32+res'] = timeit(lambda: ops.gemm(xin, w, b, residual=res, out=z32, group_row_end=ends, tile=tt))
            t['f32+res+stats+dual'] = timeit(lambda: ops.gemm(xin, w, b, residual=res, out=z32, out16=z16, group_row_end=ends, tile=tt, stats_out=stats_o))
            t['f32+lnres+stats+dual'] = timeit(lambda: ops.gemm(xin, w, b, residual=res, out=z32, out16=z16, group_row_end=ends, tile=tt, stats_out=stats_o,
                                                              ln=(_lib.LN_RESIDUAL, gam, stats, 1e-12)))
            t['f32+res+dual'] = timeit(lambda: ops.gemm(xin, w, b, residual=res, out=z32, out16=z16, group_row_end=ends, tile=tt))
        if K == 768:
            y = torch.empty(M, N, device=dev, dtype=fmt)
            epi = 1 if N == 3072 else 0
            t['h16'] = timeit(lambda: ops.gemm(xin, w, b, epilogue=epi, out=y, group_row_end=ends, tile=tt))
            t['h16+fold'] = timeit(lambda: ops.gemm(xin, w, b, epilogue=epi, out=y, group_row_end=ends, tile=tt, ln=(_lib.LN_FOLD, s, stats, 1e-12)))
            if epi:
                t['h16_noact'] = timeit(lambda: ops.gemm(xin, w, b, epilogue=0, out=y, group_row_end=ends, tile=tt))
        rec[str(tile)] = {k: round(v, 2) for k, v in t.items()}
    out[name] = rec
    print(name, json.dumps(rec), flush=True)
ln_in = R(M, 768)
t_ln = timeit(lambda: ops.add_ln(ln_in, None, gam.view(2, 768), gam.view(2, 768), 1e-12, want16=True, group_row_end=ends))
print('add_ln', round(t_ln, 2))
