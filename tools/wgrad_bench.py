"""Time vi_wgrad16 (dW = dY^T X, db = column sums of dY; MN-major tcgen05 operands, split contraction) at the cfg-4 shapes in
isolation, next to cuBLAS on the same contraction (torch.matmul of the transposed view) and to the old path's pieces (two
vi_transpose + vi_gemm16 + vi_colsum).  CUDA events around back-to-back launches.   python tools/wgrad_bench.py [--splits]"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vln_imagine_b200 import _lib, ops  # noqa: E402
from vln_imagine_b200._lib import check, lib  # noqa: E402

dev = torch.device('cuda')
ops.ensure_init(torch.zeros(1, device=dev))
reps = 30


def timeit(fn):
    for _ in range(4):
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


def wgrad_raw(dy, x, bounds, splits, ws, dW, db):
    G = len(bounds)
    check(lib.vi_wgrad16(dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0), ops._DT[dy.dtype], dy.shape[1], x.shape[1], G,
                         _lib.int_array(bounds), dW.data_ptr(), db.data_ptr(), ws.data_ptr(), ws.numel(), splits, 0, ops._stream()), 'vi_wgrad16')


g = torch.Generator().manual_seed(0)
R = lambda *s: torch.randn(*s, generator=g).to(dev)   # noqa: E731
ws = torch.empty(1 << 26, device=dev)
for name, M, ends, N, K in (('nav proj 768x768', 4416, [2048, 4416], 768, 768), ('nav qkv 2304x768', 4416, [2048, 4416], 2304, 768),
                            ('nav ffn1 3072x768', 4416, [2048, 4416], 3072, 768), ('nav ffn2 768x3072', 4416, [2048, 4416], 768, 3072),
                            ('pano proj 768x768', 2304, None, 768, 768), ('pano ffn1 3072x768', 2304, None, 3072, 768),
                            ('ctx kv 3072x768', 5440, None, 3072, 768)):
    dy, x = (R(M, N) * 0.5).bfloat16(), R(M, K).bfloat16()
    bounds = ends or [M]
    G = len(bounds)
    rows = _lib.int_array([b - (bounds[i - 1] if i else 0) for i, b in enumerate(bounds)])
    S0 = int(_lib.lib.vi_wgrad16_splits(N, K, G, rows))
    dW, db = torch.empty(G * N, K, device=dev), torch.empty(G * N, device=dev)
    rec = {'gflop': round(2e-9 * M * N * K, 1), 'auto_splits': S0}
    cand = sorted({S0, 1, 2, 3, 4, 6, 8, 12}) if '--splits' in sys.argv else [S0]
    for S in cand:
        if S > min(rows[i] for i in range(G)) // 64:
            continue
        rec['wgrad16 S=%d' % S] = round(timeit(lambda: wgrad_raw(dy, x, bounds, S, ws, dW, db)), 2)
    lo = 0
    parts = []
    for b in bounds:
        parts.append((dy[lo:b], x[lo:b]))
        lo = b
    rec['cublas bf16 (no bias grad)'] = round(timeit(lambda: [a.t() @ c for a, c in parts]), 2)
    rec['old: 2 transposes + gemm + colsum'] = round(timeit(lambda: [(ops.gemm(ops.transpose(a, ops.pad64(a.shape[0])), ops.transpose(c, ops.pad64(a.shape[0])),
                                                                       None, out_dtype=torch.float32), ops.colsum(a)) for a, c in parts]), 2)
    rec['TF/s'] = round(rec['gflop'] / rec['wgrad16 S=%d' % S0] * 1e3, 1)
    print(name, json.dumps(rec), flush=True)
