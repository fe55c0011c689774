"""Thin tensor-level wrappers over the C ABI (include/vlnimagine.h): the only module that calls the library.

PyTorch is used for device memory and streams only: every function here validates its tensors,
allocates the output with torch.empty and calls one libvlnimagine entry point on the current
stream.  Nothing falls back to ATen arithmetic.
"""
from __future__ import annotations

import os
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import EPI_NONE, EPI_GELU, EPI_RELU, MASK_ADD_NEG10000, MASK_NEG_INF, LN_FOLD, LN_RESIDUAL  # noqa: F401

HIDDEN = 768
HEADS = 12
BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
_DT = {BF16: _lib.DT_BF16, F16: _lib.DT_F16, F32: _lib.DT_F32}


class _Half:
    """The 16-bit operand format new activations / weight shadows are created in: bf16, or fp16 for inference on tensors
    whose range the host has bounded (blocks.half_format_for).  Training always runs bf16."""
    dtype = BF16


class half_format:
    """with ops.half_format(torch.float16): ...   (set by the host modules once per mode call)"""

    def __init__(self, dtype):
        if dtype not in (BF16, F16):
            raise _lib.VlnImagineError('the 16-bit operand format must be torch.bfloat16 or torch.float16')
        self.dtype = dtype

    def __enter__(self):
        self.prev = _Half.dtype
        _Half.dtype = self.dtype

    def __exit__(self, *a):
        _Half.dtype = self.prev


def h16():
    return _Half.dtype


def is16(dtype) -> bool:
    return dtype in (BF16, F16)


class _LaunchCounters:
    """Kernel launches of the process (bench.py reports them as gpu_launches): the library's own count plus
    ``other_launches``, the kernels the package issues outside it; and optional per-launch CUDA-event traces: of the
    tensor-core GEMMs with their shape (bench.py's roofline leg) and of every library entry point by name (bench.py's
    per-kernel breakdown)."""
    other_launches = 0
    gemm_trace = None          # list of (M, N, K, start_event, end_event) when enabled
    trace = None               # list of (entry point, start_event, end_event) when enabled

    @property
    def launches(self) -> int:
        return _lib.lib.vi_launch_count() + self.other_launches


_Counters = _LaunchCounters()


def _timed(trace, tag, fn, *a):
    """fn(*a); while ``trace`` is a list, bracketed by a CUDA event pair appended to it as (*tag, start, end)"""
    if trace is None:
        return fn(*a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn(*a)
    e1.record()
    trace.append((*tag, e0, e1))
    return r


class _Lib:
    """The ctypes library.  A call of an entry point raises VlnImagineError unless it returns VI_OK (the value queries of
    _lib.QUERIES return their result) and is traced while _Counters.trace is a list."""

    def __getattr__(self, name):
        fn = getattr(_lib.lib, name)
        if name in _lib.QUERIES:
            call = fn
        else:
            def call(*a):
                tr = _Counters.trace
                rc = fn(*a) if tr is None else _timed(tr, (name,), fn, *a)
                if rc:
                    raise _lib.failure(rc, name)
        setattr(self, name, call)
        return call


lib = _Lib()


def _stream():
    return torch.cuda.current_stream().cuda_stream


_initialised = set()


def ensure_init(t: torch.Tensor):
    """vi_init once per device (selects it, checks sm_100, raises shared-memory limits)"""
    if not t.is_cuda:
        raise _lib.VlnImagineError('tensor must be a CUDA tensor: vln-imagine_b200 has no CPU path')
    index = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if index not in _initialised:
        lib.vi_init(index)
        _initialised.add(index)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _groups(group_row_end: Optional[Sequence[int]]):
    """(n_groups, host int32 array of the group ends or None) of a grouped entry point"""
    if group_row_end is None:
        return 1, None
    return len(group_row_end), _lib.int_array(list(group_row_end))


_WORKSPACE = {}
RED_CHUNK = 128             # rows per partial of the library's two-stage column reductions


def _red_floats(rows: int, cols: int, n_out: int) -> int:
    return n_out * ((rows + RED_CHUNK - 1) // RED_CHUNK) * cols


def workspace(device, floats: int) -> torch.Tensor:
    """fp32 scratch of the multi-pass entry points (column reduction partials, split weight-gradient partials): one per
    device, at least 2^23 floats, grown on demand.  Every user launches on the current stream, which orders the launches
    that share it."""
    t = _WORKSPACE.get(device)
    if t is None or t.numel() < floats:
        t = _WORKSPACE[device] = torch.empty((max(floats, 1 << 23),), dtype=F32, device=device)
    return t


def _rows2d(t: torch.Tensor, name: str):
    if t.dim() != 2 or t.stride(1) != 1:
        raise _lib.VlnImagineError('%s must be a 2-D row-major view (got shape %s strides %s)' % (name, tuple(t.shape), t.stride()))
    return t.shape[0], t.shape[1], t.stride(0)


def pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def pad128(n: int) -> int:
    return (n + 127) // 128 * 128


ROW_ALIGN = 256     # streams of a row-stacked activation start on 256-row boundaries: a CTA-pair GEMM tile
                    # (256 rows) then never straddles two weight groups


def pad_rows(n: int) -> int:
    return (n + ROW_ALIGN - 1) // ROW_ALIGN * ROW_ALIGN


TILE_PAIR = 0x1000
_TILE_CANDIDATES = [256 | TILE_PAIR, 192 | TILE_PAIR, 128 | TILE_PAIR, 256, 192, 128, 96, 64]
_TILE_CACHE = {}           # GEMM signature -> tile code, filled by timing the candidates on first use
_TILE_TABLE_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'tile_table.json')


def _key_str(key):
    return repr(key[:-1])      # the device index is not part of the persisted signature


def load_tile_table(path: str = _TILE_TABLE_PATH):
    """Tile choices measured on a B200 by tools/tune_tiles.py; shapes not listed are tuned on first use."""
    import json
    try:
        with open(path) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


_TILE_TABLE = load_tile_table()


def autotune_enabled() -> bool:
    """Timing tile candidates on first use is OFF by default: shapes missing from tile_table.json use the library's cost
    model, so results and timings are reproducible from process to process and a rollout never stalls on a tuning pass.
    tools/tune_tiles.py (VLN_IMAGINE_AUTOTUNE=1) measures new shapes and rewrites the table."""
    return os.environ.get('VLN_IMAGINE_AUTOTUNE', '0') == '1'


def _table_tile(key) -> int:
    """tile from the measured table: the exact signature, else the same shape without the LayerNorm / dual-output flags"""
    for k in (key, key[:8] + key[-1:]):
        ks = _key_str(k)
        if ks in _TILE_TABLE:
            return int(_TILE_TABLE[ks])
    return 0


def _tune_tile(key, launch, N: int, pair_ok: bool) -> int:
    """Time every admissible tile shape for this GEMM signature (CUDA events, back-to-back launches) and remember
    the fastest.  Skipped (library cost model) while a CUDA graph is being captured."""
    if key in _TILE_CACHE:
        return _TILE_CACHE[key]
    if os.environ.get('VLN_IMAGINE_RETUNE', '0') == '0':
        t = _table_tile(key)
        if t or not autotune_enabled():
            _TILE_CACHE[key] = t
            return t
    if torch.cuda.is_current_stream_capturing():
        return 0
    best, best_t = 0, float('inf')
    for tile in _TILE_CANDIDATES:
        bn, pair = tile & 0xFFF, bool(tile & TILE_PAIR)
        if N % bn or (pair and not pair_ok):
            continue
        for _ in range(2):
            launch(tile)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        torch.cuda._sleep(400_000)                     # let the host queue the launches back to back
        e0.record()
        for _ in range(6):
            launch(tile)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1)
        if t < best_t:
            best, best_t = tile, t
    _TILE_CACHE[key] = best
    return best


def gemm(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None,
         residual: Optional[torch.Tensor] = None, epilogue: int = EPI_NONE,
         out_dtype: Optional[torch.dtype] = None, group_row_end: Optional[Sequence[int]] = None,
         out: Optional[torch.Tensor] = None, out16: Optional[torch.Tensor] = None, ln=None,
         stats_out: Optional[torch.Tensor] = None, tile: Optional[int] = None) -> torch.Tensor:
    """Y = epi(X W^T + bias) + residual.  x bf16 / fp16 -> tcgen05 kernel (vi_gemm16); x fp32 -> fp32 check-mode kernel.
    w is [n_groups*N, K]; group_row_end (python ints) splits the rows of x between the weight blocks.
    out16: a 16-bit tensor that receives a copy of an fp32 output.  ln = (mode, vec_a, stats, eps): LayerNorm folded into
    this contraction (_lib.LN_FOLD / LN_RESIDUAL, see include/vlnimagine.h); stats_out: float32 [N/32, M, 2] that receives
    the per-chunk row statistics of the output.  tile: the output-tile shape (width | TILE_PAIR, 0 = the library's cost model)
    instead of the measured table / autotuner; a shape the problem does not admit raises."""
    M, K, ldx = _rows2d(x, 'x')
    n_groups = 1 if group_row_end is None else len(group_row_end)
    if w.dim() != 2 or not w.is_contiguous() or w.shape[1] != K or w.shape[0] % n_groups:
        raise _lib.VlnImagineError('weight shape %s does not match x %s / %d groups' % (tuple(w.shape), tuple(x.shape), n_groups))
    N = w.shape[0] // n_groups
    _, ends = _groups(group_row_end)
    ldr = residual.stride(0) if residual is not None else 0
    if is16(x.dtype):
        if w.dtype != x.dtype:
            raise _lib.VlnImagineError('%s GEMM needs a weight of the same type (got %s)' % (x.dtype, w.dtype))
        if out is None:
            out = torch.empty((M, N), dtype=out_dtype or x.dtype, device=x.device)
        if out.dtype != F32 and out.dtype != x.dtype:
            raise _lib.VlnImagineError('GEMM output must be fp32 or the operand type')
        a = _lib.GemmArgs()
        a.x, a.ldx, a.w, a.in_dtype = x.data_ptr(), ldx, w.data_ptr(), _DT[x.dtype]
        a.bias, a.residual, a.ldr = _ptr(bias), _ptr(residual), ldr
        a.y, a.ldy, a.y_dtype = out.data_ptr(), out.stride(0), _DT[out.dtype]
        if out16 is not None:
            if out16.dtype != x.dtype:
                raise _lib.VlnImagineError('the 16-bit output copy must have the operand type')
            a.y16, a.ldy16 = out16.data_ptr(), out16.stride(0)
        a.M, a.N, a.K, a.epilogue, a.n_groups, a.group_row_end = M, N, K, epilogue, n_groups, ends
        ln_mode = 0
        if ln is not None:
            ln_mode, vec_a, stats, eps = ln
            a.ln_mode, a.ln_vec_a, a.ln_stats, a.ln_chunks, a.ln_eps = ln_mode, vec_a.data_ptr(), stats.data_ptr(), stats.shape[0], eps
            a.stats_ld = stats.shape[1]
        if stats_out is not None:
            if stats_out.shape[0] * 32 != N or stats_out.shape[1] < M or (ln is not None and ln[2].shape[1] != stats_out.shape[1]):
                raise _lib.VlnImagineError('stats_out must be [N/32, >=M, 2] with the row stride of the input statistics')
            a.stats_out, a.stats_ld = stats_out.data_ptr(), stats_out.shape[1]
        ge = tuple(group_row_end) if group_row_end is not None else None
        key = (M, N, K, ge, epilogue, bias is not None, residual is not None, 1 if out.dtype == F32 else 0,
               ln_mode, out16 is not None, stats_out is not None, x.device.index)

        def launch(tile):
            a.tile = tile
            lib.vi_gemm16(a, _stream())
        if tile is None:
            pair_ok = ge is None or all(e % 256 == 0 for e in ge[:-1])
            tile = _tune_tile(key, launch, N, pair_ok)
        _timed(_Counters.gemm_trace, (M, N, K), launch, tile)
    elif x.dtype == F32:
        if w.dtype != F32:
            raise _lib.VlnImagineError('fp32 GEMM needs an fp32 weight')
        if ln is not None or out16 is not None or stats_out is not None:
            raise _lib.VlnImagineError('LayerNorm folding exists in the tensor-core kernel only')
        if out is None:
            out = torch.empty((M, N), dtype=F32, device=x.device)
        lib.vi_gemm_f32(x.data_ptr(), ldx, w.data_ptr(), _ptr(bias), _ptr(residual), ldr, out.data_ptr(), out.stride(0), M, N, K,
                        epilogue, n_groups, ends, _stream())
    else:
        raise _lib.VlnImagineError('unsupported GEMM dtype %s' % x.dtype)
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, B: int, Lq: int, Lk: int,
              key_mask: Optional[torch.Tensor] = None, pair_dist: Optional[torch.Tensor] = None,
              bias_affine: Optional[torch.Tensor] = None, mask_mode: int = MASK_ADD_NEG10000,
              out: Optional[torch.Tensor] = None, lse: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q [B*Lq, >=768 view], k/v [B*Lk, view] -> o [B*Lq, 768]; 12 heads of 64.  One problem of attention_multi."""
    if out is None:
        out = torch.empty((B * Lq, HIDDEN), dtype=q.dtype, device=q.device)
    attention_multi([dict(q=q, k=k, v=v, out=out, B=B, Lq=Lq, Lk=Lk, key_mask=key_mask, pair_dist=pair_dist,
                          bias_affine=bias_affine, lse=lse)], mask_mode)
    return out


def attention_multi(problems, mask_mode: int = MASK_ADD_NEG10000):
    """Several attention problems in one launch.  Each problem is a dict with q, k, v (2-D row views), out,
    B, Lq, Lk and optional key_mask (uint8 [B, Lk]), pair_dist, bias_affine, lse."""
    n = len(problems)
    arr = (_lib.AttnProblem * n)()
    dtype = None
    for a, pr in zip(arr, problems):
        q, k, v, o = pr['q'], pr['k'], pr['v'], pr['out']
        _, _, a.ldq = _rows2d(q, 'q')
        _, _, a.ldk = _rows2d(k, 'k')
        _, _, a.ldv = _rows2d(v, 'v')
        a.q, a.k, a.v, a.o, a.ldo = q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), o.stride(0)
        km = pr.get('key_mask')
        if km is not None and (km.dtype != torch.uint8 or not km.is_contiguous()):
            raise _lib.VlnImagineError('key_mask must be a contiguous uint8 tensor')
        a.key_mask, a.pair_dist, a.bias_affine, a.lse = _ptr(km), _ptr(pr.get('pair_dist')), _ptr(pr.get('bias_affine')), _ptr(pr.get('lse'))
        a.B, a.Lq, a.Lk = pr['B'], pr['Lq'], pr['Lk']
        drop = pr.get('drop')                      # (p, site, seed tensor) or None: attention-probability dropout
        if drop is not None and drop[0] > 0:
            a.drop_p, a.drop_site, a.drop_seed = float(drop[0]), int(drop[1]) & 0xFFFFFFFF, drop[2].data_ptr()
        if dtype is None:
            dtype = q.dtype
        elif dtype != q.dtype:
            raise _lib.VlnImagineError('attention problems of one launch must share a dtype')
    lib.vi_attn_fwd_multi(arr, n, HEADS, _DT[dtype], mask_mode, _stream())


def _dt16(t: Optional[torch.Tensor]) -> int:
    return _DT[t.dtype] if t is not None else _lib.DT_BF16


def add_ln(a: torch.Tensor, b: Optional[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor, eps: float,
           want16: bool, want32: bool = True, group_row_end: Optional[Sequence[int]] = None):
    """LayerNorm(a [+ b]); returns (y32 or None, y16 or None)."""
    rows = a.shape[0]
    y32 = torch.empty((rows, HIDDEN), dtype=F32, device=a.device) if want32 else None
    y16 = torch.empty((rows, HIDDEN), dtype=h16(), device=a.device) if want16 else None
    lib.vi_add_ln(a.data_ptr(), _ptr(b), gamma.data_ptr(), beta.data_ptr(), eps, _ptr(y32), _ptr(y16), _dt16(y16), rows,
                  *_groups(group_row_end), _stream())
    return y32, y16


def add_ln_drop(a: torch.Tensor, b: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, dtype16, p: float,
                seed: torch.Tensor, site: int, group_row_end: Optional[Sequence[int]] = None):
    """LayerNorm(dropout(a) + b) with the counter-based mask of ``site`` -> (y32, y16 of ``dtype16``)"""
    rows = a.shape[0]
    y32 = torch.empty((rows, HIDDEN), dtype=F32, device=a.device)
    y16 = torch.empty((rows, HIDDEN), dtype=dtype16, device=a.device)
    lib.vi_add_ln_drop(a.data_ptr(), b.data_ptr(), gamma.data_ptr(), beta.data_ptr(), eps, y32.data_ptr(), y16.data_ptr(), _DT[dtype16],
                       rows, *_groups(group_row_end), float(p), seed.data_ptr(), site, _stream())
    return y32, y16


def add_ln_drop_bwd(a: torch.Tensor, b: Optional[torch.Tensor], gamma: torch.Tensor, eps: float, dy32: Optional[torch.Tensor],
                    dy16: Optional[torch.Tensor], dgamma: torch.Tensor, dbeta: torch.Tensor, accumulate: int,
                    group_row_end: Optional[Sequence[int]] = None, dxa16_dtype=None, drop=None):
    """adjoint of add_ln / add_ln_drop: dy = dy32 (+ dy16) -> (dx32, the gradient of b and, without dropout, of a; dxa16, the
    gradient of a as a 16-bit operand of ``dxa16_dtype``, or None); dgamma / dbeta [n_groups, 768] are overwritten
    (accumulate = 0) or added to (1).  drop = (p, seed tensor, site) of the forward dropout."""
    rows = a.shape[0]
    p, seed, site = drop if drop is not None else (0.0, None, 0)
    dx32 = torch.empty((rows, HIDDEN), dtype=F32, device=a.device)
    dxa16 = torch.empty((rows, HIDDEN), dtype=dxa16_dtype, device=a.device) if dxa16_dtype is not None else None
    stats = torch.empty((rows, 2), dtype=F32, device=a.device)
    ws = workspace(a.device, _red_floats(16 * rows, HIDDEN, 2))    # the fused pass reduces chunks of 8 - 32 rows (>= RED_CHUNK / 16)
    lib.vi_add_ln_drop_bwd(a.data_ptr(), _ptr(b), gamma.data_ptr(), eps, _ptr(dy32), _ptr(dy16), _ptr(dx32), None, _ptr(dxa16),
                           dgamma.data_ptr(), dbeta.data_ptr(), stats.data_ptr(), rows, *_groups(group_row_end), ws.data_ptr(),
                           ws.numel(), accumulate, float(p), _ptr(seed), site, _stream())
    return dx32, dxa16


_feat_wt_provider = None        # blocks installs a cache (transposed copies follow the weight versions like every derived tensor)


def set_feat_wt_provider(fn):
    global _feat_wt_provider
    _feat_wt_provider = fn


def embed_compose(rows: int, device, *, a=None, a2=None, a3=None, a_ln=None, feat=None, feat_w=None, feat_b=None, feat_ln=None,
                  idx=None, table=None, pos_table=None, pos_period=0, const_row=None, const_row2=None,
                  out_ln=None, eps=1e-12, y32=None, y16=None, want16=False, want32=True, ln2=None, ln2_eps=1e-5, zero_rows=0):
    """See vi_embed_compose.  *_ln are (gamma, beta) pairs.  y32 / y16 may be preallocated row views."""
    if y32 is None and want32:
        y32 = torch.empty((rows, HIDDEN), dtype=F32, device=device)
    if y16 is None and want16:
        y16 = torch.empty((rows, HIDDEN), dtype=h16(), device=device)
    args = _lib.EmbedArgs()
    args.a, args.a2, args.a3 = _ptr(a), _ptr(a2), _ptr(a3)
    if a_ln is not None:
        args.a_gamma, args.a_beta = a_ln[0].data_ptr(), a_ln[1].data_ptr()
    if feat is not None:
        args.feat, args.feat_dim = feat.data_ptr(), feat.shape[-1]
        # the kernel reads the weight of the small projection TRANSPOSED ([feat_dim, 768]: coalesced, L1-resident rows per k)
        wt = _feat_wt_provider(feat_w) if _feat_wt_provider is not None else feat_w.detach().t().contiguous().float()
        args.feat_w, args.feat_b = wt.data_ptr(), _ptr(feat_b)
        if feat_ln is not None:
            args.feat_gamma, args.feat_beta = feat_ln[0].data_ptr(), feat_ln[1].data_ptr()
    if idx is not None:
        args.idx, args.table = idx.data_ptr(), table.data_ptr()
    if pos_table is not None:
        args.pos_table, args.pos_period = pos_table.data_ptr(), pos_period
    args.const_row, args.const_row2 = _ptr(const_row), _ptr(const_row2)
    if out_ln is not None:
        args.out_gamma, args.out_beta = out_ln[0].data_ptr(), out_ln[1].data_ptr()
    args.eps = eps
    args.y32, args.y16, args.rows, args.y16_dtype = _ptr(y32), _ptr(y16), rows, _dt16(y16)
    if ln2 is not None:                               # a second LayerNorm chained on the result: y16 = LN2(y32)
        args.ln2_gamma, args.ln2_beta, args.ln2_eps = ln2[0].data_ptr(), ln2[1].data_ptr(), ln2_eps
    args.zero_rows = int(zero_rows)                   # rows behind the last one that the same launch zero-fills (y32 / y16 must cover them)
    lib.vi_embed_compose(args, _stream())
    return y32, y16


def ln_dot(h: torch.Tensor, gamma, beta, eps: float, w, b, group_row_end: Optional[Sequence[int]] = None):
    rows = h.shape[0]
    out = torch.empty((rows,), dtype=F32, device=h.device)
    lib.vi_ln_dot(h.data_ptr(), _ptr(gamma), _ptr(beta), eps, w.data_ptr(), _ptr(b), out.data_ptr(), rows, *_groups(group_row_end),
                  _stream())
    return out


def mul_bcast(x: torch.Tensor, x_batch_stride: int, s: torch.Tensor, s_batch_stride: int, n_batches: int,
              rows_per_batch: int, want16: bool, want32: bool = True):
    """y[b, r] = x[b, r] * s[b] over 768-wide rows; x / s are base views with element batch strides."""
    rows = n_batches * rows_per_batch
    y32 = torch.empty((rows, HIDDEN), dtype=F32, device=x.device) if want32 else None
    y16 = torch.empty((rows, HIDDEN), dtype=h16(), device=x.device) if want16 else None
    lib.vi_mul_bcast(x.data_ptr(), x_batch_stride, s.data_ptr(), s_batch_stride, _ptr(y32), _ptr(y16), _dt16(y16), rows,
                     rows_per_batch, _stream())
    return y32, y16


def duet_fuse_logits(g_raw, l_raw, fuse_raw, gmap_masks_u8, gmap_visited_u8, vp_nav_u8, gmap_ids, cand_ids,
                     B: int, G: int, P: int):
    dev = g_raw.device
    gl = torch.empty((B, G), dtype=F32, device=dev)
    ll = torch.empty((B, P), dtype=F32, device=dev)
    fl = torch.empty((B, G), dtype=F32, device=dev)
    lib.vi_duet_fuse_logits(g_raw.data_ptr(), l_raw.data_ptr(), _ptr(fuse_raw), gmap_masks_u8.data_ptr(), gmap_visited_u8.data_ptr(),
                            vp_nav_u8.data_ptr(), gmap_ids.data_ptr(), cand_ids.data_ptr(), gl.data_ptr(), ll.data_ptr(), fl.data_ptr(),
                            B, G, P, _stream())
    return gl, ll, fl


def mask_logits_navtype(raw: torch.Tensor, nav_types: torch.Tensor):
    out = torch.empty_like(raw)
    lib.vi_mask_logits_navtype(raw.data_ptr(), nav_types.data_ptr(), out.data_ptr(), raw.numel(), _stream())
    return out


def gather_mean(src: torch.Tensor, offsets: torch.Tensor, row_idx: torch.Tensor, R: int, want16: bool, want32: bool = True):
    y32 = torch.empty((R, HIDDEN), dtype=F32, device=src.device) if want32 else None
    y16 = torch.empty((R, HIDDEN), dtype=h16(), device=src.device) if want16 else None
    lib.vi_gather_mean(src.data_ptr(), offsets.data_ptr(), row_idx.data_ptr(), _ptr(y32), _ptr(y16), _dt16(y16), R, _stream())
    return y32, y16


def scatter_rows(src: torch.Tensor, dst_rows: torch.Tensor, dst: torch.Tensor):
    lib.vi_scatter_rows(src.data_ptr(), dst_rows.data_ptr(), dst.data_ptr(), src.shape[0], _stream())
    return dst


def cosine_loss(proj: Optional[torch.Tensor], tgt: Optional[torch.Tensor], R: int, device):
    loss = torch.empty((), dtype=F32, device=device)
    rows = torch.empty((max(R, 1),), dtype=F32, device=device)
    lib.vi_cosine_loss(_ptr(proj), _ptr(tgt), rows.data_ptr(), loss.data_ptr(), R, _stream())
    return loss, rows[:R]


def _contrastive_loss(fn, proj, tgt, negs, row_episode, neg_episode, param: float, R: int, n_negs: int, device):
    loss = torch.empty((), dtype=F32, device=device)
    scratch = torch.empty((max(R, 1) * (n_negs + 2),), dtype=F32, device=device)
    fn(_ptr(proj), _ptr(tgt), _ptr(negs), _ptr(row_episode), _ptr(neg_episode), param, scratch.data_ptr(), loss.data_ptr(), R, n_negs,
       _stream())
    return loss, scratch


def infonce_loss(proj, tgt, negs, row_episode, neg_episode, temperature: float, R: int, n_negs: int, device):
    """(loss, scratch): the forward scratch's first R * (n_negs + 1) floats are the scaled similarities the backward
    pass needs"""
    return _contrastive_loss(lib.vi_infonce_loss, proj, tgt, negs, row_episode, neg_episode, temperature, R, n_negs, device)


def margin_loss(proj, tgt, negs, row_episode, neg_episode, margin: float, R: int, n_negs: int, device):
    """(loss, scratch): the forward scratch's first R * (n_negs + 1) floats are the cosines the backward pass needs"""
    return _contrastive_loss(lib.vi_margin_loss, proj, tgt, negs, row_episode, neg_episode, margin, R, n_negs, device)


def copy_rows(src: torch.Tensor, src_bs: int, src_rs: int, n_batches: int, rows_per_batch: int,
              dst32: Optional[torch.Tensor], dst16: Optional[torch.Tensor], dst_bs: int, dst_rs: int):
    """dst[b, r] = src[b, r] over 768-wide rows with element strides (see vi_copy_rows)."""
    lib.vi_copy_rows(src.data_ptr(), src_bs, src_rs, _ptr(dst32), _ptr(dst16), _dt16(dst16), dst_bs, dst_rs, n_batches,
                     rows_per_batch, _stream())


def cast_h16(src: torch.Tensor, dst: Optional[torch.Tensor] = None, dtype=None):
    """fp32 -> the current 16-bit operand format (or ``dtype`` / the type of ``dst``)"""
    src = src.contiguous()
    if dst is None:
        dst = torch.empty(src.shape, dtype=dtype or h16(), device=src.device)
    lib.vi_cast_h16(src.data_ptr(), dst.data_ptr(), _DT[dst.dtype], src.numel(), _stream())
    return dst


def gather_rows(store: torch.Tensor, idx: torch.Tensor, dtype, drop=None) -> torch.Tensor:
    """rows of a device feature store: out[r] = store[idx[r]] (zero row for an index outside the store) as a dense
    [idx.numel(), F] tensor of ``dtype`` (fp32, or a 16-bit GEMM operand format); drop = (p, seed tensor, site): the mask and
    product of ``dropout`` on the dense fp32 rows (vi_gather_rows)"""
    n_store, F, ld = _rows2d(store, 'store')
    if idx.dtype != torch.int32:
        raise _lib.VlnImagineError('feature row indices must be int32 (got %s)' % idx.dtype)
    idx = idx.to(store.device, non_blocking=True).contiguous()
    out = torch.empty((idx.numel(), F), dtype=dtype, device=store.device)
    d32, d16 = (out, None) if dtype == F32 else (None, out)
    p, seed, site = drop if drop is not None else (0.0, None, 0)
    lib.vi_gather_rows(store.data_ptr(), _DT[store.dtype], ld, n_store, idx.data_ptr(), idx.numel(), F, _ptr(d32), _ptr(d16),
                       _dt16(d16), float(p), _ptr(seed), int(site) & 0xFFFFFFFF, _stream())
    return out


def ce_rows(logits: torch.Tensor, labels: torch.Tensor, n_cols: int) -> torch.Tensor:
    """per-row cross-entropy over the first n_cols columns of fp32 logits [R, ld] (F.cross_entropy, reduction='none')"""
    R, _, ld = _rows2d(logits, 'logits')
    out = torch.empty((R,), dtype=F32, device=logits.device)
    lib.vi_ce_rows(logits.data_ptr(), ld, labels.long().contiguous().data_ptr(), n_cols, out.data_ptr(), R, _stream())
    return out


def kl_rows(logits: torch.Tensor, targets: torch.Tensor, n_cols: int) -> torch.Tensor:
    """per-row KL(targets || softmax(logits)) over the first n_cols columns (F.kl_div(log_softmax, targets, 'none').sum(1))"""
    R, _, ld = _rows2d(logits, 'logits')
    _, _, ldt = _rows2d(targets, 'targets')
    out = torch.empty((R,), dtype=F32, device=logits.device)
    lib.vi_kl_rows(logits.data_ptr(), ld, targets.data_ptr(), ldt, n_cols, out.data_ptr(), R, _stream())
    return out


def _xent_out(R: int, ld_out: int, dtype, device):
    out = torch.empty((R, ld_out), dtype=dtype, device=device)
    return (out, None) if dtype == F32 else (None, out)


def ce_rows_bwd(logits: torch.Tensor, labels: torch.Tensor, n_cols: int, dloss: torch.Tensor, dtype=F32,
                ld_out: Optional[int] = None) -> torch.Tensor:
    """gradient of ce_rows w.r.t. the logits: dloss[r] * (softmax(logits[r, :n_cols]) - one_hot(labels[r])) as [R, ld_out] rows of
    ``dtype`` (fp32, or the 16-bit operand of the gradient GEMMs); columns n_cols .. ld_out - 1 (default: the logits' width) are 0"""
    R, W, ld = _rows2d(logits, 'logits')
    d32, d16 = _xent_out(R, ld_out or W, dtype, logits.device)
    dloss = dloss.float().contiguous()
    lib.vi_ce_rows_bwd(logits.data_ptr(), ld, labels.long().contiguous().data_ptr(), n_cols, dloss.data_ptr(), _ptr(d32), _ptr(d16),
                       _dt16(d16), ld_out or W, R, _stream())
    return d32 if d32 is not None else d16


def kl_rows_bwd(logits: torch.Tensor, targets: torch.Tensor, n_cols: int, dloss: torch.Tensor, dtype=F32,
                ld_out: Optional[int] = None) -> torch.Tensor:
    """gradient of kl_rows w.r.t. the logits: dloss[r] * (softmax(logits[r, :n_cols]) * sum(targets[r]) - targets[r]), laid out as
    in ce_rows_bwd"""
    R, W, ld = _rows2d(logits, 'logits')
    _, _, ldt = _rows2d(targets, 'targets')
    d32, d16 = _xent_out(R, ld_out or W, dtype, logits.device)
    dloss = dloss.float().contiguous()
    lib.vi_kl_rows_bwd(logits.data_ptr(), ld, targets.data_ptr(), ldt, n_cols, dloss.data_ptr(), _ptr(d32), _ptr(d16),
                       _dt16(d16), ld_out or W, R, _stream())
    return d32 if d32 is not None else d16


# ----------------------------------------------------------------------------------------------
# backward-pass entry points (the autograd nodes of autograd_ops call these)
def transpose(src: torch.Tensor, pad_rows: Optional[int] = None) -> torch.Tensor:
    """[rows, cols] view -> [cols, pad_rows] (zero padded columns)"""
    rows, cols = src.shape
    pr = pad_rows or rows
    dst = torch.empty((cols, pr), dtype=src.dtype, device=src.device)
    lib.vi_transpose(src.data_ptr(), src.stride(0), dst.data_ptr(), dst.stride(0), rows, cols, pr, _DT[src.dtype], _stream())
    return dst


def colsum(x: torch.Tensor) -> torch.Tensor:
    rows, cols = x.shape
    out = torch.empty((cols,), dtype=F32, device=x.device)
    ws = workspace(x.device, _red_floats(rows, cols, 1))
    lib.vi_colsum(x.data_ptr(), x.stride(0), _DT[x.dtype], out.data_ptr(), rows, cols, ws.data_ptr(), ws.numel(), _stream())
    return out


def wgrad16_ok(dy16: torch.Tensor, x16: torch.Tensor) -> bool:
    return (is16(dy16.dtype) and x16.dtype == dy16.dtype and dy16.shape[1] % 128 == 0 and x16.shape[1] % 64 == 0
            and dy16.stride(1) == 1 and x16.stride(1) == 1 and dy16.stride(0) % 8 == 0 and x16.stride(0) % 8 == 0
            and dy16.data_ptr() % 16 == 0 and x16.data_ptr() % 16 == 0)


def wgrad16(dy16: torch.Tensor, x16: torch.Tensor, ends, want_db: bool, out=None, accumulate: int = 0):
    """(dW [n_groups * N, K] fp32, db [n_groups * N] fp32 or None) of a (grouped) dense layer from the 16-bit row-major dY [M, N]
    and X [M, K] as they are (vi_wgrad16: MN-major tcgen05 operands, no transposed copies, bias gradient on the tensor cores,
    the library's choice of split).  out = (dW, db) preallocated; accumulate = 1 adds to them."""
    M, N = dy16.shape
    K = x16.shape[1]
    bounds = [min(int(e), M) for e in ends] if ends is not None else [M]
    G = len(bounds)
    rows = _lib.int_array([b - (bounds[i - 1] if i else 0) for i, b in enumerate(bounds)])
    ws = workspace(dy16.device, lib.vi_wgrad16_workspace(N, K, G, rows, 0))
    if out is not None:
        dW, db = out
    else:
        dW = torch.empty((G * N, K), dtype=F32, device=dy16.device)
        db = torch.empty((G * N,), dtype=F32, device=dy16.device) if want_db else None
    _timed(_Counters.gemm_trace, (bounds[-1], N, K), lib.vi_wgrad16, dy16.data_ptr(), dy16.stride(0), x16.data_ptr(), x16.stride(0),
           _DT[dy16.dtype], N, K, G, _lib.int_array(bounds), dW.data_ptr(), _ptr(db), ws.data_ptr(), ws.numel(), 0, int(accumulate),
           _stream())
    return dW, db


def dropout(x: torch.Tensor, p: float, seed: torch.Tensor, site: int) -> torch.Tensor:
    """y = x * keep / (1 - p) with the counter-based mask of (seed, site); the same call on a gradient is the backward pass"""
    x = x.contiguous()
    y = torch.empty_like(x)
    lib.vi_dropout(x.data_ptr(), y.data_ptr(), x.numel(), float(p), seed.data_ptr(), site, _DT[x.dtype], _stream())
    return y


def act_fwd(x: torch.Tensor, act: int) -> torch.Tensor:
    """GELU (EPI_GELU) or ReLU (EPI_RELU) of a contiguous tensor"""
    y = torch.empty_like(x)
    lib.vi_act_fwd(x.data_ptr(), y.data_ptr(), x.numel(), act, _DT[x.dtype], _stream())
    return y


def act_bwd(x: torch.Tensor, dy: torch.Tensor, act: int) -> torch.Tensor:
    dx = torch.empty_like(x)
    lib.vi_act_bwd(x.data_ptr(), dy.data_ptr(), dx.data_ptr(), x.numel(), act, _DT[x.dtype], _stream())
    return dx


def attention_bwd(q, k, v, do, dq, dk, dv, B: int, Lq: int, Lk: int, mask_mode: int, key_mask=None, pair_dist=None,
                  bias_affine=None, d_affine=None, drop=None):
    """adjoint of one attention problem into the row views dq / dk / dv; d_affine (fp32 [2]) accumulates the gradient of the GASA
    affine when pair_dist is given; drop = (p, site, seed tensor) of the forward dropout.  The long-sequence kernels keep their
    softmax statistics (or, in the fp32 check mode, the P / dS rows) in the shared workspace."""
    ws = workspace(q.device, lib.vi_attn_bwd_workspace(B, HEADS, Lq, Lk, _DT[q.dtype]))
    lib.vi_attn_bwd(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), do.data_ptr(), do.stride(0),
                    dq.data_ptr(), dq.stride(0), dk.data_ptr(), dk.stride(0), dv.data_ptr(), dv.stride(0), _DT[q.dtype], _ptr(key_mask),
                    _ptr(pair_dist), _ptr(bias_affine), _ptr(d_affine) if pair_dist is not None else None, B, HEADS, Lq, Lk, mask_mode,
                    float(drop[0]) if drop else 0.0, (int(drop[1]) & 0xFFFFFFFF) if drop else 0, drop[2].data_ptr() if drop else None,
                    ws.data_ptr(), ws.numel(), _stream())


def feat_wgrad(dt: torch.Tensor, feat: torch.Tensor, w_shape, want_db: bool):
    """(dW [768, feat_dim], db [768] or None) of the small-feature linear of embed_compose"""
    dW = torch.empty(w_shape, dtype=F32, device=dt.device)
    db = torch.empty((HIDDEN,), dtype=F32, device=dt.device) if want_db else None
    ws = workspace(dt.device, _red_floats(dt.shape[0], HIDDEN, 17))
    lib.vi_feat_wgrad(dt.data_ptr(), feat.data_ptr(), feat.shape[1], dW.data_ptr(), _ptr(db), dt.shape[0], ws.data_ptr(), ws.numel(),
                      _stream())
    return dW, db


def scatter_add_rows(src: torch.Tensor, idx: Optional[torch.Tensor], dst: torch.Tensor, period: int = 1) -> torch.Tensor:
    """dst[idx[r]] += src[r] (int64 idx), or dst[r % period] += src[r] when idx is None"""
    lib.vi_scatter_add_rows(src.data_ptr(), _ptr(idx), period, dst.data_ptr(), src.shape[0], _stream())
    return dst


def rowdot_bwd(dout: torch.Tensor, x: torch.Tensor, w: torch.Tensor, group_row_end: Optional[Sequence[int]] = None):
    """adjoint of ln_dot without its LayerNorm: (dx, dw [n_groups, 768], db [n_groups, 768] - the bias gradient replicated over
    the columns)"""
    rows = x.shape[0]
    n_groups, ends = _groups(group_row_end)
    dx = torch.empty_like(x)
    dw = torch.empty((n_groups, HIDDEN), dtype=F32, device=x.device)
    db = torch.empty((n_groups, HIDDEN), dtype=F32, device=x.device)
    ws = workspace(x.device, _red_floats(rows, HIDDEN, 2))
    lib.vi_rowdot_bwd(dout.data_ptr(), x.data_ptr(), w.data_ptr(), dx.data_ptr(), dw.data_ptr(), db.data_ptr(), rows, n_groups, ends,
                      ws.data_ptr(), ws.numel(), _stream())
    return dx, dw, db


def duet_fuse_logits_bwd(g_raw, l_raw, fuse_raw, gmap_masks_u8, gmap_visited_u8, vp_nav_u8, gmap_ids, cand_ids, dgl, dll, dfl,
                         B: int, G: int, P: int):
    """adjoint of duet_fuse_logits: (d g_raw, d l_raw, d fuse_raw or None)"""
    dg = torch.empty_like(g_raw)
    dl = torch.empty_like(l_raw)
    df = torch.empty((B,), dtype=F32, device=g_raw.device) if fuse_raw is not None else None
    lib.vi_duet_fuse_logits_bwd(g_raw.data_ptr(), l_raw.data_ptr(), _ptr(fuse_raw), gmap_masks_u8.data_ptr(), gmap_visited_u8.data_ptr(),
                                vp_nav_u8.data_ptr(), gmap_ids.data_ptr(), cand_ids.data_ptr(), _ptr(dgl), _ptr(dll), _ptr(dfl),
                                dg.data_ptr(), dl.data_ptr(), _ptr(df), B, G, P, _stream())
    return dg, dl, df


def cosine_loss_bwd(proj, tgt, dloss, R: int, want_proj: bool, want_tgt: bool):
    """adjoint of cosine_loss: (dproj or None, dtgt or None)"""
    dp = torch.empty_like(proj) if want_proj else None
    dt = torch.empty_like(tgt) if want_tgt else None
    lib.vi_cosine_loss_bwd(proj.data_ptr(), tgt.data_ptr(), dloss.data_ptr(), _ptr(dp), _ptr(dt), R, _stream())
    return dp, dt


def contrastive_loss_bwd(form: str, proj, tgt, negs, row_episode, neg_episode, param: float, scratch, dloss, R: int, n_negs: int,
                         want_tgt: bool, want_negs: bool):
    """adjoint of infonce_loss (form 'infonce', param = temperature) or margin_loss ('margin', param = margin) from its forward
    scratch: (dproj, dtgt or None, dnegs or None).  Without dtgt / dnegs the call is the one-launch proj-only adjoint."""
    dp = torch.empty_like(proj)
    dt = torch.empty_like(tgt) if want_tgt else None
    dn = torch.empty_like(negs) if want_negs else None
    work = torch.empty(R * (n_negs + 1), dtype=F32, device=proj.device) if want_negs and n_negs else None
    fn = lib.vi_infonce_loss_bwd if form == 'infonce' else lib.vi_margin_loss_bwd
    fn(proj.data_ptr(), tgt.data_ptr(), _ptr(negs), row_episode.data_ptr(), _ptr(neg_episode), param, scratch.data_ptr(),
       dloss.data_ptr(), dp.data_ptr(), _ptr(dt), _ptr(dn), _ptr(work), R, n_negs, _stream())
    return dp, dt, dn


def mul_bcast_bwd_s(dy: torch.Tensor, x: torch.Tensor, B: int, R: int) -> torch.Tensor:
    """ds[b] = sum_r dy[b, r] * x[b, r] (the scale gradient of mul_bcast, fp32 [B, R, 768] operands)"""
    ds = torch.empty((B, HIDDEN), dtype=F32, device=x.device)
    lib.vi_mul_bcast_bwd_s(dy.data_ptr(), x.data_ptr(), ds.data_ptr(), B, R, _stream())
    return ds


# ----------------------------------------------------------------------------------------------
# imitation + A2C fine-tuning of HAMT (vi_rl.cu)
def policy_sample(logits: torch.Tensor, stop_idx: torch.Tensor, seed: torch.Tensor, site: int, ended: torch.Tensor):
    """one sampling step of the agent over fp32 logits [B, O] (-inf = not admissible): (actions int64 [B], log p[a] [B], entropy [B],
    step mask [B] = not ended before this step); ``ended`` (uint8 [B]) is updated in place with actions == stop_idx"""
    B, O, ld = _rows2d(logits, 'logits')
    if ended.dtype != torch.uint8 or not ended.is_contiguous() or stop_idx.dtype != torch.int64:
        raise _lib.VlnImagineError('policy_sample: ended must be contiguous uint8 and stop_idx int64')
    dev = logits.device
    actions = torch.empty((B,), dtype=torch.int64, device=dev)
    logp, ent, mask = (torch.empty((B,), dtype=F32, device=dev) for _ in range(3))
    lib.vi_policy_sample(logits.data_ptr(), ld, O, B, stop_idx.contiguous().data_ptr(), seed.data_ptr(), int(site) & 0xFFFFFFFF,
                         actions.data_ptr(), logp.data_ptr(), ent.data_ptr(), ended.data_ptr(), mask.data_ptr(), _stream())
    return actions, logp, ent, mask


def policy_bwd(logits: torch.Tensor, actions: torch.Tensor, g_logp: Optional[torch.Tensor], g_ent: Optional[torch.Tensor]):
    """d logits [B, O] of g_logp . log p[a] + g_ent . entropy (policy_sample's outputs for the given actions)"""
    B, O, ld = _rows2d(logits, 'logits')
    d = torch.empty((B, O), dtype=F32, device=logits.device)
    c = lambda t: t.float().contiguous() if t is not None else None      # noqa: E731
    g_logp, g_ent = c(g_logp), c(g_ent)
    lib.vi_policy_bwd(logits.data_ptr(), ld, O, B, actions.data_ptr(), _ptr(g_logp), _ptr(g_ent), d.data_ptr(), O, _stream())
    return d


def _a2c_operands(values, logp, ent, masks, rewards):
    ts = [t.float().contiguous() for t in (values, logp, ent, masks, rewards)]
    if any(t.shape != ts[0].shape or t.dim() != 2 for t in ts):
        raise _lib.VlnImagineError('a2c_loss: values, logp, entropy, masks and rewards must all be [T, B]')
    return ts


def a2c_loss(values, logp, ent, masks, rewards, boot: Optional[torch.Tensor], ended: Optional[torch.Tensor], gamma: float,
             entropy_weight: float, normalize: str) -> torch.Tensor:
    """fp32 [4]: (total, policy, critic, entropy) A2C loss of [T, B] inputs (vi_a2c_loss); boot [B] is a constant (None = 0),
    ended (uint8 [B]) the flags after the last step"""
    v, lp, e, m, r = _a2c_operands(values, logp, ent, masks, rewards)
    T, B = v.shape
    out = torch.empty((4,), dtype=F32, device=v.device)
    boot = boot.float().contiguous() if boot is not None else None
    lib.vi_a2c_loss(v.data_ptr(), lp.data_ptr(), e.data_ptr(), m.data_ptr(), r.data_ptr(), _ptr(boot), _ptr(ended), T, B, float(gamma),
                    float(entropy_weight), _lib.A2C_NORM[normalize], out.data_ptr(), _stream())
    return out


def a2c_loss_bwd(values, logp, ent, masks, rewards, boot, ended, gamma: float, entropy_weight: float, normalize: str,
                 gout: torch.Tensor):
    """(dvalues, dlogp, dentropy) [T, B] of a2c_loss from gout = d(total, policy, critic, entropy)"""
    v, lp, e, m, r = _a2c_operands(values, logp, ent, masks, rewards)
    T, B = v.shape
    dv, dlp, de = (torch.empty((T, B), dtype=F32, device=v.device) for _ in range(3))
    boot = boot.float().contiguous() if boot is not None else None
    gout = gout.float().contiguous()
    lib.vi_a2c_loss_bwd(v.data_ptr(), lp.data_ptr(), e.data_ptr(), m.data_ptr(), r.data_ptr(), _ptr(boot), _ptr(ended), T, B,
                        float(gamma), float(entropy_weight), _lib.A2C_NORM[normalize], gout.data_ptr(), dv.data_ptr(), dlp.data_ptr(),
                        de.data_ptr(), _stream())
    return dv, dlp, de


def value_head(h: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, drop=None) -> torch.Tensor:
    """v [rows] = dropout(h) . w2 + b2 over contiguous fp32 [rows, 512] (vi_value_head); drop = (p, seed tensor, site)"""
    rows = h.shape[0]
    if h.dtype != F32 or not h.is_contiguous() or h.shape[1] != 512:
        raise _lib.VlnImagineError('value_head: h must be contiguous fp32 [rows, 512]')
    p, seed, site = drop if drop is not None else (0.0, None, 0)
    v = torch.empty((rows,), dtype=F32, device=h.device)
    lib.vi_value_head(h.data_ptr(), rows, w2.data_ptr(), b2.data_ptr(), float(p), _ptr(seed), int(site) & 0xFFFFFFFF, v.data_ptr(),
                      _stream())
    return v


def value_head_bwd(dv: torch.Tensor, h: torch.Tensor, w2: torch.Tensor, dtype, drop=None):
    """(dh [rows, 512] of ``dtype`` - fp32, or the 16-bit operand of the first layer's gradient GEMMs -, dw2 [512], db2 [1])"""
    rows = h.shape[0]
    p, seed, site = drop if drop is not None else (0.0, None, 0)
    dh = torch.empty((rows, 512), dtype=dtype, device=h.device)
    d32, d16 = (dh, None) if dtype == F32 else (None, dh)
    dw2 = torch.empty((512,), dtype=F32, device=h.device)
    db2 = torch.empty((1,), dtype=F32, device=h.device)
    dv = dv.float().contiguous()
    lib.vi_value_head_bwd(dv.data_ptr(), h.data_ptr(), rows, w2.data_ptr(), float(p), _ptr(seed), int(site) & 0xFFFFFFFF, _ptr(d32),
                          _ptr(d16), _dt16(d16), dw2.data_ptr(), db2.data_ptr(), _stream())
    return dh, dw2, db2
