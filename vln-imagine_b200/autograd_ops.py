"""torch.autograd.Function wrappers: forward AND backward of every differentiable step are libvlnimagine kernels.

Used when a mode is called with autograd recording (fine-tuning, BASELINE.json cfg-4).  The autograd engine only
chains the nodes and accumulates gradients at fan-out points (residual branches) and into ``.grad``; it performs
no model arithmetic itself.  Conventions:

* dense layers: ``dX = dY W`` runs the tcgen05 GEMM on the transposed bf16 weight shadow; ``dW = dY^T X`` and ``db`` come
  from vi_wgrad16 on dY and X as they lie in memory (all groups of a row-stacked layer in one launch).  The fp32 check mode
  runs the GEMM on kernel-transposed copies of dY and X and takes ``db`` as a fixed-order column sum, group by group;
* the training forward keeps pre-activations: GELU / ReLU are their own kernels instead of GEMM epilogues;
* LayerNorm returns the fp32 residual-stream tensor and its bf16 operand copy; its backward takes both gradients;
* the embedding composer is decomposed into primitives (small-feature linear, LayerNorm, row gather, sum);
* dropout is not applied (probabilities must be 0 for gradient parity; see DESIGN.md).
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch
from torch.autograd import Function

from . import _lib, ops
from .ops import BF16, F32, HIDDEN, EPI_GELU, EPI_NONE, EPI_RELU, MASK_ADD_NEG10000, _ptr, _stream, check, lib, _launched


def needs_grad(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and torch.is_tensor(t) and t.requires_grad for t in tensors)


def pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def _dt(t: torch.Tensor) -> int:
    return _lib.DT_BF16 if t.dtype == BF16 else _lib.DT_F32


def transpose(src: torch.Tensor, pad_rows: Optional[int] = None) -> torch.Tensor:
    """[rows, cols] view -> [cols, pad_rows] (zero padded columns)"""
    rows, cols = src.shape
    pr = pad_rows or rows
    dst = torch.empty((cols, pr), dtype=src.dtype, device=src.device)
    check(lib.vi_transpose(src.data_ptr(), src.stride(0), dst.data_ptr(), dst.stride(0), rows, cols, pr, _dt(src), _stream()),
          'vi_transpose')
    _launched(1)
    return dst


_SCRATCH = {}
RED_CHUNK = 128


def reduce_scratch(device, rows: int, cols: int, n_out: int) -> torch.Tensor:
    """fp32 workspace of the two-stage column reductions (caller-owned, one per device, grown on demand; launches
    that share it are ordered by the stream they run on)"""
    need = n_out * ((rows + RED_CHUNK - 1) // RED_CHUNK) * cols
    t = _SCRATCH.get(device)
    if t is None or t.numel() < need:
        t = torch.empty((max(need, 1 << 22),), dtype=F32, device=device)
        _SCRATCH[device] = t
    return t


def colsum(x: torch.Tensor) -> torch.Tensor:
    rows, cols = x.shape
    out = torch.empty((cols,), dtype=F32, device=x.device)
    sc = reduce_scratch(x.device, rows, cols, 1)
    check(lib.vi_colsum(x.data_ptr(), x.stride(0), _dt(x), out.data_ptr(), rows, cols, sc.data_ptr(), sc.numel(), _stream()),
          'vi_colsum')
    _launched(2)
    return out


_WGRAD_WS = {}


class _GradAcc:
    """Gradient accumulation fused into the kernels (opt-in, ``fused_grad_accumulation``).  A parameter of this path is used once
    per navigation step, so autograd ends an iteration with one small ``add`` kernel per parameter per step (~1500 launches at 6
    steps).  With the switch on, the dense-layer and LayerNorm backward nodes add their parameter gradients straight into one fp32
    accumulator per weight pack (vi_wgrad16 / vi_add_ln_drop_bwd with accumulate = 1: TMA reduce-add or a read-modify-write with one
    writer per element, in backward order - deterministic) and hand autograd ``None``; when the backward pass ends, ONE multi-tensor
    add moves the accumulators into ``.grad`` (created if missing), which is what the optimiser / the flat all-reduce buffer see.
    Not for modules whose parameters carry autograd hooks (DistributedDataParallel): those keep the plain path."""
    enabled = False
    buffers = {}            # key (ids of the pack's parameters) -> dict(tensors..., live=bool, params=[...])
    live = []               # entries holding gradients of the backward pass in flight
    queued = False


class fused_grad_accumulation:
    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        self.prev = _GradAcc.enabled
        _GradAcc.enabled = self.on
        if self.on:                                   # a backward pass that died half-way must not leak into this one
            for e in _GradAcc.live:
                e['live'] = False
            _GradAcc.live, _GradAcc.queued = [], False
        return self

    def __exit__(self, *exc):
        _GradAcc.enabled = self.prev
        return False


def _acc_entry(params, shapes, device):
    """the accumulators of one pack: tensors of ``shapes`` + the parameter slices they feed"""
    key = tuple(id(p) for p in params) + tuple(tuple(s) for s in shapes)
    e = _GradAcc.buffers.get(key)
    # ids are only unique among LIVE objects: an entry of a model that is gone must not be handed to a new one whose parameters
    # happen to reuse the ids (its slices would feed the dead parameters)
    if e is None or e['t'][0].device != device or len(e['params']) != len(params) or any(a is not b for a, b in zip(e['params'], params)):
        e = {'t': [torch.empty(tuple(sh), dtype=F32, device=device) for sh in shapes], 'live': False, 'params': list(params)}
        _GradAcc.buffers[key] = e
    return e


def release_accumulators():
    """drop every accumulator (and the references to the parameters they feed): call when a model is retired"""
    _GradAcc.buffers.clear()
    _GradAcc.live, _GradAcc.queued = [], False


def _acc_begin(e) -> int:
    """1 when the entry already holds gradients of this backward pass (the kernel must add), else 0 (overwrite)"""
    beta = 1 if e['live'] else 0
    if not e['live']:
        e['live'] = True
        _GradAcc.live.append(e)
    if not _GradAcc.queued:
        _GradAcc.queued = True
        torch.autograd.Variable._execution_engine.queue_callback(_acc_flush)
    return beta


def _acc_flush():
    """end of the backward pass: accumulators -> .grad (one multi-tensor add)"""
    dsts, srcs = [], []
    for e in _GradAcc.live:
        for p, src in e['slices']:
            if not p.requires_grad:
                continue
            if p.grad is None:
                p.grad = src.reshape(p.shape).clone()
            else:
                dsts.append(p.grad)
                srcs.append(src.reshape(p.shape))
        e['live'] = False
    _GradAcc.live = []
    _GradAcc.queued = False
    if dsts:
        torch._foreach_add_(dsts, srcs)
        _launched(1)


def wgrad16(dy16: torch.Tensor, x16: torch.Tensor, ends, want_db: bool, out=None, accumulate: int = 0):
    """(dW [n_groups * N, K] fp32, db [n_groups * N] fp32 or None) of a (grouped) dense layer from the 16-bit row-major dY [M, N]
    and X [M, K] as they are (vi_wgrad16: MN-major tcgen05 operands, no transposed copies, bias gradient on the tensor cores).
    out = (dW, db) preallocated; accumulate = 1 adds to them."""
    M, N = dy16.shape
    K = x16.shape[1]
    bounds = [min(int(e), M) for e in ends] if ends is not None else [M]
    G = len(bounds)
    rows = _lib.int_array([b - (bounds[i - 1] if i else 0) for i, b in enumerate(bounds)])
    S = int(_lib.lib.vi_wgrad16_splits(N, K, G, rows))               # host-side queries: not launches
    need = int(_lib.lib.vi_wgrad16_workspace(N, K, G, rows, S))
    ws = None
    if need > 0:
        ws = _WGRAD_WS.get(dy16.device)
        if ws is None or ws.numel() < need:
            ws = torch.empty((max(need, 1 << 23),), dtype=F32, device=dy16.device)
            _WGRAD_WS[dy16.device] = ws
    if out is not None:
        dW, db = out
    else:
        dW = torch.empty((G * N, K), dtype=F32, device=dy16.device)
        db = torch.empty((G * N,), dtype=F32, device=dy16.device) if want_db else None
    tr = ops._Counters.gemm_trace                                    # bench.py: tensor-core launches with their FLOPs
    if tr is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    check(lib.vi_wgrad16(dy16.data_ptr(), dy16.stride(0), x16.data_ptr(), x16.stride(0), ops._DT[dy16.dtype], N, K, G,
                         _lib.int_array(bounds), dW.data_ptr(), _ptr(db), _ptr(ws), ws.numel() if ws is not None else 0, S,
                         int(accumulate), _stream()), 'vi_wgrad16')
    if tr is not None:
        e1.record()
        tr.append((bounds[-1], N, K, e0, e1))
    _launched(2 if S > 1 else 1)
    return dW, db


def wgrad16_ok(dy16: torch.Tensor, x16: torch.Tensor) -> bool:
    return (ops.is16(dy16.dtype) and x16.dtype == dy16.dtype and dy16.shape[1] % 128 == 0 and x16.shape[1] % 64 == 0
            and dy16.stride(1) == 1 and x16.stride(1) == 1 and dy16.stride(0) % 8 == 0 and x16.stride(0) % 8 == 0
            and dy16.data_ptr() % 16 == 0 and x16.data_ptr() % 16 == 0)


def to_operand(t: torch.Tensor, lowp: bool) -> torch.Tensor:
    """gradient tensor -> GEMM operand dtype of the current precision mode (contiguous)"""
    t = t.contiguous()
    if lowp and t.dtype != BF16:
        return ops.cast_h16(t, dtype=BF16)
    if not lowp and t.dtype != F32:
        return t.float()
    return t


# ----------------------------------------------------------------------------------------------
# dropout: counter-based masks keyed by (device seed, site id, element index); nothing is stored for the backward pass
class _DropState:
    seeds = {}              # device -> int32 [1] tensor (read by the kernels as uint32)
    site = 0                # python-side site counter: every dropout layer call of the process gets its own id


def dropout_seed(device) -> torch.Tensor:
    t = _DropState.seeds.get(device)
    if t is None:
        base = int(torch.randint(0, 2 ** 31 - 1, (1,)).item())          # CPU generator: follows torch.manual_seed
        t = torch.full((1,), base, dtype=torch.int32, device=device)
        _DropState.seeds[device] = t
    return t


def advance_dropout_seeds():
    """called from the optimizer-step hook (blocks._WeightsEpoch): eager or captured into the update graph"""
    for t in _DropState.seeds.values():
        t.add_(1)


def next_site() -> int:
    _DropState.site = (_DropState.site + 1) & 0x7FFFFFFF
    return _DropState.site


def dropout_raw(x: torch.Tensor, p: float, site: int) -> torch.Tensor:
    """y = x * keep / (1 - p) (no autograd); the same call on a gradient is the backward pass"""
    x = x.contiguous()
    y = torch.empty_like(x)
    check(lib.vi_dropout(x.data_ptr(), y.data_ptr(), x.numel(), float(p), dropout_seed(x.device).data_ptr(), site, _dt(x), _stream()),
          'vi_dropout')
    _launched(1)
    return y


class DropoutFn(Function):
    @staticmethod
    def forward(ctx, x, p, site):
        ctx.p, ctx.site = p, site
        return dropout_raw(x, p, site)

    @staticmethod
    def backward(ctx, dy):
        return dropout_raw(dy, ctx.p, ctx.site), None, None


def dropout(x: torch.Tensor, p: float) -> torch.Tensor:
    if p <= 0:
        return x
    if x.dtype not in (BF16, F32):
        raise _lib.VlnImagineError('dropout: bf16 / fp32 tensors only')
    return DropoutFn.apply(x, p, next_site())


class CastBf16Fn(Function):
    """fp32 -> bf16 operand copy; the gradient passes back in fp32."""

    @staticmethod
    def forward(ctx, x):
        return ops.cast_h16(x, dtype=BF16)

    @staticmethod
    def backward(ctx, dy):
        return dy.float()


class LinearFn(Function):
    """y = x W^T + b [+ residual] for a (grouped) LinearPack; parameters are passed for gradient routing."""

    @staticmethod
    def forward(ctx, x, residual, pack, lowp, out_dtype, ends, *params):
        w, b = pack.get(lowp)
        y = ops.gemm(x, w, b, residual=residual, epilogue=EPI_NONE, out_dtype=out_dtype, group_row_end=ends)
        ctx.save_for_backward(x)
        ctx.pack, ctx.lowp, ctx.ends, ctx.has_res = pack, lowp, ends, residual is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dx, grads = _linear_bwd(ctx.pack, x, to_operand(dy, ctx.lowp), ctx.lowp, ctx.ends, ctx.needs_input_grad[0])
        return (dx, dy if ctx.has_res else None, None, None, None, None, *grads)


def _linear_bwd(pack, x, dyo, lowp, ends, need_dx):
    """(dX, parameter gradients in grad_sources() order) of y = x W^T + b from dY in the operand format of the precision mode.
    ``pack`` provides get_t / weights / biases; its stacked weight may be padded with zero rows past the parameters (the
    gradients handed back are the parameters' rows)."""
    M, K = x.shape
    n_groups = 1 if ends is None else len(ends)
    N = dyo.shape[1]
    dx = None
    if need_dx:
        wt = pack.get_t(lowp, n_groups)                             # [n_groups*K, N]
        dx = ops.gemm(dyo, wt, None, out_dtype=x.dtype, group_row_end=ends)
    if lowp and wgrad16_ok(dyo, x):
        return dx, _lin_param_grads(pack, dyo, x, ends)
    dW = torch.empty((n_groups * N, K), dtype=F32, device=x.device)   # fp32 check mode / odd shapes: transposed copies
    db = torch.empty((n_groups * N,), dtype=F32, device=x.device) if pack.biases is not None else None
    bounds = [0] + (list(ends) if ends is not None else [M])
    for g in range(n_groups):
        r0, r1 = bounds[g], min(bounds[g + 1], M)
        rp = pad64(r1 - r0) if lowp else r1 - r0
        dyT = transpose(dyo[r0:r1], rp)                             # [N, rp]
        xT = transpose(x[r0:r1], rp)                                # [K, rp]
        ops.gemm(dyT, xT, None, out_dtype=F32, out=dW[g * N:(g + 1) * N])
        if db is not None:
            db[g * N:(g + 1) * N] = colsum(dyo[r0:r1])
    return dx, _lin_grads(pack, dW, db)


def linear(x, pack, lowp, residual=None, out_dtype=None, ends=None):
    """differentiable dense layer (no fused activation); pack = blocks.LinearPack"""
    out_dtype = out_dtype or (BF16 if lowp else F32)
    return LinearFn.apply(x, residual, pack, lowp, out_dtype, ends, *pack.grad_sources())


class PaddedLinearFn(Function):
    """scores = x W^T + b of a dense layer whose output width is padded with zero weight rows (pretrain._PaddedLinear: the tied
    MLM decoder 30522 -> 30592, the MRC classifier 1000 -> 1024; multiples of 128, the column granule of vi_wgrad16).
    Returns (scores fp32 [M, n_pad], handle).  ``handle`` (an [M, n_pad] view of one element, in the operand format of the
    precision mode) is where the loss node (CERowsFn / KLRowsFn) sends d scores, so the gradient reaches this node as the
    16-bit GEMM operand its loss kernel wrote, with no cast pass.  A gradient of the fp32 scores themselves (another loss)
    is cast to the operand format and added.  Backward: dX through the transposed shadow
    of the padded weight, dW (first n rows: for the tied decoder autograd adds them to the embedding lookup's scatter-add)
    and db through vi_wgrad16 (the fp32 check mode: transposed copies)."""

    @staticmethod
    def forward(ctx, x, pack, lowp, *params):
        w, b = pack.get_train(lowp)
        y = ops.gemm(x, w, b, out_dtype=F32)
        ctx.save_for_backward(x)
        ctx.pack, ctx.lowp = pack, lowp
        ctx.set_materialize_grads(False)
        handle = torch.zeros((), dtype=BF16 if lowp else F32, device=x.device).expand(y.shape)
        return y, handle

    @staticmethod
    def backward(ctx, dy, dh):
        (x,) = ctx.saved_tensors
        g = dh.contiguous() if dh is not None else None
        if dy is not None:
            g = to_operand(dy, ctx.lowp) if g is None else g + to_operand(dy, ctx.lowp)
        dx, grads = _linear_bwd(ctx.pack, x, g, ctx.lowp, None, ctx.needs_input_grad[0])
        return (dx, None, None, *grads)


def padded_linear(x, pack, lowp):
    """differentiable padded dense layer -> (scores, gradient handle); see PaddedLinearFn"""
    return PaddedLinearFn.apply(x, pack, lowp, *pack.grad_sources())


class CERowsFn(Function):
    """per-row cross-entropy (ops.ce_rows) over the first n_cols columns of fp32 ``logits``; the gradient w.r.t. the logits is
    written by vi_ce_rows_bwd in the dtype of ``handle`` (bf16: the operand of the gradient GEMMs; fp32 in the check mode) and
    returned for ``handle``, which is the logits tensor itself or PaddedLinearFn's handle."""

    @staticmethod
    def forward(ctx, logits, handle, labels, n_cols):
        ctx.save_for_backward(logits, labels)
        ctx.n_cols, ctx.dtype, ctx.ld_out = n_cols, handle.dtype, handle.shape[1]
        return ops.ce_rows(logits, labels, n_cols)

    @staticmethod
    def backward(ctx, dloss):
        logits, labels = ctx.saved_tensors
        return None, ops.ce_rows_bwd(logits, labels, ctx.n_cols, dloss, ctx.dtype, ctx.ld_out), None, None


class KLRowsFn(Function):
    """per-row KL(targets || softmax(logits)) (ops.kl_rows); gradient as in CERowsFn (vi_kl_rows_bwd), none for the targets"""

    @staticmethod
    def forward(ctx, logits, handle, targets, n_cols):
        targets = targets.contiguous()
        ctx.save_for_backward(logits, targets)
        ctx.n_cols, ctx.dtype, ctx.ld_out = n_cols, handle.dtype, handle.shape[1]
        return ops.kl_rows(logits, targets, n_cols)

    @staticmethod
    def backward(ctx, dloss):
        logits, targets = ctx.saved_tensors
        return None, ops.kl_rows_bwd(logits, targets, ctx.n_cols, dloss, ctx.dtype, ctx.ld_out), None, None


class ActFn(Function):
    @staticmethod
    def forward(ctx, x, act):
        x = x.contiguous()
        y = torch.empty_like(x)
        check(lib.vi_act_fwd(x.data_ptr(), y.data_ptr(), x.numel(), act, _dt(x), _stream()), 'vi_act_fwd')
        _launched(1)
        ctx.save_for_backward(x)
        ctx.act = act
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dy = dy.contiguous()
        if dy.dtype != x.dtype:
            dy = dy.to(x.dtype)
        dx = torch.empty_like(x)
        check(lib.vi_act_bwd(x.data_ptr(), dy.data_ptr(), dx.data_ptr(), x.numel(), ctx.act, _dt(x), _stream()), 'vi_act_bwd')
        _launched(1)
        return dx, None


class LayerNormFn(Function):
    """(y32, y16) = LN(a [+ b]); y16 is None-like (empty) in fp32 mode.  Backward sums the two incoming gradients."""

    @staticmethod
    def forward(ctx, a, b, gamma, beta, eps, lowp, ends, n_params, *params):
        a = a.contiguous()
        y32, y16 = ops.add_ln(a, b, gamma, beta, eps, want16=lowp, group_row_end=ends)
        ctx.save_for_backward(a, b if b is not None else a.new_empty(0), gamma)
        ctx.eps, ctx.ends, ctx.has_b, ctx.n_params = eps, ends, b is not None, n_params
        ctx.b_needs = b is not None and b.requires_grad
        ctx.a_needs = a.requires_grad
        ctx.param_srcs = list(params)
        if y16 is None:
            y16 = a.new_empty(0)
            ctx.mark_non_differentiable(y16)
        return y32, y16

    @staticmethod
    def backward(ctx, dy32, dy16):
        a, b, gamma = ctx.saved_tensors
        b = b if ctx.has_b else None
        rows = a.shape[0]
        ends = ctx.ends
        n_groups = 1 if ends is None else len(ends)
        if dy16 is not None and dy16.numel() == 0:
            dy16 = None
        if dy32 is None and dy16 is None:
            return (None,) * (8 + ctx.n_params)
        if dy32 is not None:
            dy32 = dy32.contiguous()
        if dy16 is not None:
            dy16 = dy16.contiguous()
        dx = torch.empty_like(a)
        dg, dbt, acc, pg = _ln_param_grads(ctx.param_srcs, n_groups, a.device)
        stats = torch.empty((rows, 2), dtype=F32, device=a.device)
        sc = reduce_scratch(a.device, 16 * rows, HIDDEN, 2)           # the fused pass reduces chunks of 8 - 32 rows (>= RED_CHUNK / 16)
        check(lib.vi_add_ln_drop_bwd(a.data_ptr(), _ptr(b), gamma.data_ptr(), ctx.eps, _ptr(dy32), _ptr(dy16), dx.data_ptr(), None,
                                     None, dg.data_ptr(), dbt.data_ptr(), stats.data_ptr(), rows, n_groups,
                                     _lib.int_array(list(ends)) if ends is not None else None, sc.data_ptr(), sc.numel(), acc,
                                     0.0, None, 0, _stream()), 'vi_add_ln_drop_bwd')
        _launched(2)
        return (dx if ctx.a_needs else None, dx if ctx.b_needs else None, None, None, None, None, None, None, *pg)


class DenseResLNFn(Function):
    """(y32, y16) = LN(dropout(x W^T + bias) + res) as ONE autograd node (BertSelfOutput / BertOutput, D/models/vilmodel.py:151-155,
    190-194; 16-bit mode).  Chaining LinearFn -> DropoutFn -> LayerNormFn costs, per layer and direction, a dropout pass over the
    fp32 rows and an fp32 -> bf16 cast of the gradient; here the mask is applied inside the LayerNorm kernels (vi_add_ln_drop,
    vi_add_ln_drop_bwd) and the backward kernel emits dropout(dx) directly as the 16-bit operand of the weight / input gradient
    GEMMs.  p == 0: the residual rides in the GEMM epilogue as before.  Parameter gradients: accumulated in the kernels when
    fused_grad_accumulation is on, returned to autograd otherwise."""

    @staticmethod
    def forward(ctx, x, res32, pack, lnpack, eps, ends, p, site, n_lin, *params):
        w, b = pack.get(True)
        g, be = lnpack.get()
        rows = x.shape[0]
        n_groups = 1 if ends is None else len(ends)
        ln_ends = ends if len(lnpack.g.tensors) > 1 else None
        earr = _lib.int_array(list(ln_ends)) if ln_ends is not None else None
        if p > 0:
            y32 = torch.empty((rows, HIDDEN), dtype=F32, device=x.device)
            y16 = torch.empty((rows, HIDDEN), dtype=x.dtype, device=x.device)
            d = ops.gemm(x, w, b, out_dtype=F32, group_row_end=ends)
            check(lib.vi_add_ln_drop(d.data_ptr(), res32.data_ptr(), g.data_ptr(), be.data_ptr(), eps, y32.data_ptr(), y16.data_ptr(),
                                     ops._DT[y16.dtype], rows, 1 if ln_ends is None else len(ln_ends), earr, float(p),
                                     dropout_seed(x.device).data_ptr(), site, _stream()), 'vi_add_ln_drop')
            _launched(1)
            ctx.save_for_backward(x, d, res32, g)
        else:
            d = ops.gemm(x, w, b, residual=res32, out_dtype=F32, group_row_end=ends)
            y32, y16 = ops.add_ln(d, None, g, be, eps, want16=True, group_row_end=ln_ends)
            ctx.save_for_backward(x, d, d.new_empty(0), g)
        ctx.pack, ctx.lnpack, ctx.eps, ctx.ends, ctx.ln_ends, ctx.p, ctx.site, ctx.n_lin = pack, lnpack, eps, ends, ln_ends, p, site, n_lin
        ctx.n_params = len(params)
        ctx.res_needs = res32.requires_grad
        return y32, y16

    @staticmethod
    def backward(ctx, dy32, dy16):
        x, d, res32, g = ctx.saved_tensors
        pack, lnpack, ends, ln_ends, p = ctx.pack, ctx.lnpack, ctx.ends, ctx.ln_ends, ctx.p
        rows = d.shape[0]
        dev = d.device
        n_groups = 1 if ends is None else len(ends)
        n_ln = 1 if ln_ends is None else len(ln_ends)
        if dy16 is not None and dy16.numel() == 0:
            dy16 = None
        dy32 = dy32.contiguous() if dy32 is not None else None
        dy16 = dy16.contiguous() if dy16 is not None else None
        ln_srcs = lnpack.grad_sources()
        dg, dbt, acc, ln_grads = _ln_param_grads(ln_srcs, n_ln, dev)
        dres = torch.empty((rows, HIDDEN), dtype=F32, device=dev)
        da16 = torch.empty((rows, HIDDEN), dtype=x.dtype, device=dev)
        stats = torch.empty((rows, 2), dtype=F32, device=dev)
        sc = reduce_scratch(dev, 16 * rows, HIDDEN, 2)
        check(lib.vi_add_ln_drop_bwd(d.data_ptr(), res32.data_ptr() if p > 0 else None, g.data_ptr(), ctx.eps, _ptr(dy32), _ptr(dy16),
                                     dres.data_ptr(), None, da16.data_ptr(), dg.data_ptr(), dbt.data_ptr(), stats.data_ptr(), rows, n_ln,
                                     _lib.int_array(list(ln_ends)) if ln_ends is not None else None, sc.data_ptr(), sc.numel(), acc,
                                     float(p), dropout_seed(dev).data_ptr() if p > 0 else None, ctx.site, _stream()), 'vi_add_ln_drop_bwd')
        _launched(2)
        # dense layer: dX = dA W, dW = dA^T X, db = column sums of dA with dA = da16
        K = x.shape[1]
        N = da16.shape[1]
        dx = None
        if ctx.needs_input_grad[0]:
            dx = ops.gemm(da16, pack.get_t(True, n_groups), None, out_dtype=x.dtype, group_row_end=ends)
        if not (wgrad16_ok(da16, x) and N * n_groups == sum(w_.shape[0] for w_ in pack.weights)):
            raise _lib.VlnImagineError('DenseResLNFn: the dense layer must be a multiple of 128 x 64 (got N=%d, K=%d)' % (N, K))
        lin_grads = _lin_param_grads(pack, da16, x, ends)
        return (dx, dres if ctx.res_needs else None, None, None, None, None, None, None, None, *lin_grads, *ln_grads)


def _lin_slices(pack, tensors):
    """(parameter, accumulator slice) pairs of a LinearPack's stacked weight / bias accumulators"""
    sl, off = [], 0
    for wsrc in pack.weights:
        sl.append((wsrc, tensors[0][off:off + wsrc.shape[0]]))
        off += wsrc.shape[0]
    off = 0
    for bsrc, wsrc in zip(pack.biases or [], pack.weights):
        if bsrc is not None:
            sl.append((bsrc, tensors[1][off:off + wsrc.shape[0]]))
        off += wsrc.shape[0]
    return sl


def _lin_param_grads(pack, dy16, x16, ends):
    """weight and bias gradients of a LinearPack from the 16-bit dY and X (vi_wgrad16), in grad_sources() order.  With
    fused_grad_accumulation on (and one accumulator covering the whole pack) they are added into the pack's accumulators and
    autograd gets None for every parameter; otherwise they are returned per parameter."""
    n_groups = 1 if ends is None else len(ends)
    N, K = dy16.shape[1], x16.shape[1]
    has_b = pack.biases is not None
    if _GradAcc.enabled and N * n_groups == sum(w.shape[0] for w in pack.weights):
        bs = [b for b in pack.biases if b is not None] if has_b else []
        e = _acc_entry(pack.weights + bs, [(n_groups * N, K)] + ([(n_groups * N,)] if has_b else []), x16.device)
        if 'slices' not in e:
            e['slices'] = _lin_slices(pack, e['t'])
        acc = _acc_begin(e)
        wgrad16(dy16, x16, ends, has_b, out=(e['t'][0], e['t'][1] if has_b else None), accumulate=acc)
        return [None] * len(pack.grad_sources())
    dW, db = wgrad16(dy16, x16, ends, has_b)
    return _lin_grads(pack, dW, db)


def _ln_param_grads(srcs, n_groups: int, device):
    """(dgamma, dbeta, accumulate, grads) for the LayerNorm parameters srcs = gammas + betas of n_groups groups, the buffers
    and flag vi_add_ln_drop_bwd writes into.  With fused_grad_accumulation on they are the pack's accumulators and grads is all
    None; otherwise fresh [n_groups, 768] buffers whose rows are the gradients autograd gets (grads, in srcs order)."""
    half = len(srcs) // 2
    if _GradAcc.enabled and half == n_groups:
        e = _acc_entry(srcs, [(n_groups, HIDDEN), (n_groups, HIDDEN)], device)
        if 'slices' not in e:
            e['slices'] = [(srcs[i], e['t'][0][i]) for i in range(half)] + [(srcs[half + i], e['t'][1][i]) for i in range(half)]
        acc = _acc_begin(e)
        dg, dbt = e['t']
        return dg, dbt, acc, [None] * len(srcs)
    dg = torch.empty((n_groups, HIDDEN), dtype=F32, device=device)
    dbt = torch.empty((n_groups, HIDDEN), dtype=F32, device=device)
    grads = [dg[i] if srcs[i].requires_grad else None for i in range(half)] + \
            [dbt[i] if srcs[half + i].requires_grad else None for i in range(half)]
    return dg, dbt, 0, grads


def _lin_grads(pack, dW, db):
    """gradients of a LinearPack's parameters in grad_sources() order from the stacked dW / db"""
    grads, off = [], 0
    for wsrc in pack.weights:
        n = wsrc.shape[0]
        grads.append(dW[off:off + n] if wsrc.requires_grad else None)
        off += n
    if pack.biases is not None:
        off = 0
        for bsrc, wsrc in zip(pack.biases, pack.weights):
            n = wsrc.shape[0]
            if bsrc is not None:
                grads.append(db[off:off + n] if bsrc.requires_grad else None)
            off += n
    return grads


def dense_res_ln(x, res32, pack, lnpack, eps, ends, p):
    """differentiable LN(dropout(x W^T + b) + res) -> (y32, y16), 16-bit mode (see DenseResLNFn)"""
    lin_srcs, ln_srcs = pack.grad_sources(), lnpack.grad_sources()
    site = next_site() if p > 0 else 0
    return DenseResLNFn.apply(x, res32, pack, lnpack, eps, ends, float(p), site, len(lin_srcs), *lin_srcs, *ln_srcs)


def dense_res_ln_ok(x, pack, lnpack, ends) -> bool:
    n_groups = 1 if ends is None else len(ends)
    N = sum(w_.shape[0] for w_ in pack.weights)
    return (ops.is16(x.dtype) and x.shape[1] % 64 == 0 and N % n_groups == 0 and (N // n_groups) == HIDDEN and x.stride(1) == 1
            and x.stride(0) % 8 == 0 and len(lnpack.g.tensors) in (1, n_groups))


def layer_norm(a, b, lnpack, eps, lowp, ends=None):
    """differentiable LayerNorm(a [+ b]) -> (y32, y16 or None); lnpack = blocks.LNPack"""
    g, be = lnpack.get()
    srcs = lnpack.grad_sources()
    y32, y16 = LayerNormFn.apply(a, b, g, be, eps, lowp, ends, len(srcs), *srcs)
    return y32, (y16 if lowp else None)


class AttentionFn(Function):
    """Multi-stream attention.  ``spec`` = list of problems {q: (base index, row0, col0), k: ..., v: ..., B, Lq, Lk,
    key_mask, pair_dist, out_row0}; tensors = distinct base tensors (2-D) [+ the two GASA parameters last]."""

    @staticmethod
    def forward(ctx, spec, rows_out, mask_mode, n_bases, *tensors):
        bases = tensors[:n_bases]
        out = torch.empty((rows_out, HIDDEN), dtype=bases[0].dtype, device=bases[0].device)
        covered = 0
        probs = []
        for s in spec:
            def view(key, L):
                bi, r0, c0 = s[key]
                return bases[bi][r0:r0 + s['B'] * L, c0:c0 + HIDDEN]
            probs.append(dict(q=view('q', s['Lq']), k=view('k', s['Lk']), v=view('v', s['Lk']),
                              out=out[s['out_row0']:s['out_row0'] + s['B'] * s['Lq']], B=s['B'], Lq=s['Lq'], Lk=s['Lk'],
                              key_mask=s.get('key_mask'), pair_dist=s.get('pair_dist'), bias_affine=s.get('bias_affine'),
                              drop=s.get('drop')))
            covered += s['B'] * s['Lq']
        if covered < rows_out:
            out.zero_()
        ops.attention_multi(probs, mask_mode)
        ctx.save_for_backward(*bases)
        ctx.spec, ctx.mask_mode, ctx.n_bases, ctx.n_extra = spec, mask_mode, n_bases, len(tensors) - n_bases
        return out

    @staticmethod
    def backward(ctx, dout):
        bases = ctx.saved_tensors
        dout = dout.contiguous()
        grads = [torch.zeros_like(b) if ctx.needs_input_grad[4 + i] else None for i, b in enumerate(bases)]
        d_affine = None
        for s in ctx.spec:
            def view(t, key, L):
                bi, r0, c0 = s[key]
                return t[bi][r0:r0 + s['B'] * L, c0:c0 + HIDDEN]
            q, k, v = view(bases, 'q', s['Lq']), view(bases, 'k', s['Lk']), view(bases, 'v', s['Lk'])
            need = [grads[s[key][0]] is not None for key in ('q', 'k', 'v')]
            if not any(need):
                continue
            tmp = lambda n: torch.empty((n, HIDDEN), dtype=q.dtype, device=q.device)   # noqa: E731
            dq = view(grads, 'q', s['Lq']) if need[0] else tmp(s['B'] * s['Lq'])
            dk = view(grads, 'k', s['Lk']) if need[1] else tmp(s['B'] * s['Lk'])
            dv = view(grads, 'v', s['Lk']) if need[2] else tmp(s['B'] * s['Lk'])
            do = dout[s['out_row0']:s['out_row0'] + s['B'] * s['Lq']]
            if do.dtype != q.dtype:
                do = do.to(q.dtype)
            if s.get('pair_dist') is not None and d_affine is None:
                d_affine = torch.zeros((2,), dtype=F32, device=q.device)
            drop = s.get('drop') if (s.get('drop') is not None and s['drop'][0] > 0) else None
            check(lib.vi_attn_bwd(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), do.data_ptr(),
                                  do.stride(0), dq.data_ptr(), dq.stride(0), dk.data_ptr(), dk.stride(0), dv.data_ptr(),
                                  dv.stride(0), _dt(q), _ptr(s.get('key_mask')), _ptr(s.get('pair_dist')),
                                  _ptr(s.get('bias_affine')), _ptr(d_affine) if s.get('pair_dist') is not None else None,
                                  s['B'], ops.HEADS, s['Lq'], s['Lk'], ctx.mask_mode,
                                  float(drop[0]) if drop else 0.0, (int(drop[1]) & 0xFFFFFFFF) if drop else 0,
                                  drop[2].data_ptr() if drop else None, _stream()), 'vi_attn_bwd')
            _launched(1)
        extra = [None] * ctx.n_extra
        if ctx.n_extra == 2 and d_affine is not None:                   # sprel_linear.weight [1,1], .bias [1]
            extra = [d_affine[0:1].view(1, 1), d_affine[1:2]]
        return (None, None, None, None, *grads, *extra)


class SmallLinearFn(Function):
    """t = feat W^T + b for the tiny geometric features (feat_dim <= 16), fp32."""

    @staticmethod
    def forward(ctx, feat, w, b):
        feat = feat.contiguous()
        y = ops.gemm(feat, w.detach().contiguous(), b.detach() if b is not None else None)
        ctx.save_for_backward(feat)
        ctx.has_b, ctx.wshape = b is not None, w.shape
        return y

    @staticmethod
    def backward(ctx, dt):
        (feat,) = ctx.saved_tensors
        dt = dt.contiguous()
        fd = feat.shape[1]
        dW = torch.empty(ctx.wshape, dtype=F32, device=dt.device)
        db = torch.empty((HIDDEN,), dtype=F32, device=dt.device) if ctx.has_b else None
        sc = reduce_scratch(dt.device, dt.shape[0], HIDDEN, 17)
        check(lib.vi_feat_wgrad(dt.data_ptr(), feat.data_ptr(), fd, dW.data_ptr(), _ptr(db), dt.shape[0], sc.data_ptr(), sc.numel(),
                                _stream()), 'vi_feat_wgrad')
        _launched(2)
        return None, dW, db


class GatherRowsFn(Function):
    """rows = table[idx] (or table[row % period] when idx is None); adjoint = scatter-add."""

    @staticmethod
    def forward(ctx, table, idx, period, rows):
        table = table.contiguous()
        if idx is not None:
            y32, _ = ops.embed_compose(rows, table.device, idx=idx, table=table)
        else:
            y32, _ = ops.embed_compose(rows, table.device, pos_table=table, pos_period=period)
        ctx.save_for_backward(idx if idx is not None else table.new_empty(0, dtype=torch.int64))
        ctx.has_idx, ctx.period, ctx.tshape = idx is not None, period, table.shape
        return y32

    @staticmethod
    def backward(ctx, dy):
        (idx,) = ctx.saved_tensors
        dy = dy.contiguous()
        dt = torch.zeros(ctx.tshape, dtype=F32, device=dy.device)
        check(lib.vi_scatter_add_rows(dy.data_ptr(), idx.data_ptr() if ctx.has_idx else None, ctx.period or 1, dt.data_ptr(),
                                      dy.shape[0], _stream()), 'vi_scatter_add_rows')
        _launched(1)
        return dt, None, None, None


class SumRowsFn(Function):
    """y = sum of [rows, 768] tensors + broadcast [768] rows."""

    @staticmethod
    def forward(ctx, n_full, *tensors):
        full, consts = tensors[:n_full], tensors[n_full:]
        rows = full[0].shape[0]
        if n_full > 3 or len(consts) > 2:
            raise _lib.VlnImagineError('SumRowsFn: at most 3 row tensors and 2 constant rows')
        y32, _ = ops.embed_compose(rows, full[0].device, a=full[0].contiguous(),
                                   a2=full[1].contiguous() if n_full > 1 else None,
                                   a3=full[2].contiguous() if n_full > 2 else None,
                                   const_row=consts[0].detach() if len(consts) > 0 else None,
                                   const_row2=consts[1].detach() if len(consts) > 1 else None)
        ctx.n_full, ctx.n_const = n_full, len(consts)
        ctx.needs = [t.requires_grad for t in tensors]
        return y32

    @staticmethod
    def backward(ctx, dy):
        dy = dy.contiguous()
        g = [dy if ctx.needs[i] else None for i in range(ctx.n_full)]
        cs = None
        for i in range(ctx.n_const):
            if ctx.needs[ctx.n_full + i]:
                cs = colsum(dy) if cs is None else cs
                g.append(cs)
            else:
                g.append(None)
        return (None, *g)


class RowDotFn(Function):
    """out[r] = x[r] . w[g] + b[g]  (tail of ClsPrediction / NextActionPrediction), grouped rows."""

    @staticmethod
    def forward(ctx, x, wstack, bstack, ends, n_heads, *params):
        x = x.contiguous()
        rows = x.shape[0]
        out = torch.empty((rows,), dtype=F32, device=x.device)
        # the dot-product tail of vi_ln_dot without its LayerNorm (gamma = beta = NULL): one warp per row, all groups in one launch
        n_groups = 1 if ends is None else len(ends)
        check(lib.vi_ln_dot(x.data_ptr(), None, None, 0.0, wstack.data_ptr(), bstack.data_ptr(), out.data_ptr(), rows, n_groups,
                            _lib.int_array([min(int(e), rows) for e in ends]) if ends is not None else None, _stream()), 'vi_ln_dot')
        _launched(1)
        ctx.save_for_backward(x, wstack)
        ctx.ends, ctx.n_heads = ends, n_heads
        return out

    @staticmethod
    def backward(ctx, dout):
        x, wstack = ctx.saved_tensors
        dout = dout.contiguous()
        rows = x.shape[0]
        ends = ctx.ends
        n_groups = 1 if ends is None else len(ends)
        dx = torch.empty_like(x)
        dw = torch.empty((n_groups, HIDDEN), dtype=F32, device=x.device)
        db = torch.empty((n_groups, HIDDEN), dtype=F32, device=x.device)       # the sum replicated over the columns
        sc = reduce_scratch(x.device, rows, HIDDEN, 2)
        check(lib.vi_rowdot_bwd(dout.data_ptr(), x.data_ptr(), wstack.data_ptr(), dx.data_ptr(), dw.data_ptr(), db.data_ptr(), rows,
                                n_groups, _lib.int_array(list(ends)) if ends is not None else None, sc.data_ptr(), sc.numel(),
                                _stream()), 'vi_rowdot_bwd')
        _launched(4)
        pg = [dw[i].view(1, HIDDEN) for i in range(ctx.n_heads)] + [db[i, 0:1] for i in range(ctx.n_heads)]
        return (dx, None, None, None, None, *pg)


class FuseLogitsFn(Function):
    @staticmethod
    def forward(ctx, g_raw, l_raw, fuse_raw, gm, gv, nav, gids, cids, B, G, P):
        g_raw, l_raw = g_raw.contiguous(), l_raw.contiguous()
        gl, ll, fl = ops.duet_fuse_logits(g_raw, l_raw, fuse_raw, gm, gv, nav, gids, cids, B, G, P)
        ctx.save_for_backward(g_raw, l_raw, fuse_raw if fuse_raw is not None else g_raw.new_empty(0), gm, gv, nav, gids, cids)
        ctx.dims, ctx.has_fuse = (B, G, P), fuse_raw is not None
        return gl, ll, fl

    @staticmethod
    def backward(ctx, dgl, dll, dfl):
        g_raw, l_raw, fuse_raw, gm, gv, nav, gids, cids = ctx.saved_tensors
        B, G, P = ctx.dims
        c = lambda t: t.contiguous() if t is not None else None      # noqa: E731
        dgl, dll, dfl = c(dgl), c(dll), c(dfl)
        dg = torch.empty_like(g_raw)
        dl = torch.empty_like(l_raw)
        df = torch.empty((B,), dtype=F32, device=g_raw.device) if ctx.has_fuse else None
        check(lib.vi_duet_fuse_logits_bwd(g_raw.data_ptr(), l_raw.data_ptr(), fuse_raw.data_ptr() if ctx.has_fuse else None,
                                          gm.data_ptr(), gv.data_ptr(), nav.data_ptr(), gids.data_ptr(), cids.data_ptr(),
                                          _ptr(dgl), _ptr(dll), _ptr(dfl), dg.data_ptr(), dl.data_ptr(), _ptr(df), B, G, P,
                                          _stream()), 'vi_duet_fuse_logits_bwd')
        _launched(1)
        return dg, dl, df, None, None, None, None, None, None, None, None


class GatherSlotsFn(Function):
    """rows = src[slot[r]] (unit gather of the imagination slots that take part in the alignment loss)."""

    @staticmethod
    def forward(ctx, src, unit, slot, R, lowp):
        y32, y16 = ops.gather_mean(src, unit, slot, R, want16=lowp, want32=not lowp)
        ctx.save_for_backward(slot)
        ctx.shape = src.shape
        return y16 if lowp else y32

    @staticmethod
    def backward(ctx, dy):
        (slot,) = ctx.saved_tensors
        d = torch.zeros(ctx.shape, dtype=F32, device=dy.device)
        ops.scatter_rows(dy.float().contiguous(), slot, d)               # slots are unique: a plain row scatter
        return d, None, None, None, None


class ScatterSlotsFn(Function):
    """out = base with rows slot[r] replaced by rows[r] (the projected imaginations written back, vilmodel.py:646)."""

    @staticmethod
    def forward(ctx, base, rows, slot, unit):
        out = base.clone()
        ops.scatter_rows(rows.contiguous(), slot, out)
        ctx.save_for_backward(slot, unit)
        return out

    @staticmethod
    def backward(ctx, dout):
        slot, unit = ctx.saved_tensors
        dout = dout.contiguous()
        R = slot.shape[0]
        drows, _ = ops.gather_mean(dout, unit, slot, R, want16=False)
        dbase = dout.clone()
        dbase.index_fill_(0, slot.long(), 0.0)
        return dbase, drows, None, None


class CosineLossFn(Function):
    @staticmethod
    def forward(ctx, proj, tgt, R):
        proj, tgt = proj.contiguous(), tgt.contiguous()
        loss, _ = ops.cosine_loss(proj, tgt, R, proj.device)
        ctx.save_for_backward(proj, tgt)
        ctx.R = R
        ctx.needs = (proj.requires_grad, tgt.requires_grad)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        proj, tgt = ctx.saved_tensors
        dloss = dloss.contiguous().float().view(1)
        dp = torch.empty_like(proj) if ctx.needs[0] else None
        dt = torch.empty_like(tgt) if ctx.needs[1] else None
        check(lib.vi_cosine_loss_bwd(proj.data_ptr(), tgt.data_ptr(), dloss.data_ptr(), _ptr(dp), _ptr(dt), ctx.R, _stream()),
              'vi_cosine_loss_bwd')
        _launched(1)
        return dp, dt, None


class InfoNCELossFn(Function):
    """compute_contrastive_loss_infonce (models/vilmodel.py:657-687) with constant noun-phrase means; grad w.r.t. proj"""

    @staticmethod
    def forward(ctx, proj, tgt, negs, row_ep, neg_ep, temperature, R, n_negs):
        proj = proj.contiguous()
        loss, scratch = ops.infonce_loss(proj, tgt, negs, row_ep, neg_ep, temperature, R, n_negs, proj.device)
        ctx.save_for_backward(proj, tgt, scratch)
        ctx.extra = (negs, row_ep, neg_ep, float(temperature), R, n_negs)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        proj, tgt, scratch = ctx.saved_tensors
        negs, row_ep, neg_ep, temperature, R, n_negs = ctx.extra
        dloss = dloss.contiguous().float().view(1)
        dp = torch.empty_like(proj)
        check(lib.vi_infonce_loss_bwd(proj.data_ptr(), tgt.data_ptr(), _ptr(negs), row_ep.data_ptr(), _ptr(neg_ep), temperature,
                                      scratch.data_ptr(), dloss.data_ptr(), dp.data_ptr(), R, n_negs, _stream()),
              'vi_infonce_loss_bwd')
        _launched(1)
        return dp, None, None, None, None, None, None, None


class MarginLossFn(Function):
    """compute_contrastive_loss_margin (H/models/vilmodel_cmt.py:825-856) with constant noun-phrase means; grad w.r.t. proj"""

    @staticmethod
    def forward(ctx, proj, tgt, negs, row_ep, neg_ep, margin, R, n_negs):
        proj = proj.contiguous()
        loss, scratch = ops.margin_loss(proj, tgt, negs, row_ep, neg_ep, margin, R, n_negs, proj.device)
        ctx.save_for_backward(proj, tgt, scratch)
        ctx.extra = (negs, row_ep, neg_ep, float(margin), R, n_negs)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        proj, tgt, scratch = ctx.saved_tensors
        negs, row_ep, neg_ep, margin, R, n_negs = ctx.extra
        dloss = dloss.contiguous().float().view(1)
        dp = torch.empty_like(proj)
        check(lib.vi_margin_loss_bwd(proj.data_ptr(), tgt.data_ptr(), _ptr(negs), row_ep.data_ptr(), _ptr(neg_ep), margin,
                                     scratch.data_ptr(), dloss.data_ptr(), dp.data_ptr(), R, n_negs, _stream()),
              'vi_margin_loss_bwd')
        _launched(1)
        return dp, None, None, None, None, None, None, None


class MulBcastFn(Function):
    """y[b, r, :] = x[b, r, :] * s[b, :]   (x [B, R, 768], s [B, 768], both contiguous fp32) -> bf16 or fp32 rows [B*R, 768]"""

    @staticmethod
    def forward(ctx, x, s, lowp):
        x, s = x.contiguous(), s.contiguous()
        B, R, _ = x.shape
        y32, y16 = ops.mul_bcast(x, R * HIDDEN, s, HIDDEN, B, R, want16=lowp, want32=not lowp)
        ctx.save_for_backward(x, s)
        return y16 if lowp else y32

    @staticmethod
    def backward(ctx, dy):
        x, s = ctx.saved_tensors
        B, R, _ = x.shape
        dy = dy.float().contiguous().view(B, R, HIDDEN)
        dx, _ = ops.mul_bcast(dy, R * HIDDEN, s, HIDDEN, B, R, want16=False)
        ds = torch.empty_like(s)
        check(lib.vi_mul_bcast_bwd_s(dy.data_ptr(), x.data_ptr(), ds.data_ptr(), B, R, _stream()), 'vi_mul_bcast_bwd_s')
        _launched(1)
        return dx.view(B, R, HIDDEN), ds, None


class RaggedMeanFn(Function):
    """y[r] = mean of src[row_idx[offsets[r]:offsets[r+1]]] over RAGGED segments whose rows may repeat across segments (the
    noun-phrase / instruction token means of the alignment loss, D/models/vilmodel.py:617-641,781-806).  Adjoint: source row j
    receives sum over the segments r that contain it of dy[r] / len_r (a scatter-add of scaled copies).  Used when the text encoder
    trains through the alignment loss (fix_lang_inside_cosine_model off, :1256-1262)."""

    @staticmethod
    def forward(ctx, src, offsets, row_idx, R):
        src = src.contiguous()
        y32, _ = ops.gather_mean(src, offsets, row_idx, R, want16=False)
        ctx.save_for_backward(offsets, row_idx)
        ctx.shape, ctx.R = src.shape, R
        return y32

    @staticmethod
    def backward(ctx, dy):
        offsets, row_idx = ctx.saved_tensors
        dy = dy.contiguous()
        dev = dy.device
        R, n = ctx.R, row_idx.shape[0]
        lens = (offsets[1:R + 1] - offsets[:R]).long()
        inv = (1.0 / lens.to(F32))[:, None].expand(R, HIDDEN).contiguous()            # per-segment scale as a 768-wide row
        g, _ = ops.mul_bcast(dy, HIDDEN, inv, HIDDEN, R, 1, want16=False)              # dy[r] / len_r
        seg_of = torch.repeat_interleave(torch.arange(R, device=dev, dtype=torch.int64), lens, output_size=n)
        rows, _ = ops.embed_compose(n, dev, idx=seg_of, table=g)                       # one scaled copy per member row
        d = torch.zeros(ctx.shape, dtype=F32, device=dev)
        check(lib.vi_scatter_add_rows(rows.data_ptr(), row_idx.long().data_ptr(), 1, d.data_ptr(), n, _stream()), 'vi_scatter_add_rows')
        _launched(1)
        return d, None, None, None


class SegmentMeanFn(Function):
    """y[r] = mean of src[row_idx[offsets[r]:offsets[r+1]]] (equal-sized segments of ``seg`` rows, every source row in at most one
    segment): torch.mean over a token axis (HistoryEmbeddings' panorama mean, H/models/vilmodel_cmt.py:610; the imagination mean of
    act_pred_token 'ob_imagine_text', :1199).  Adjoint: every source row of segment r receives dy[r] / seg."""

    @staticmethod
    def forward(ctx, src, offsets, row_idx, R, seg):
        src = src.contiguous()
        y32, _ = ops.gather_mean(src, offsets, row_idx, R, want16=False)
        ctx.save_for_backward(row_idx)
        ctx.shape, ctx.R, ctx.seg = src.shape, R, seg
        return y32

    @staticmethod
    def backward(ctx, dy):
        (row_idx,) = ctx.saved_tensors
        dy = dy.contiguous()
        dev = dy.device
        R, seg = ctx.R, ctx.seg
        inv = torch.full((HIDDEN,), 1.0 / seg, dtype=F32, device=dev)
        g, _ = ops.mul_bcast(dy, HIDDEN, inv, 0, R, 1, want16=False)                  # dy / seg
        seg_of = torch.arange(R, device=dev, dtype=torch.int64).repeat_interleave(seg)
        rows, _ = ops.embed_compose(R * seg, dev, idx=seg_of, table=g)                # one copy per member row
        d = torch.zeros(ctx.shape, dtype=F32, device=dev)
        ops.scatter_rows(rows, row_idx, d)
        return d, None, None, None, None
