"""Transformer blocks of the navigation hot path, expressed as sequences of libvlnimagine launches.

Shared by the DUET (duet.py) and HAMT (hamt.py) host modules.  Activations travel as a pair
(fp32 residual stream, bf16 GEMM operand copy); in the fp32 check mode only the fp32 tensor exists.
Several token streams that run the same layer shape with different weights (DUET global/local
encoders, HAMT language/vision streams) are stacked along the row axis, each stream starting on
a 128-row boundary, and go through ONE grouped launch per GEMM / LayerNorm.
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional, Sequence

import torch

from . import autograd_ops as ag
from . import ops
from .feature_store import FeatureRows
from .ops import BF16, F32, HIDDEN, EPI_GELU, EPI_NONE, EPI_RELU, MASK_ADD_NEG10000, MASK_NEG_INF  # noqa: F401


# ----------------------------------------------------------------------------------------------
# training switch: while it is on, every block below records autograd nodes whose forward AND backward are
# libvlnimagine kernels (autograd_ops.py); while it is off the blocks are plain launch sequences
# ----------------------------------------------------------------------------------------------
class _Mode:
    train = False
    p_hidden = 0.0          # nn.Dropout(hidden_dropout_prob) sites (train() mode only)
    p_attn = 0.0            # attention_probs_dropout_prob
    p_head = 0.0            # pred_head_dropout_prob (HAMT NextActionPrediction)


class grad_mode:
    """with blocks.grad_mode(flag, drop=(p_hidden, p_attn)): ...  (set by the host modules once per mode call)"""

    def __init__(self, flag: bool, drop=(0.0, 0.0)):
        self.flag = bool(flag)
        self.drop = drop if self.flag else (0.0, 0.0)

    def __enter__(self):
        self.prev = (_Mode.train, _Mode.p_hidden, _Mode.p_attn, _Mode.p_head)
        _Mode.train, _Mode.p_hidden, _Mode.p_attn = self.flag, float(self.drop[0]), float(self.drop[1])
        _Mode.p_head = float(self.drop[2]) if len(self.drop) > 2 else 0.0

    def __exit__(self, *a):
        _Mode.train, _Mode.p_hidden, _Mode.p_attn, _Mode.p_head = self.prev


def _attn_drop(device, p=None):
    """(p, site, seed tensor) for an attention problem, or None"""
    p = _Mode.p_attn if p is None else p
    return (p, ag.next_site(), ag.dropout_seed(device)) if p > 0 else None


def _dense_res_ln(x, lin: 'LinearPack', res32, ln: 'LNPack', eps, lowp, ends):
    """training: LN(dropout(x W^T + b) + res)  (BertSelfOutput / BertOutput, D/models/vilmodel.py:151-155,190-194)"""
    if lowp and ag.dense_res_ln_ok(x, lin, ln, ends):
        y32, y16 = ag.dense_res_ln(x, res32, lin, ln, eps, ends, _Mode.p_hidden)       # one autograd node, dropout inside the LN kernels
        return Act(y32, y16)
    if _Mode.p_hidden > 0:
        d = ag.dropout(ag.linear(x, lin, lowp, out_dtype=F32, ends=ends), _Mode.p_hidden)
        return layer_norm(d, res32, ln, eps, lowp, ends)
    return layer_norm(ag.linear(x, lin, lowp, residual=res32, out_dtype=F32, ends=ends), None, ln, eps, lowp, ends)


def training() -> bool:
    return _Mode.train


# ----------------------------------------------------------------------------------------------
# derived weights (bf16 shadow copies, stacked groups), refreshed when a source parameter changes
# ----------------------------------------------------------------------------------------------
class _WeightsEpoch:
    """Counts optimiser steps process-wide.  Fused optimisers (torch.optim.AdamW(fused=True), apex) update parameters
    in place WITHOUT bumping their autograd version counters, so the version alone cannot tell that a derived copy is
    stale; a global optimizer-step hook can."""
    value = 0
    hooked = False

    @classmethod
    def install(cls):
        if cls.hooked:
            return
        cls.hooked = True
        try:
            from torch.optim.optimizer import register_optimizer_step_post_hook

            def _bump(optimizer, args, kwargs):
                cls.value += 1
                ag.advance_dropout_seeds()
            register_optimizer_step_post_hook(_bump)
        except ImportError:                                    # very old torch: version counters only
            pass


def weights_epoch() -> int:
    return _WeightsEpoch.value


def touch_weights():
    """call after updating parameters by any means that neither bumps tensor versions nor runs an optimizer step"""
    _WeightsEpoch.value += 1


class Pack:
    """Device tensors derived from parameters; rebuilt when any source's version / storage changes or an optimiser
    has stepped (in-place update, load_state_dict, .cuda()).  fp32 masters stay the nn.Parameters themselves."""

    def __init__(self, sources: Sequence[torch.Tensor], build):
        _WeightsEpoch.install()
        self.sources = list(sources)
        self._build = build
        self._key = None
        self._val = None

    def get(self):
        key = (_WeightsEpoch.value,) + tuple((p._version, p.data_ptr()) for p in self.sources)
        if key != self._key:
            with torch.no_grad():
                self._val = self._build()
            self._key = key
        return self._val


_FEAT_WT = {}


def feat_wt(w: torch.Tensor) -> torch.Tensor:
    """[feat_dim, 768] transposed fp32 copy of the weight of a small feature projection (nn.Linear(feat_dim, 768).weight), as
    vi_embed_compose reads it; cached per parameter and rebuilt with the weight version like every derived tensor"""
    e = _FEAT_WT.get(id(w))
    if e is None or e[0] is not w:
        e = (w, Pack([w], lambda: w.detach().t().contiguous().float()))
        _FEAT_WT[id(w)] = e
    return e[1].get()


ops.set_feat_wt_provider(feat_wt)


class LinearPack:
    """Rows-stacked weight [sum N_i, K] (+ bias) of one or several nn.Linear-shaped parameter sets."""

    def __init__(self, weights: Sequence[torch.Tensor], biases: Optional[Sequence[Optional[torch.Tensor]]] = None,
                 n_groups: int = 1):
        self.n_groups = n_groups           # row groups the stacked weight serves (DUET global | local, HAMT language | vision)
        self.weights = list(weights)
        self.biases = None if biases is None or all(b is None for b in biases) else list(biases)
        srcs = self.weights + ([b for b in self.biases if b is not None] if self.biases else [])
        self._pack = Pack(srcs, self._make)

    def _make(self):
        ws = [w.detach() for w in self.weights]
        w32 = (torch.cat(ws, 0) if len(ws) > 1 else ws[0]).contiguous()
        b = None
        if self.biases is not None:
            bs = [(b.detach() if b is not None else torch.zeros(w.shape[0], device=w.device)) for b, w in zip(self.biases, ws)]
            b = (torch.cat(bs, 0) if len(bs) > 1 else bs[0]).contiguous().float()
        return {'w32': w32, 'b': b}

    @staticmethod
    def _w16(v, fmt):
        key = ('w16', fmt)
        if key not in v:
            v[key] = ops.cast_h16(v['w32'], dtype=fmt)
        return v[key]

    def get(self, lowp: bool):
        """(weight, bias): the 16-bit shadow in the current operand format (ops.h16()) or the fp32 master"""
        v = self._pack.get()
        return (self._w16(v, ops.h16()) if lowp else v['w32']), v['b']

    def get_folded(self, ln: 'LNPack', n_groups: int):
        """LayerNorm ``ln`` (over this layer's 768 INPUT features) folded into the contraction, for vi_gemm16's VI_LN_FOLD:
        (W * gamma in the current 16-bit format [n_groups * N, K], s = its row sums, c = W beta + b), all per row group.
        Either side is broadcast when it has a single group (HAMT: shared cross-attention weights under per-stream
        LayerNorms).  Built once per weight version with torch ops in fp64 (weight preparation, not the data path)."""
        v = self._pack.get()
        g, be = ln.get()
        key = ('fold', id(ln), ops.h16(), n_groups)
        tok = (ln.g._pack._key, ln.b._pack._key)
        hit = v.get(key)
        if hit is not None and hit[0] == tok:
            return hit[1]
        with torch.no_grad():
            w = v['w32'].double()
            K = w.shape[1]
            G_lin = self.n_groups
            if G_lin not in (1, n_groups):
                raise ValueError('a pack of %d weight groups cannot serve a call with %d row groups' % (G_lin, n_groups))
            N = w.shape[0] // G_lin
            w = w.view(G_lin, N, K).expand(n_groups, N, K)
            gg = g.double().view(-1, K)
            bb = be.double().view(-1, K)
            gg = gg.expand(n_groups, K) if gg.shape[0] == 1 else gg
            bb = bb.expand(n_groups, K) if bb.shape[0] == 1 else bb
            wg16 = ops.cast_h16((w * gg[:, None, :]).float().reshape(n_groups * N, K).contiguous())
            s = wg16.double().sum(1).float().contiguous()
            c = torch.einsum('gnk,gk->gn', w, bb).reshape(n_groups * N)
            if v['b'] is not None:
                c = c + v['b'].double().view(G_lin, N).expand(n_groups, N).reshape(n_groups * N)
            val = (wg16, s, c.float().contiguous())
        v[key] = (tok, val)
        return val

    def get_grouped(self, lowp: bool, n_groups: int):
        """(weight, bias) for a call with ``n_groups`` row groups: a single-group pack is replicated (shared weights under
        per-group epilogue vectors)"""
        w, b = self.get(lowp)
        if self.n_groups == n_groups:
            return w, b
        if self.n_groups != 1:
            raise ValueError('a pack of %d weight groups cannot serve a call with %d row groups' % (self.n_groups, n_groups))
        v = self._pack.get()
        key = ('rep', w.dtype, n_groups)
        if key not in v:
            v[key] = (w.repeat(n_groups, 1).contiguous(), b.repeat(n_groups).contiguous() if b is not None else None)
        return v[key]

    def get_res_bias(self, ln: 'LNPack', n_groups: int):
        """beta of ``ln`` (over this layer's 768 OUTPUT features) + this layer's bias, [n_groups * 768], and gamma likewise:
        the two epilogue vectors of VI_LN_RESIDUAL"""
        v = self._pack.get()
        g, be = ln.get()
        key = ('resb', id(ln), n_groups)
        tok = (ln.g._pack._key, ln.b._pack._key)
        hit = v.get(key)
        if hit is not None and hit[0] == tok:
            return hit[1]
        with torch.no_grad():
            N = g.shape[-1]
            gg = g.view(-1, N)
            bb = be.view(-1, N)
            gg = (gg.expand(n_groups, N) if gg.shape[0] == 1 else gg).reshape(-1).contiguous()
            bb = (bb.expand(n_groups, N) if bb.shape[0] == 1 else bb).reshape(-1)
            if v['b'] is not None:
                bias = v['b'].view(-1, N)
                bb = bb + (bias.expand(n_groups, N) if bias.shape[0] == 1 else bias).reshape(-1)
            val = (gg, bb.contiguous())
        v[key] = (tok, val)
        return val

    def get_token(self):
        """changes whenever a source parameter does (in-place update or re-allocation)"""
        self._pack.get()
        return self._pack._key

    def get_t(self, lowp: bool, n_groups: int = 1):
        """per-group transposed weight [n_groups * K, N] (the B operand of the input-gradient GEMM), cached with
        the pack"""
        v = self._pack.get()
        key = ('t', lowp, n_groups)
        if key not in v:
            w = self._w16(v, BF16) if lowp else v['w32']
            n = w.shape[0] // n_groups
            with torch.no_grad():
                v[key] = torch.cat([ops.transpose(w[g * n:(g + 1) * n]) for g in range(n_groups)], 0).contiguous()
        return v[key]

    def grad_sources(self):
        """the parameters in the order LinearFn.backward returns their gradients"""
        return self.weights + ([b for b in self.biases if b is not None] if self.biases else [])


class StackPack:
    """[n, ...] stack of same-shaped vectors (LayerNorm gains/biases, head vectors) for grouped row kernels."""

    def __init__(self, tensors: Sequence[torch.Tensor]):
        self.tensors = list(tensors)
        self._pack = Pack(self.tensors, self._make)

    def _make(self):
        ts = [t.detach().reshape(-1) for t in self.tensors]
        return (torch.stack(ts, 0) if len(ts) > 1 else ts[0]).contiguous().float()

    def get(self):
        return self._pack.get()


class LNPack:
    def __init__(self, lns):
        self.g = StackPack([ln.weight for ln in lns])
        self.b = StackPack([ln.bias for ln in lns])

    def get(self):
        return self.g.get(), self.b.get()

    def grad_sources(self):
        return self.g.tensors + self.b.tensors


# ----------------------------------------------------------------------------------------------
# 16-bit operand format of the inference path
# ----------------------------------------------------------------------------------------------
_F16_MAX = 65504.0


def range_bound(model: torch.nn.Module) -> float:
    """Worst-case magnitude of any 16-bit tensor of the forward pass, from the weights alone.  Every tensor-core operand on
    this path is a LayerNorm output, a projection of one, a GELU / softmax-weighted average of projections, or the raw
    residual sum in front of a LayerNorm, so with A = max ||LN(x)||_2 <= sqrt(768) max|gamma| + ||beta||_2 and
    R = max row norm of any weight matrix:  projections <= R A + max|b| =: Y,  FFN outputs <= R sqrt(3072) Y + max|b|,
    residual sums <= A + that.  (Raw input features enter through a LayerNorm-ed projection and are cast with saturation.)"""
    A, R, bmax = 0.0, 0.0, 0.0
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.LayerNorm):
                A = max(A, float(m.weight.abs().max()) * m.weight.numel() ** 0.5 + float(m.bias.norm()))
            elif isinstance(m, torch.nn.Linear):
                R = max(R, float(m.weight.norm(dim=1).max()))
                if m.bias is not None:
                    bmax = max(bmax, float(m.bias.abs().max()))
            elif isinstance(m, torch.nn.MultiheadAttention):
                R = max(R, float(m.in_proj_weight.norm(dim=1).max()))
                bmax = max(bmax, float(m.in_proj_bias.abs().max()))
    Y = R * A + bmax
    return A + R * (3072 ** 0.5) * Y + bmax


def operand_format(model: torch.nn.Module, cache: dict, wanted: str = 'auto'):
    """torch.float16 or torch.bfloat16 for the 16-bit tensors of an inference call.  'auto': fp16 (same tensor-core rate,
    8x smaller rounding error than bf16 - what the >= 99.5 % action-agreement bar needs on near-tied logits) when
    ``range_bound`` proves that nothing can reach the fp16 range, else bf16.  Autograd-recording calls always use bf16."""
    if wanted == 'bf16' or torch.is_grad_enabled():
        return BF16
    if wanted == 'f16':
        return ops.F16
    if wanted != 'auto':
        raise ValueError("operand16 must be 'auto', 'f16' or 'bf16'")
    from .graphs import weights_token
    tok = weights_token(model, cache)
    if cache.get('fmt_tok') != tok:
        cache['fmt_tok'], cache['fmt'] = tok, (ops.F16 if range_bound(model) < 0.5 * _F16_MAX else BF16)
    return cache['fmt']


# ----------------------------------------------------------------------------------------------
# activations
# ----------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Pending:
    """A LayerNorm that has not been applied yet (inference, 16-bit mode): the activation holds the RAW pre-LayerNorm rows and
    the per-chunk row statistics their producer wrote; consumers fold the normalisation into their own contraction
    (vi_gemm16: VI_LN_FOLD for the next projection, VI_LN_RESIDUAL for the next residual add) - no LayerNorm pass."""
    stats: torch.Tensor                   # fp32 [24, rows, 2]: (mean, M2) of every 32-column chunk
    ln: 'LNPack'
    eps: float


@dataclasses.dataclass
class Act:
    f32: torch.Tensor                     # [rows, 768] fp32 residual stream
    b16: Optional[torch.Tensor] = None    # 16-bit copy fed to the tensor-core GEMMs (None in fp32 mode)
    pend: Optional[Pending] = None        # set: f32 / b16 are the raw rows of a pending LayerNorm

    def operand(self, lowp: bool):
        if self.pend is not None:
            raise RuntimeError('this activation carries a pending LayerNorm: use blocks.gemm_act / blocks.materialize')
        return self.b16 if lowp else self.f32


@dataclasses.dataclass
class Stream:
    """One token stream inside a row-stacked activation."""
    row0: int                       # first row (multiple of 128)
    B: int
    L: int                          # tokens per episode (padded length)
    mask: Optional[torch.Tensor]    # uint8 [B, L] key-padding mask (1 = valid) or None
    group: int = 0                  # weight block this stream uses
    pair_dist: Optional[torch.Tensor] = None   # fp32 [B, L, L] graph distances (GASA) or None
    bias_affine: Optional[torch.Tensor] = None  # device {w, b}
    affine_params: Optional[tuple] = None       # (sprel_linear.weight, .bias): gradient routing in training

    @property
    def rows(self):
        return self.B * self.L

    def view(self, t: torch.Tensor):
        return t[self.row0:self.row0 + self.rows]


def stack_layout(token_counts: Sequence[int]):
    """Row offsets for streams stacked on ops.ROW_ALIGN-row boundaries -> (row0 list, group_row_end list, total rows)."""
    row0, ends, cur = [], [], 0
    for i, n in enumerate(token_counts):
        row0.append(cur)
        last = i == len(token_counts) - 1
        cur = cur + n if last else ops.pad_rows(cur + n)
        ends.append(cur)
    return row0, ends, cur


_CTX_BUFFERS = {}


def _ctx_buffer(rows: int, like: torch.Tensor, streams) -> torch.Tensor:
    """Attention output buffer for a row-stacked activation.  The rows between streams (padding up to the next
    128-row boundary) are never written by the attention kernel but do flow through the following GEMM, whose
    rows are independent: they are zeroed so that the padding stays finite.
    Inference consumes the buffer at once (the output projection that follows reads it on the same stream), so one
    buffer per layout is allocated and zeroed ONCE and reused by every layer and every step - it used to cost one fill
    launch per attention call (8 of the ~70 launches of a DUET step).  Autograd keeps the attention output for the
    backward pass and therefore gets a fresh buffer each time."""
    pads = [(a.row0 + a.rows, b.row0) for a, b in zip(streams[:-1], streams[1:]) if b.row0 > a.row0 + a.rows]
    key = None
    if not _Mode.train and not torch.is_grad_enabled():
        key = (rows, like.dtype, like.device, tuple((s.row0, s.rows) for s in streams))
        ctx = _CTX_BUFFERS.get(key)
        if ctx is not None:
            return ctx
    ctx = torch.empty((rows, HIDDEN), dtype=like.dtype, device=like.device)
    for r0, r1 in pads:
        ctx[r0:r1].zero_()
    # never keep memory of a graph's private pool, and never evict: captured graphs hold raw pointers to these buffers
    if key is not None and not torch.cuda.is_current_stream_capturing() and len(_CTX_BUFFERS) < 256:
        _CTX_BUFFERS[key] = ctx
    return ctx


def _call_groups(lin: 'LinearPack', ln: Optional['LNPack'], ends):
    """(n_groups, ends) of a grouped call: as many groups as the weights or the LayerNorm vectors need"""
    n = max(lin.n_groups, len(ln.g.tensors) if ln is not None else 1)
    if n > 1 and (ends is None or len(ends) != n):
        raise ValueError('a call over %d weight / LayerNorm groups needs %d row-group ends' % (n, n))
    return n, (list(ends) if n > 1 else None)


def gemm_act(x: Act, lin: 'LinearPack', lowp: bool, ends=None, epilogue=EPI_NONE, out_dtype=None) -> torch.Tensor:
    """epi(x W^T + b) over an activation (inference); a pending LayerNorm of x is folded into the contraction."""
    if x.pend is not None:
        n, e = _call_groups(lin, x.pend.ln, ends)
        wg, sv, c = lin.get_folded(x.pend.ln, n)
        return ops.gemm(x.b16, wg, c, epilogue=epilogue, out_dtype=out_dtype, group_row_end=e,
                        ln=(ops.LN_FOLD, sv, x.pend.stats, x.pend.eps))
    n, e = _call_groups(lin, None, ends)
    w, b = lin.get(lowp)
    return ops.gemm(x.operand(lowp), w, b, epilogue=epilogue, out_dtype=out_dtype, group_row_end=e)


def linear_residual_ln(x, lin: 'LinearPack', res: Act, ln: LNPack, eps, lowp, ends=None, defer=False) -> Act:
    """LN(x W^T + b + res) (inference).  16-bit mode: ONE contraction writes the raw sum (fp32 + 16-bit) and its row
    statistics, the LayerNorm stays pending for the consumers (``defer``) or is applied by one row kernel; a pending
    LayerNorm of ``res`` is applied to the residual inside the same epilogue.  fp32 check mode: GEMM + row kernel."""
    if isinstance(res, torch.Tensor):
        res = Act(res)
    if not lowp:
        if res.pend is not None:
            res = materialize(res, lowp, ends)
        n, e = _call_groups(lin, ln, ends)
        w, b = lin.get_grouped(lowp, n)
        g, be = ln.get()
        ao = ops.gemm(x, w, b, residual=res.f32, out_dtype=F32, group_row_end=e)
        y32, y16 = ops.add_ln(ao, None, g, be, eps, want16=lowp, group_row_end=e if len(ln.g.tensors) > 1 else None)
        return Act(y32, y16)
    rows = x.shape[0]
    z32 = torch.empty((rows, HIDDEN), dtype=F32, device=x.device)
    z16 = torch.empty((rows, HIDDEN), dtype=x.dtype, device=x.device)
    stats = torch.empty((HIDDEN // 32, rows, 2), dtype=F32, device=x.device)
    if res.pend is not None:
        n, e = _call_groups(lin, res.pend.ln, ends)
        w, _ = lin.get_grouped(lowp, n)
        g, bb = lin.get_res_bias(res.pend.ln, n)
        ops.gemm(x, w, bb, residual=res.f32, out=z32, out16=z16, group_row_end=e, stats_out=stats,
                 ln=(ops.LN_RESIDUAL, g, res.pend.stats, res.pend.eps))
    else:
        n, e = _call_groups(lin, None, ends)
        w, b = lin.get(lowp)
        ops.gemm(x, w, b, residual=res.f32, out=z32, out16=z16, group_row_end=e, stats_out=stats)
    out = Act(z32, z16, Pending(stats, ln, eps))
    return out if defer else materialize(out, lowp, ends)


def materialize(x: Act, lowp: bool, ends=None, want16: bool = True) -> Act:
    """apply a pending LayerNorm with the row kernel (outputs of the encoder, inputs of the heads)"""
    if x.pend is None:
        return x
    g, be = x.pend.ln.get()
    y32, y16 = ops.add_ln(x.f32, None, g, be, x.pend.eps, want16=lowp and want16,
                          group_row_end=list(ends) if (ends is not None and len(x.pend.ln.g.tensors) > 1) else None)
    return Act(y32, y16)


def layer_norm(x32, res32, ln: LNPack, eps, lowp, ends=None) -> Act:
    if _Mode.train:
        y32, y16 = ag.layer_norm(x32, res32, ln, eps, lowp, ends)
        return Act(y32, y16)
    g, b = ln.get()
    y32, y16 = ops.add_ln(x32, res32, g, b, eps, want16=lowp, group_row_end=ends)
    return Act(y32, y16)


# ----------------------------------------------------------------------------------------------
# blocks
# ----------------------------------------------------------------------------------------------
class SelfFFNPack:
    """Weights of BertAttention + BertIntermediate + BertOutput for one or several stacked streams."""

    def __init__(self, attns, inters, outs):
        # attns: modules with .self.{query,key,value} and .output.{dense,LayerNorm}
        n = len(attns)
        self.qkv = LinearPack([w for a in attns for w in (a.self.query.weight, a.self.key.weight, a.self.value.weight)],
                              [b for a in attns for b in (a.self.query.bias, a.self.key.bias, a.self.value.bias)], n_groups=n)
        self.o = LinearPack([a.output.dense.weight for a in attns], [a.output.dense.bias for a in attns], n_groups=n)
        self.ln1 = LNPack([a.output.LayerNorm for a in attns])
        self.w1 = LinearPack([m.dense.weight for m in inters], [m.dense.bias for m in inters], n_groups=n)
        self.w2 = LinearPack([m.dense.weight for m in outs], [m.dense.bias for m in outs], n_groups=n)
        self.ln2 = LNPack([m.LayerNorm for m in outs])


def attn(x: Act, qkv: LinearPack, o: LinearPack, ln: LNPack, streams: List[Stream], ends, lowp: bool, eps=1e-12,
         kv_of=None) -> Act:
    """LN(x + O(attn(QKV(x)))) over all rows, the LayerNorm left pending in inference.  Stream i reads the keys / values of
    streams[kv_of[i]] (default: its own, self-attention).  HAMT's cross-modal layer is kv_of = (1, 0): both directions share
    one QKV / output projection (H/models/vilmodel_cmt.py:385-397).  Group ends reach a call only when its weights or
    LayerNorm have per-stream groups."""
    rows = x.f32.shape[0]
    kvs = streams if kv_of is None else [streams[j] for j in kv_of]
    if _Mode.train:
        xin = x.operand(lowp)
        t = ag.linear(xin, qkv, lowp, ends=_call_groups(qkv, None, ends)[1])
        spec, extras = [], ()
        for s, k in zip(streams, kvs):
            spec.append(dict(q=(0, s.row0, 0), k=(0, k.row0, HIDDEN), v=(0, k.row0, 2 * HIDDEN), B=s.B, Lq=s.L, Lk=k.L,
                             key_mask=k.mask, pair_dist=s.pair_dist, bias_affine=s.bias_affine, out_row0=s.row0,
                             drop=_attn_drop(xin.device)))
            if s.pair_dist is not None and s.affine_params is not None:
                extras = tuple(s.affine_params)
        ctx = ag.AttentionFn.apply(spec, rows, MASK_ADD_NEG10000, 1, t, *extras)
        return _dense_res_ln(ctx, o, x.f32, ln, eps, lowp, _call_groups(o, ln, ends)[1])
    t = gemm_act(x, qkv, lowp, ends)                                   # [rows, 2304]
    ctx = _ctx_buffer(rows, t, streams)
    ops.attention_multi([dict(q=s.view(t)[:, 0:HIDDEN], k=k.view(t)[:, HIDDEN:2 * HIDDEN], v=k.view(t)[:, 2 * HIDDEN:3 * HIDDEN],
                              out=s.view(ctx), B=s.B, Lq=s.L, Lk=k.L, key_mask=k.mask, pair_dist=s.pair_dist,
                              bias_affine=s.bias_affine) for s, k in zip(streams, kvs)])
    return linear_residual_ln(ctx, o, x, ln, eps, lowp, ends, defer=True)


def self_attn_ffn(x: Act, pk: SelfFFNPack, streams: List[Stream], ends, lowp: bool, eps=1e-12, defer=False) -> Act:
    """Post-LN BERT layer: LN(x + O(attn(QKV(x)))) then LN(y + W2 gelu(W1 y)).  ``defer``: the last LayerNorm may stay
    pending for the next block (blocks.Pending).
    Reference: BertLayer, VLN-DUET/map_nav_src/models/vilmodel.py:196-209 (and :80-194)."""
    y = attn(x, pk.qkv, pk.o, pk.ln1, streams, ends, lowp, eps)
    return ffn(y, pk.w1, pk.w2, pk.ln2, ends, lowp, eps, defer=defer)


def ffn(y: Act, w1: LinearPack, w2: LinearPack, ln2: LNPack, ends, lowp: bool, eps=1e-12, defer=False) -> Act:
    if _Mode.train:
        h = ag.ActFn.apply(ag.linear(y.operand(lowp), w1, lowp, ends=ends), EPI_GELU)
        return _dense_res_ln(h, w2, y.f32, ln2, eps, lowp, ends)
    h = gemm_act(y, w1, lowp, ends, epilogue=EPI_GELU)                 # [rows, 3072]
    return linear_residual_ln(h, w2, y, ln2, eps, lowp, ends, defer=defer)


class CrossPack:
    """BertXAttention weights: query / output per stream group; key+value stacked per context user."""

    def __init__(self, xatts):
        n = len(xatts)
        self.q = LinearPack([x.att.query.weight for x in xatts], [x.att.query.bias for x in xatts], n_groups=n)
        self.kv = LinearPack([w for x in xatts for w in (x.att.key.weight, x.att.value.weight)],
                             [b for x in xatts for b in (x.att.key.bias, x.att.value.bias)])
        self.o = LinearPack([x.output.dense.weight for x in xatts], [x.output.dense.bias for x in xatts], n_groups=n)
        self.ln = LNPack([x.output.LayerNorm for x in xatts])


def cross_attn(x: Act, ctxs, pk: CrossPack, streams: List[Stream], ends, lowp: bool, eps=1e-12, defer=False) -> Act:
    """LN(x + O(attn(Q(x), K(ctx), V(ctx)))).  ctxs[i] = (kv, col0, ctx_len, key_mask) is the context of streams[i]: the
    projected context [B*ctx_len, *] with its K at columns col0 and V at col0+768.  Streams may share one kv tensor.
    Reference: BertXAttention, VLN-DUET/map_nav_src/models/vilmodel.py:302-364."""
    rows = x.f32.shape[0]
    if _Mode.train:
        xin = x.operand(lowp)
        q = ag.linear(xin, pk.q, lowp, ends=ends)
        kvs, spec = [], []
        for s, (kv, c0, n, m) in zip(streams, ctxs):
            if not any(kv is t for t in kvs):
                kvs.append(kv)
            bi = 1 + next(i for i, t in enumerate(kvs) if t is kv)
            spec.append(dict(q=(0, s.row0, 0), k=(bi, 0, c0), v=(bi, 0, c0 + HIDDEN), B=s.B, Lq=s.L, Lk=n, key_mask=m,
                             out_row0=s.row0, drop=_attn_drop(xin.device)))
        ctx = ag.AttentionFn.apply(spec, rows, MASK_ADD_NEG10000, 1 + len(kvs), q, *kvs)
        return _dense_res_ln(ctx, pk.o, x.f32, pk.ln, eps, lowp, ends)
    q = gemm_act(x, pk.q, lowp, ends)
    ctx = _ctx_buffer(rows, q, streams)
    ops.attention_multi([dict(q=s.view(q), k=kv[:, c0:c0 + HIDDEN], v=kv[:, c0 + HIDDEN:c0 + 2 * HIDDEN], out=s.view(ctx),
                              B=s.B, Lq=s.L, Lk=n, key_mask=m) for s, (kv, c0, n, m) in zip(streams, ctxs)])
    return linear_residual_ln(ctx, pk.o, x, pk.ln, eps, lowp, ends, defer=defer)


def linear(x: torch.Tensor, pk: LinearPack, lowp: bool, out_dtype=None, ends=None, residual=None, epilogue=EPI_NONE) -> torch.Tensor:
    """y = epi(x W^T + b) [+ residual] for a LinearPack; differentiable in training (the activation as its own node)."""
    if _Mode.train:
        y = ag.linear(x, pk, lowp, residual=residual, out_dtype=out_dtype, ends=ends)
        return ag.ActFn.apply(y, epilogue) if epilogue != EPI_NONE else y
    w, b = pk.get(lowp)
    return ops.gemm(x, w, b, residual=residual, epilogue=epilogue, out_dtype=out_dtype or (x.dtype if lowp else F32),
                    group_row_end=ends)


def stack_rows(parts: Sequence[torch.Tensor], row0: Sequence[int]) -> torch.Tensor:
    """fp32 rows of several streams -> one tensor with stream i at row0[i] (stack_layout) and zero rows in the gaps
    between streams"""
    out, cur = [], 0
    for p, r0 in zip(parts, row0):
        if r0 > cur:
            out.append(torch.zeros((r0 - cur, HIDDEN), dtype=F32, device=p.device))
        out.append(p)
        cur = r0 + p.shape[0]
    return torch.cat(out, 0)


def embed_streams(specs, row0: Sequence[int], rows: int, device, lowp: bool) -> Act:
    """Input embeddings of several streams (one ``embed`` keyword dict per stream, with its 'rows') stacked on the
    stack_layout boundaries.  Inference: each composer launch writes its slice of one preallocated activation and
    zero-fills the gap behind it.  Training: one ``embed`` node per stream, stacked by stack_rows."""
    if _Mode.train:
        return as_act(stack_rows([embed(device=device, **kw).f32 for kw in specs], row0), lowp)
    x32 = torch.empty((rows, HIDDEN), dtype=F32, device=device)
    x16 = torch.empty((rows, HIDDEN), dtype=ops.h16(), device=device) if lowp else None
    for i, kw in enumerate(specs):
        r0, r1 = row0[i], (row0[i + 1] if i + 1 < len(row0) else rows)
        embed(device=device, y32=x32[r0:r1], y16=x16[r0:r1] if lowp else None, zero_rows=r1 - r0 - kw['rows'], **kw)
    return Act(x32, x16)


def stack_segments(parts, row0: Sequence[int], lowp: bool) -> Act:
    """Streams made of token segments: parts[i] lists the fp32 [B, n_k, 768] segments that stream i concatenates along its
    tokens, stacked on the stack_layout boundaries.  Inference: one vi_copy_rows per segment into one preallocated
    activation, the gap behind each stream zero-filled.  Training: torch.cat per stream, stacked by stack_rows."""
    if _Mode.train:
        return as_act(stack_rows([(s[0] if len(s) == 1 else torch.cat(s, 1)).reshape(-1, HIDDEN) for s in parts], row0), lowp)
    B, dev = parts[0][0].shape[0], parts[0][0].device
    lens = [sum(seg.shape[1] for seg in s) for s in parts]
    rows = row0[-1] + B * lens[-1]
    x32 = torch.empty((rows, HIDDEN), dtype=F32, device=dev)
    x16 = torch.empty((rows, HIDDEN), dtype=ops.h16(), device=dev) if lowp else None
    for i in range(len(parts) - 1):
        r0, r1 = row0[i] + B * lens[i], row0[i + 1]
        if r1 > r0:
            x32[r0:r1].zero_()
            if lowp:
                x16[r0:r1].zero_()
    for s, r0, n in zip(parts, row0, lens):
        for seg in s:
            k = seg.shape[1]
            ops.copy_rows(seg, k * HIDDEN, HIDDEN, B, k, x32[r0:], x16[r0:] if lowp else None, n * HIDDEN, HIDDEN)
            r0 += k
    return Act(x32, x16)


def take_rows(v: torch.Tensor, lowp: Optional[bool] = None) -> torch.Tensor:
    """[B, n, 768] view of episode-strided fp32 rows -> contiguous [B * n, 768] rows (fp32); with ``lowp`` given, the GEMM
    operand of that precision instead.  Inference: one vi_copy_rows reading the view in place."""
    if _Mode.train:
        y = v.reshape(-1, HIDDEN)
        return y.contiguous() if lowp is None else operand(y, lowp)
    B, n = v.shape[0], v.shape[1]
    y32 = torch.empty((B * n, HIDDEN), dtype=F32, device=v.device) if not lowp else None
    y16 = torch.empty((B * n, HIDDEN), dtype=ops.h16(), device=v.device) if lowp else None
    ops.copy_rows(v, v.stride(0), HIDDEN, B, n, y32, y16, n * HIDDEN, HIDDEN)
    return y16 if lowp else y32


def mul_bcast(x: torch.Tensor, s: torch.Tensor, lowp: bool) -> torch.Tensor:
    """y[b, r] = x[b, r] * s[b] for x a [B, n, 768] and s a [B, 768] view of fp32 rows -> the [B * n, 768] GEMM operand.
    Inference: one vi_mul_bcast reading both views in place.  Training: MulBcastFn."""
    if _Mode.train:
        return ag.MulBcastFn.apply(x, s, lowp)
    y32, y16 = ops.mul_bcast(x, x.stride(0), s, s.stride(0), x.shape[0], x.shape[1], want16=lowp, want32=not lowp)
    return y16 if lowp else y32


def mask_logits(raw: torch.Tensor, keep: torch.Tensor) -> torch.Tensor:
    """raw logits, one per row -> logits shaped like ``keep`` with -inf where keep == 0 (padding navigation type, no object).
    Inference: vi_mask_logits_navtype.  Training: masked_fill."""
    if _Mode.train:
        return raw.view(keep.shape).masked_fill(keep == 0, float('-inf'))
    return ops.mask_logits_navtype(raw, keep.long().contiguous().view(-1)).view(keep.shape)


def gather_rows(src: torch.Tensor, idx, n: int, lowp: Optional[bool] = None) -> torch.Tensor:
    """rows = src[idx] (fp32); with ``lowp`` given, the GEMM operand of that precision instead.  Inference: one
    vi_gather_mean over unit segments.  Training: GatherRowsFn (adjoint: scatter-add)."""
    dev = src.device
    if _Mode.train:
        y = ag.GatherRowsFn.apply(src, torch.as_tensor(idx).to(dev, torch.int64, non_blocking=True), 0, n)
        return y if lowp is None else operand(y, lowp)
    unit = torch.arange(n + 1, dtype=torch.int32, device=dev)
    idx = torch.as_tensor(idx).to(dev, torch.int32, non_blocking=True)
    if lowp is None:
        return ops.gather_mean(src, unit, idx, n, want16=False)[0]
    y32, y16 = ops.gather_mean(src, unit, idx, n, want16=lowp, want32=not lowp)
    return y16 if lowp else y32


def segment_mean(src: torch.Tensor, offsets, rows, n: int, seg: Optional[int] = None) -> torch.Tensor:
    """y[r] = mean of src[rows[offsets[r]:offsets[r+1]]] over ragged segments (int32 index arrays).  Inference: one
    vi_gather_mean.  Training: RaggedMeanFn (a source row may sit in several segments); with ``seg`` given, disjoint segments
    of ``seg`` rows each, SegmentMeanFn (its adjoint is a plain row scatter)."""
    offsets = torch.as_tensor(offsets).to(src.device)
    rows = torch.as_tensor(rows).to(src.device)
    if _Mode.train:
        if seg is not None:
            return ag.SegmentMeanFn.apply(src, offsets, rows, n, seg)
        return ag.RaggedMeanFn.apply(src, offsets, rows, n)
    return ops.gather_mean(src, offsets, rows, n, want16=False)[0]


def as_act(x32: torch.Tensor, lowp: bool) -> Act:
    """fp32 rows -> activation pair (adds the bf16 operand copy in bf16 mode)."""
    x32 = x32.contiguous()
    if _Mode.train:
        return Act(x32, ag.CastBf16Fn.apply(x32) if lowp else None)
    return Act(x32, ops.cast_h16(x32) if lowp else None)


def operand(x32: torch.Tensor, lowp: bool) -> torch.Tensor:
    """fp32 rows -> GEMM operand of the current precision (differentiable in training)"""
    x32 = x32.contiguous()
    if not lowp:
        return x32
    return ag.CastBf16Fn.apply(x32) if _Mode.train else ops.cast_h16(x32)


def feature_operand(x, lowp: bool) -> torch.Tensor:
    """image features (dense [..., F] or feature_store.FeatureRows) -> the [rows, F] operand of their first GEMM (fp32 rows when
    not ``lowp``).  Dense: the cast of ``operand``.  FeatureRows: one vi_gather_rows from the store, with the environment
    dropout the host module attached (same mask and values as dropout on the dense tensor followed by the cast)."""
    if isinstance(x, FeatureRows):
        dtype = (BF16 if _Mode.train else ops.h16()) if lowp else F32
        return x.gather(dtype, ag.dropout_seed(x.device) if x.drop is not None else None)
    return operand(x.float().reshape(-1, x.shape[-1]), lowp)


def embed(rows: int, device, *, a=None, a_ln=None, a2=None, feat=None, feat_lin=None, feat_ln=None, idx=None, table=None,
          pos_table=None, pos_period=0, const_rows=(), out_ln=None, eps=1e-12, lowp=False, y32=None, y16=None,
          dropout=False, chain_ln=None, chain_eps=1e-5, zero_rows=0, want32=True) -> Act:
    """Input-embedding composer  LN_out([LN_a](a) + a2 + LN_f(W feat + b) + table[idx] + pos[row % period] + consts).
    *_ln are nn.LayerNorm-like parameter holders, feat_lin an nn.Linear-like holder.  Inference: ONE fused kernel
    (vi_embed_compose), which also zero-fills ``zero_rows`` rows behind the output; ``want32=False`` skips its fp32 output
    when the 16-bit one is all the caller reads.  Training: the same sum built from differentiable primitives (autograd_ops)."""
    ln_pair = lambda m: (m.weight, m.bias) if m is not None else None      # noqa: E731
    if not _Mode.train:
        consts = list(const_rows) + [None, None]
        if chain_ln is not None:
            # inference, 16-bit mode: the 16-bit output is chain_ln(result), the operand of the first pre-norm contraction
            o32, o16 = ops.embed_compose(rows, device, a=a, a_ln=ln_pair(a_ln), feat=feat,
                                         feat_w=feat_lin.weight if feat_lin is not None else None,
                                         feat_b=feat_lin.bias if feat_lin is not None else None, feat_ln=ln_pair(feat_ln),
                                         idx=idx, table=table, pos_table=pos_table, pos_period=pos_period,
                                         const_row=consts[0], const_row2=consts[1], out_ln=ln_pair(out_ln), eps=eps,
                                         want16=True, want32=True, ln2=ln_pair(chain_ln), ln2_eps=chain_eps)
            return Act(o32, o16)
        o32, o16 = ops.embed_compose(rows, device, a=a, a2=a2, a_ln=ln_pair(a_ln), feat=feat,
                                     feat_w=feat_lin.weight if feat_lin is not None else None,
                                     feat_b=feat_lin.bias if feat_lin is not None else None, feat_ln=ln_pair(feat_ln),
                                     idx=idx, table=table, pos_table=pos_table, pos_period=pos_period,
                                     const_row=consts[0], const_row2=consts[1], out_ln=ln_pair(out_ln), eps=eps,
                                     y32=y32, y16=y16, want16=lowp and y16 is None and (y32 is None), want32=want32,
                                     zero_rows=zero_rows)
        return Act(o32, o16)
    terms = []
    if a is not None:
        if a_ln is not None:
            t, _ = ag.LayerNormFn.apply(a, None, a_ln.weight, a_ln.bias, eps, False, None, 2, a_ln.weight, a_ln.bias)
            terms.append(t)
        else:
            terms.append(a)
    if a2 is not None:
        terms.append(a2)
    if feat is not None:
        t = ag.SmallLinearFn.apply(feat, feat_lin.weight, feat_lin.bias)
        if feat_ln is not None:
            t, _ = ag.LayerNormFn.apply(t, None, feat_ln.weight, feat_ln.bias, eps, False, None, 2, feat_ln.weight, feat_ln.bias)
        terms.append(t)
    if idx is not None:
        terms.append(ag.GatherRowsFn.apply(table, idx, 0, rows))
    if pos_table is not None:
        terms.append(ag.GatherRowsFn.apply(pos_table, None, pos_period, rows))
    consts = list(const_rows)
    while len(terms) > 3:                                     # the fused sum kernel takes three row tensors
        terms = [ag.SumRowsFn.apply(3, *terms[:3])] + terms[3:]
    s = ag.SumRowsFn.apply(len(terms), *terms, *consts) if (len(terms) > 1 or consts) else terms[0]
    drop = dropout and _Mode.p_hidden > 0                     # nn.Dropout after the embedding LayerNorm (vilmodel.py:77,1124)
    if out_ln is not None:
        o32, o16 = ag.LayerNormFn.apply(s, None, out_ln.weight, out_ln.bias, eps, lowp and not drop, None, 2, out_ln.weight, out_ln.bias)
        if drop:
            o32 = ag.dropout(o32, _Mode.p_hidden)
            return Act(o32, ag.CastBf16Fn.apply(o32) if lowp else None)
        return Act(o32, o16 if lowp else None)
    if drop:
        s = ag.dropout(s, _Mode.p_hidden)
    return Act(s, ag.CastBf16Fn.apply(s) if lowp else None)


def mask_u8(m: Optional[torch.Tensor]):
    """bool mask -> the uint8 view the kernels read (zero-copy for contiguous bool tensors)."""
    if m is None:
        return None
    if m.dtype == torch.bool and m.is_contiguous():
        return m.view(torch.uint8)
    return m.to(torch.uint8).contiguous()


class PanoLayerPack:
    """Weights of one pre-norm TransformerEncoderLayer of the panorama encoder."""

    def __init__(self, layer):
        self.norm1 = LNPack([layer.norm1])
        self.qkv = LinearPack([layer.self_attn.in_proj_weight], [layer.self_attn.in_proj_bias])
        self.o = LinearPack([layer.self_attn.out_proj.weight], [layer.self_attn.out_proj.bias])
        self.norm2 = LNPack([layer.norm2])
        self.w1 = LinearPack([layer.linear1.weight], [layer.linear1.bias])
        self.w2 = LinearPack([layer.linear2.weight], [layer.linear2.bias])


def pano_layer(x32: torch.Tensor, pk: PanoLayerPack, B: int, L: int, key_mask, lowp: bool, eps=1e-5) -> torch.Tensor:
    """Pre-norm layer: x += O(attn(QKV(LN1 x))) ; x += W2 gelu(W1 LN2 x).  The key-padding mask is the
    -inf kind of nn.MultiheadAttention.  Reference: TransformerEncoderLayer.forward_pre,
    VLN-DUET/map_nav_src/models/transformer.py:170-182."""
    h = layer_norm(x32, None, pk.norm1, eps, lowp)
    if _Mode.train:
        qkv = ag.linear(h.operand(lowp), pk.qkv, lowp)
        ph = _Mode.p_hidden
        spec = [dict(q=(0, 0, 0), k=(0, 0, HIDDEN), v=(0, 0, 2 * HIDDEN), B=B, Lq=L, Lk=L, key_mask=key_mask, out_row0=0,
                     drop=_attn_drop(x32.device, ph))]
        ctx = ag.AttentionFn.apply(spec, B * L, MASK_NEG_INF, 1, qkv)
        if ph > 0:                                            # src + dropout1(src2); linear2(dropout(act)); src + dropout2
            x32 = ag.SumRowsFn.apply(2, x32, ag.dropout(ag.linear(ctx, pk.o, lowp, out_dtype=F32), ph))
            h = layer_norm(x32, None, pk.norm2, eps, lowp)
            f = ag.dropout(ag.ActFn.apply(ag.linear(h.operand(lowp), pk.w1, lowp), EPI_GELU), ph)
            return ag.SumRowsFn.apply(2, x32, ag.dropout(ag.linear(f, pk.w2, lowp, out_dtype=F32), ph))
        x32 = ag.linear(ctx, pk.o, lowp, residual=x32, out_dtype=F32)
        h = layer_norm(x32, None, pk.norm2, eps, lowp)
        f = ag.ActFn.apply(ag.linear(h.operand(lowp), pk.w1, lowp), EPI_GELU)
        return ag.linear(f, pk.w2, lowp, residual=x32, out_dtype=F32)
    w, b = pk.qkv.get(lowp)
    qkv = ops.gemm(h.operand(lowp), w, b)
    ctx = ops.attention(qkv[:, 0:HIDDEN], qkv[:, HIDDEN:2 * HIDDEN], qkv[:, 2 * HIDDEN:3 * HIDDEN], B, L, L,
                        key_mask=key_mask, mask_mode=MASK_NEG_INF)
    w, b = pk.o.get(lowp)
    x32 = ops.gemm(ctx, w, b, residual=x32, out_dtype=F32)
    h = layer_norm(x32, None, pk.norm2, eps, lowp)
    w, b = pk.w1.get(lowp)
    f = ops.gemm(h.operand(lowp), w, b, epilogue=EPI_GELU)
    w, b = pk.w2.get(lowp)
    return ops.gemm(f, w, b, residual=x32, out_dtype=F32)


def _dense_raw(x16: torch.Tensor, lin: 'LinearPack', res32: torch.Tensor, want_stats: bool):
    """x W^T + b + res -> (fp32 rows, 16-bit copy, row statistics) of a pre-norm residual stream (16-bit mode)"""
    rows = x16.shape[0]
    w, b = lin.get(True)
    z32 = torch.empty((rows, HIDDEN), dtype=F32, device=x16.device)
    if not want_stats:
        ops.gemm(x16, w, b, residual=res32, out=z32)
        return z32, None, None
    z16 = torch.empty((rows, HIDDEN), dtype=x16.dtype, device=x16.device)
    stats = torch.empty((HIDDEN // 32, rows, 2), dtype=F32, device=x16.device)
    ops.gemm(x16, w, b, residual=res32, out=z32, out16=z16, stats_out=stats)
    return z32, z16, stats


def pano_encoder_folded(x: Act, layers, B: int, L: int, key_mask, eps=1e-5) -> torch.Tensor:
    """The pre-norm panorama encoder layers (inference, 16-bit mode) with every LayerNorm folded into the contraction that
    follows it: x.f32 is the residual stream, x.b16 = norm1 of the first layer applied to it (chained in the embedding
    kernel).  Returns the raw fp32 stream for the final norm.  Reference: TransformerEncoderLayer.forward_pre,
    VLN-DUET/map_nav_src/models/transformer.py:170-182."""
    x32, h16, stats = x.f32, x.b16, None
    for i, pk in enumerate(layers):
        if i == 0:
            w, b = pk.qkv.get(True)
            qkv = ops.gemm(h16, w, b)
        else:
            qkv = gemm_act(Act(x32, h16, Pending(stats, pk.norm1, eps)), pk.qkv, True)
        ctx = ops.attention(qkv[:, 0:HIDDEN], qkv[:, HIDDEN:2 * HIDDEN], qkv[:, 2 * HIDDEN:3 * HIDDEN], B, L, L,
                            key_mask=key_mask, mask_mode=MASK_NEG_INF)
        x32, h16, stats = _dense_raw(ctx, pk.o, x32, True)
        f = gemm_act(Act(x32, h16, Pending(stats, pk.norm2, eps)), pk.w1, True, epilogue=EPI_GELU)
        x32, h16, stats = _dense_raw(f, pk.w2, x32, i + 1 < len(layers))
    return x32


class ClsHeadPack:
    """ClsPrediction / NextActionPrediction weights for one or several row groups:
    Linear -> ReLU -> LayerNorm -> Linear(768, 1)."""

    def __init__(self, heads, last_index=3):
        self.w0 = LinearPack([h.net[0].weight for h in heads], [h.net[0].bias for h in heads], n_groups=len(heads))
        self.ln = LNPack([h.net[2] for h in heads])
        self.w1 = StackPack([h.net[last_index].weight for h in heads])
        self.b1 = StackPack([h.net[last_index].bias for h in heads])
        self.has_dropout = last_index == 4


def cls_head(x: torch.Tensor, pk: ClsHeadPack, lowp: bool, ends=None, eps=1e-12) -> torch.Tensor:
    """x [rows, K] operand (bf16 or fp32) -> raw logit per row (fp32)."""
    if _Mode.train:
        h = ag.ActFn.apply(ag.linear(x, pk.w0, lowp, out_dtype=F32, ends=ends), EPI_RELU)
        y32, _ = ag.layer_norm(h, None, pk.ln, eps, False, ends)
        if pk.has_dropout and _Mode.p_head > 0:               # NextActionPrediction net.3 (H/models/vilmodel_cmt.py:953-963)
            y32 = ag.dropout(y32, _Mode.p_head)
        n = len(pk.w1.tensors)
        return ag.RowDotFn.apply(y32, pk.w1.get(), pk.b1.get(), ends, n, *pk.w1.tensors, *pk.b1.tensors)
    w, b = pk.w0.get(lowp)
    h = ops.gemm(x, w, b, epilogue=EPI_RELU, out_dtype=F32, group_row_end=ends)
    g, be = pk.ln.get()
    return ops.ln_dot(h, g, be, eps, pk.w1.get(), pk.b1.get(), group_row_end=ends)
