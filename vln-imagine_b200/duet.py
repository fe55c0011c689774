"""DUET-Imagine on libvlnimagine: drop-in for ``models.model.VLNBert`` / ``models.vilmodel.GlocalTextPathNavCMT``.

Same constructor (``VLNBert(args)``), same ``forward(mode, batch)`` modes and return types, same
parameter names as the reference (VLN-DUET/map_nav_src/models/model.py:12-48,
models/vilmodel.py:1022-1288), so the reference's unmodified agent (r2r/agent.py) can hold it as
``self.vln_bert``.  Every floating-point operation is a libvlnimagine kernel launch; torch is used
for device memory, streams, views and integer / boolean plumbing (mask casts, length -> mask).

Precision: ``model.precision = 'bf16'`` (default: bf16 tensor-core GEMM / attention operands, fp32
accumulation, fp32 residual stream, LayerNorm, softmax and heads) or ``'fp32'`` (check mode).
"""
from __future__ import annotations

import collections
import itertools
import struct
import os
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from . import autograd_ops as ag
from . import blocks, graphs, ops, params
from .blocks import Stream
from .config import duet_config
from .ops import F32, HIDDEN


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t if (t.dtype == F32 and t.is_contiguous()) else t.float().contiguous()


class _IdTable:
    """Viewpoint-id strings -> int32 ids.  Ids only need to agree between gmap_vpids and vp_cand_vpids of
    the same call; one growing table per model is the simplest way to guarantee that.  The agent hands ~1700
    strings per step at batch 64, so the hot loop is C-level end to end: the table maps a key to the 4 bytes of
    its id, one ``map`` + ``bytes.join`` over the chained rows builds the int32 buffer (converting a Python list
    of ints to numpy costs more than the dictionary look-ups)."""

    def __init__(self):
        self.ids = {}

    def encode(self, lists, width: int, pad: int) -> np.ndarray:
        rows = [row[:width] if len(row) > width else row for row in lists]
        lens = np.fromiter(map(len, rows), dtype=np.int64, count=len(rows))
        ids = self.ids
        try:
            buf = b''.join(map(ids.__getitem__, itertools.chain.from_iterable(rows)))
        except KeyError:
            for k in itertools.chain.from_iterable(rows):
                if k not in ids:
                    ids[k] = struct.pack('<i', len(ids))
            buf = b''.join(map(ids.__getitem__, itertools.chain.from_iterable(rows)))
        out = np.full((len(rows), width), pad, np.int32)
        if buf:
            out[np.arange(width)[None, :] < lens[:, None]] = np.frombuffer(buf, dtype='<i4')
        return out


class AlignRows:
    """Host-side flattening of the ragged alignment inputs (sub_instr_imag_flag, noun_phrase_segs) of
    AlignWithContrastiveLoss.forward (models/vilmodel.py:598-655) into index arrays:
      row r  <->  imagination (b, i) that is flagged 'True' and has >= 1 noun phrase;
      tok_offsets / tok_rows : tokens of all its noun-phrase spans (inclusive ends, duplicates kept);
      np_offsets / np_rows / np_episode : one entry per noun phrase of every flagged sub-instruction
      (the InfoNCE negatives, :716-741)."""

    def __init__(self, B, L, I, flags, noun_phrase_segs):
        slot, tok_off, tok_rows, ep = [], [0], [], []
        np_off, np_rows, np_ep = [0], [], []
        for b in range(B):
            for i, f in enumerate(flags[b]):
                if f != 'True':
                    continue
                spans = noun_phrase_segs[b][i]
                for s, e in spans:
                    if e >= s:
                        np_rows.extend(b * L + t for t in range(s, e + 1))
                        np_off.append(len(np_rows))
                        np_ep.append(b)
                if len(spans) == 0:
                    continue
                for s, e in spans:
                    if not (0 <= s and e < L):
                        raise ValueError('noun-phrase span [%d, %d] outside the instruction (L=%d)' % (s, e, L))
                    tok_rows.extend(b * L + t for t in range(s, e + 1))
                if i >= I:
                    raise ValueError('imagination slot %d >= %d' % (i, I))
                slot.append(b * I + i)
                tok_off.append(len(tok_rows))
                ep.append(b)
        self.R, self.n_negs = len(slot), len(np_ep)
        i32 = lambda x: torch.tensor(x, dtype=torch.int32)   # noqa: E731
        self.slot, self.tok_off, self.tok_rows, self.ep = i32(slot), i32(tok_off), i32(tok_rows), i32(ep)
        self.np_off, self.np_rows, self.np_ep = i32(np_off), i32(np_rows), i32(np_ep)
        self.unit = torch.arange(self.R + 1, dtype=torch.int32)

    def to(self, device):
        for k in ('slot', 'tok_off', 'tok_rows', 'ep', 'np_off', 'np_rows', 'np_ep', 'unit'):
            setattr(self, k, getattr(self, k).to(device, non_blocking=True))
        return self


def reverie_align_rows(B, L, I, txt_masks) -> AlignRows:
    """AlignRows of the REVERIE alignment modules (models/vilmodel.py:781-888): one imagination per instruction (slot 0), its
    target = the mean of ALL valid instruction tokens; the InfoNCE negatives = the instruction means of the other episodes."""
    valid = txt_masks.detach().to('cpu', torch.bool).numpy()
    r = AlignRows.__new__(AlignRows)
    tok_rows, tok_off = [], [0]
    for b in range(B):
        cols = np.flatnonzero(valid[b])
        if cols.size == 0:
            raise ValueError('episode %d has no valid instruction token' % b)
        tok_rows.extend((b * L + cols).tolist())
        tok_off.append(len(tok_rows))
    i32 = lambda x: torch.tensor(x, dtype=torch.int32)   # noqa: E731
    r.R, r.n_negs = B, B
    r.slot, r.tok_off, r.tok_rows, r.ep = i32([b * I for b in range(B)]), i32(tok_off), i32(tok_rows), i32(list(range(B)))
    r.np_off, r.np_rows, r.np_ep = i32(tok_off), i32(tok_rows), i32(list(range(B)))
    r.unit = torch.arange(B + 1, dtype=torch.int32)
    return r


_ALIGN_ROWS = collections.OrderedDict()


def _align_rows(B, L, I, flags, noun_phrase_segs, dev):
    """AlignRows of a batch, kept for the last few batches: an iteration that is replayed on the same episode batch
    (CUDA-graph capture of a fine-tuning step, benchmarks) must not rebuild and re-upload the index arrays.  The key holds
    the CONTENT of the ragged lists, not their identity."""
    key = (B, L, I, str(dev), tuple(tuple(f) for f in flags),
           tuple(tuple(tuple(tuple(sp) for sp in spans) for spans in segs) for segs in noun_phrase_segs))
    rows = _ALIGN_ROWS.get(key)
    if rows is None:
        rows = AlignRows(B, L, I, flags, noun_phrase_segs).to(dev)
        _ALIGN_ROWS[key] = rows
        while len(_ALIGN_ROWS) > 4:
            _ALIGN_ROWS.popitem(last=False)
    return rows


def align_forward(model, align_txt_embeds, align_imagine_embeds, flags, noun_phrase_segs, lowp: bool, rows: AlignRows = None):
    """Shared by DUET and HAMT.  Returns (loss 0-d tensor, imagine embeds with projected rows written back).  ``rows``: index
    arrays already built by the caller (REVERIE) instead of the sub-instruction annotation.  With autograd recording the
    projection MLP, the loss and the write-back of the projected rows (models/vilmodel.py:646) are differentiable; the text
    operands of the loss - the positive noun-phrase means and, for the contrastive forms, the noun-phrase means of the negatives,
    both built from ``align_txt_embeds`` - train when the text requires grad (fix_lang_inside_cosine_model off, :1256-1262)."""
    cfg = model.config
    B, L, _ = align_txt_embeds.shape
    I = align_imagine_embeds.shape[1]
    dev = align_txt_embeds.device
    rows = rows.to(dev) if rows is not None else _align_rows(B, L, I, flags, noun_phrase_segs, dev)
    txt = _f32c(align_txt_embeds).view(B * L, HIDDEN)
    img = _f32c(align_imagine_embeds).view(B * I, HIDDEN)
    if rows.R == 0:
        # the reference returns the python int 0 here (models/vilmodel.py:650-651); a 0-d tensor is a superset
        return torch.zeros((), dtype=F32, device=dev), img.clone().view(B, I, HIDDEN)
    pk = model._pk()['align']
    train = blocks.training()
    if train:
        if cfg.aux_loss_type not in ('cosine', 'contrastive-InfoNCE', 'constrastive-margin'):
            raise NotImplementedError('backward of aux_loss_type %r' % cfg.aux_loss_type)
        x = ag.GatherSlotsFn.apply(img, rows.unit, rows.slot, rows.R, lowp)
        if model.training:
            x = ag.dropout(x, 0.15)                           # MLPProjectionHead.dropout (models/vilmodel.py:578,585)
    else:
        x32, x16 = ops.gather_mean(img, rows.unit, rows.slot, rows.R, want16=lowp, want32=not lowp)
        x = x16 if lowp else x32
    for j, lp in enumerate(pk):
        last = j == len(pk) - 1
        x = blocks.linear(x, lp, lowp, out_dtype=F32 if (last or not lowp) else x.dtype, epilogue=ops.EPI_NONE if last else ops.EPI_RELU)
    tgt = blocks.segment_mean(txt, rows.tok_off, rows.tok_rows, rows.R)
    negs, neg_ep = None, None
    if rows.n_negs and cfg.aux_loss_type != 'cosine':         # AlignWithContrastiveLossWithNegativeSamples (:689-779)
        negs = blocks.segment_mean(txt, rows.np_off, rows.np_rows, rows.n_negs)
        neg_ep = rows.np_ep
    if cfg.aux_loss_type == 'cosine':
        loss = ag.CosineLossFn.apply(x, tgt, rows.R) if train else ops.cosine_loss(x, tgt, rows.R, dev)[0]
    elif cfg.aux_loss_type == 'contrastive-InfoNCE':
        args = (x, tgt, negs, rows.ep, neg_ep, float(cfg.infonce_temperature), rows.R, rows.n_negs)
        loss = ag.InfoNCELossFn.apply(*args) if train else ops.infonce_loss(*args, dev)[0]
    elif cfg.aux_loss_type == 'constrastive-margin':          # (sic) H/r2r/parser.py:117, H/models/vilmodel_cmt.py:825-856
        args = (x, tgt, negs, rows.ep, neg_ep, float(cfg.contrastive_margin_value), rows.R, rows.n_negs)
        loss = ag.MarginLossFn.apply(*args) if train else ops.margin_loss(*args, dev)[0]
    else:
        raise NotImplementedError('aux_loss_type %r' % cfg.aux_loss_type)
    out = ag.ScatterSlotsFn.apply(img, x, rows.slot, rows.unit) if train else ops.scatter_rows(x, rows.slot, img.clone())
    return loss, out.view(B, I, HIDDEN)


_ARANGE = {}


def _arange(n: int, dev) -> torch.Tensor:
    """0 .. n-1 on ``dev``, built once per length (one launch less per step; a constant, so it is safe inside captured graphs as
    long as it was created outside of one - the first call of every mode runs eagerly)"""
    key = (n, str(dev))
    t = _ARANGE.get(key)
    if t is None:
        t = torch.arange(n, device=dev)
        if not torch.cuda.is_current_stream_capturing():
            _ARANGE[key] = t
    return t


class GlocalTextPathNavCMT(nn.Module):
    """models/vilmodel.py:1022-1288 (R2R configuration: no object branch)."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        self.embeddings = params.BertEmbeddingsP(config)
        self.lang_encoder = params.LayerStack('layer', [params.BertLayerP() for _ in range(config.num_l_layers)])
        self.img_embeddings = params.DuetImageEmbeddingsP(config)
        self.local_encoder = params.LocalVPEncoderP(config)
        self.global_encoder = params.GlobalMapEncoderP(config)
        self.global_sap_head = params.ClsPredictionP()
        self.local_sap_head = params.ClsPredictionP()
        self.sap_fuse_linear = params.ClsPredictionP(input_size=2 * HIDDEN) if config.glocal_fuse else None
        if config.obj_feat_size > 0:                           # REVERIE object grounding (:1039-1040); inference only here
            self.og_head = params.ClsPredictionP()
        if config.imagine_enc_pano:
            if config.bypass_imag_encoder:
                self.imagine_embeddings = params.BypassImagineEmbeddingsP()
            else:
                raise NotImplementedError('bypass_imag_encoder=False (imagination encoder) is not on the released path')
            if config.use_cosine_aux_loss or config.no_loss_test:
                if config.aux_loss_type not in ('cosine', 'contrastive-InfoNCE'):
                    raise NotImplementedError('aux_loss_type %r' % config.aux_loss_type)
                self.contrastive_alignment_model = params.AlignModelP()
        params.bert_init_(self)
        if config.fix_lang_embedding or config.fix_local_branch:
            for m in (self.embeddings, self.lang_encoder):
                for p in m.parameters():
                    p.requires_grad = False
        if config.fix_pano_embedding or config.fix_local_branch:
            for p in self.img_embeddings.parameters():
                p.requires_grad = False
        if config.fix_local_branch:
            for m in (self.local_encoder, self.local_sap_head) + ((self.og_head,) if config.obj_feat_size > 0 else ()):
                for p in m.parameters():
                    p.requires_grad = False
        self.precision = os.environ.get('VLN_IMAGINE_PRECISION', 'bf16')
        # 16-bit operand format of inference calls in the 'bf16' (= 16-bit tensor-core) mode: 'auto' picks fp16 when the weights
        # prove it safe (blocks.operand_format), 'bf16' / 'f16' force one
        self.operand16 = os.environ.get('VLN_IMAGINE_OPERAND16', 'auto')
        self._fmt_cache = {}
        self._packs = None
        self._ids = _IdTable()
        self.context_cache = os.environ.get('VLN_IMAGINE_CONTEXT_CACHE', '1') != '0'
        self._ctx_slots = {}
        self.context_hits = self.context_misses = 0

    # -- derived weights ------------------------------------------------------------------------
    def _pk(self):
        if self._packs is None:
            pk = {}
            pk['lang'] = [blocks.SelfFFNPack([l.attention], [l.intermediate], [l.output]) for l in self.lang_encoder.layer]
            ie = self.img_embeddings
            pk['img_linear'] = blocks.LinearPack([ie.img_linear.weight], [ie.img_linear.bias])
            pk['pano'] = [blocks.PanoLayerPack(l) for l in ie.pano_encoder.layers]
            pk['pano_norm'] = blocks.LNPack([ie.pano_encoder.norm])
            gl, ll = self.global_encoder.encoder.x_layers, self.local_encoder.encoder.x_layers
            pk['x_cross'] = [blocks.CrossPack([g.visual_attention, l.visual_attention]) for g, l in zip(gl, ll)]
            pk['x_self'] = [blocks.SelfFFNPack([g.visn_self_att, l.visn_self_att], [g.visn_inter, l.visn_inter],
                                               [g.visn_output, l.visn_output]) for g, l in zip(gl, ll)]
            pk['sap'] = blocks.ClsHeadPack([self.global_sap_head, self.local_sap_head])
            if self.config.obj_feat_size > 0:
                pk['og'] = blocks.ClsHeadPack([self.og_head])
                if ie.obj_linear is not None:
                    pk['obj_linear'] = blocks.LinearPack([ie.obj_linear.weight], [ie.obj_linear.bias])
            if self.global_encoder.sprel_linear is not None:
                sl = self.global_encoder.sprel_linear
                pk['sprel'] = blocks.StackPack([sl.weight, sl.bias])         # device {w, b} of the GASA bias
            if self.sap_fuse_linear is not None:
                pk['fuse'] = blocks.ClsHeadPack([self.sap_fuse_linear])
            if hasattr(self, 'contrastive_alignment_model'):
                ip = self.contrastive_alignment_model.image_proj
                pk['align'] = [blocks.LinearPack([ip.fc1.weight]), blocks.LinearPack([ip.fc2.weight]),
                               blocks.LinearPack([ip.fc3.weight])]
            self._packs = pk
        return self._packs

    def _apply(self, fn, *a, **k):          # .cuda() / .to(): derived tensors are rebuilt lazily
        self._packs = None
        self._ctx_slots = {}
        return super()._apply(fn, *a, **k)

    @property
    def lowp(self):
        if self.precision not in ('bf16', 'fp32'):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        return self.precision == 'bf16'

    def _guard(self, t: torch.Tensor):
        ops.ensure_init(t)            # raises on CPU tensors: there is no fallback path

    def _recording(self, *inputs) -> bool:
        """True when this call must record autograd nodes (fine-tuning): gradients are enabled and a parameter
        or an input asks for one."""
        if not torch.is_grad_enabled():
            return False
        return any(torch.is_tensor(t) and t.requires_grad for t in inputs) or any(p.requires_grad for p in self.parameters())

    def _drop(self):
        """(hidden, attention-probability) dropout of this call: the config's probabilities in train() mode, else none.
        Dropout exists on the autograd-recording path only (as in the reference, eval() / no_grad inference has none)."""
        if not self.training:
            return (0.0, 0.0)
        ph, pa = float(self.config.hidden_dropout_prob), float(self.config.attention_probs_dropout_prob)
        if (ph > 0 or pa > 0) and not self.lowp:
            raise NotImplementedError('dropout is implemented for the bf16 kernels only: use eval() or p = 0 in the fp32 check mode')
        if (ph > 0 or pa > 0) and not torch.is_grad_enabled():
            raise NotImplementedError('train() mode with dropout under torch.no_grad() is not supported: call .eval() for inference')
        return (ph, pa)

    # -- modes ------------------------------------------------------------------------------------
    def forward_text(self, txt_ids, txt_masks):
        """'language': BertEmbeddings (:49-78) + 9 post-LN layers (:414-434); entry :1075-1079."""
        self._guard(txt_ids)
        lowp = self.lowp
        B, L = txt_ids.shape
        e = self.embeddings
        with blocks.grad_mode(self._recording() and not self.config.fix_lang_embedding, self._drop()):
            x = blocks.embed(B * L, txt_ids.device, idx=txt_ids.long().contiguous().view(-1), table=e.word_embeddings.weight,
                             pos_table=e.position_embeddings.weight, pos_period=L,
                             const_rows=(e.token_type_embeddings.weight[0],), out_ln=e.LayerNorm, lowp=lowp, dropout=True)
            s = [Stream(0, B, L, blocks.mask_u8(txt_masks))]
            for pk in self._pk()['lang']:
                x = blocks.self_attn_ffn(x, pk, s, None, lowp, defer=True)
            x = blocks.materialize(x, lowp, want16=False)
        out = x.f32.view(B, L, HIDDEN)
        if self.config.fix_lang_embedding:
            out = out.detach()
        return out

    def forward_imagination(self, imagine_feats, imagine_masks=None):
        """'imagine' (bypass encoder): features + type embedding 0.  :562-573, :1081-1085."""
        self._guard(imagine_feats)
        B, I, _ = imagine_feats.shape
        with blocks.grad_mode(self._recording(imagine_feats), self._drop()):
            y = blocks.embed(B * I, imagine_feats.device, a=_f32c(imagine_feats).view(B * I, HIDDEN),
                             const_rows=(self.imagine_embeddings.type_embedding.weight[0],))
        return y.f32.view(B, I, HIDDEN)

    def forward_panorama_per_step(self, view_img_fts, obj_img_fts, loc_fts, nav_types, view_lens, obj_lens):
        """'panorama'.  :1087-1131 + transformer.py:71-89,170-182."""
        if obj_img_fts is not None:
            return self._panorama_with_objects(view_img_fts, obj_img_fts, loc_fts, nav_types, view_lens, obj_lens)
        self._guard(view_img_fts)
        lowp = self.lowp
        B, V, Fd = view_img_fts.shape
        dev = view_img_fts.device
        pk = self._pk()
        ie = self.img_embeddings
        v32 = _f32c(view_img_fts).view(B * V, Fd)
        pano_masks = _arange(V, dev)[None, :] < view_lens.to(dev)[:, None]                  # ops.py:36-44
        km = blocks.mask_u8(pano_masks)
        with blocks.grad_mode(self._recording(view_img_fts) and not self.config.fix_pano_embedding, self._drop()):
            a = blocks.linear(blocks.operand(v32, lowp), pk['img_linear'], lowp, out_dtype=F32)
            folded = lowp and not blocks.training() and len(pk['pano']) > 0
            x = blocks.embed(B * V, dev, a=a, a_ln=ie.img_layer_norm, feat=_f32c(loc_fts).view(B * V, -1),
                             feat_lin=ie.loc_linear, feat_ln=ie.loc_layer_norm,
                             idx=nav_types.long().contiguous().view(-1), table=ie.nav_type_embedding.weight,
                             const_rows=(self.embeddings.token_type_embeddings.weight[1],), out_ln=ie.layer_norm,
                             dropout=True, chain_ln=ie.pano_encoder.layers[0].norm1 if folded else None)
            if folded:
                x32 = blocks.pano_encoder_folded(x, pk['pano'], B, V, km)
            else:
                x32 = x.f32
                for lp in pk['pano']:
                    x32 = blocks.pano_layer(x32, lp, B, V, km, lowp)
            y32 = blocks.layer_norm(x32, None, pk['pano_norm'], 1e-12, False).f32
        out = y32.view(B, V, HIDDEN)
        if self.config.fix_pano_embedding:
            out = out.detach()
        return out, pano_masks

    def _panorama_with_objects(self, view_img_fts, obj_img_fts, loc_fts, nav_types, view_lens, obj_lens):
        """'panorama' with the REVERIE object boxes (:1096-1114): per episode the LayerNorm-ed object embeddings follow the
        LayerNorm-ed view embeddings, zero padded to the longest; everything after that is the R2R path over P = max(view_len
        + obj_len) tokens.  The ragged concatenation is one row gather over [views ; objects ; a zero row] (adjoint in training:
        a scatter-add)."""
        self._guard(view_img_fts)
        lowp, pk, ie = self.lowp, self._pk(), self.img_embeddings
        B, V, _ = view_img_fts.shape
        O = obj_img_fts.shape[1]
        dev = view_img_fts.device
        vl = [int(x) for x in view_lens.tolist()]              # host lengths: the reference loops over them as well (:1106-1113)
        ol = [int(x) for x in obj_lens.tolist()]
        P = max(a + b for a, b in zip(vl, ol))
        if loc_fts.shape[1] != P or nav_types.shape[1] != P:
            raise ValueError('loc_fts / nav_types must cover max(view_len + obj_len) = %d tokens' % P)
        idx = np.full((B, P), B * V + B * O, np.int64)         # row B * V + B * O: the appended zero row
        for i in range(B):
            idx[i, :vl[i]] = i * V + np.arange(vl[i])
            idx[i, vl[i]:vl[i] + ol[i]] = B * V + i * O + np.arange(ol[i])
        pano_lens = (view_lens + obj_lens).to(dev)
        pano_masks = torch.arange(P, device=dev)[None, :] < pano_lens[:, None]
        km = blocks.mask_u8(pano_masks)
        recording = self._recording(view_img_fts, obj_img_fts) and not self.config.fix_pano_embedding
        with blocks.grad_mode(recording, self._drop()):
            v32 = _f32c(view_img_fts).view(B * V, -1)
            o32 = _f32c(obj_img_fts).view(B * O, -1)
            nv = blocks.layer_norm(blocks.linear(blocks.operand(v32, lowp), pk['img_linear'], lowp, out_dtype=F32), None,
                                   blocks.LNPack([ie.img_layer_norm]), 1e-12, False).f32
            if ie.obj_linear is not None:                      # obj_feat_size != image_feat_size (:464-468)
                olin, oln = pk['obj_linear'], ie.obj_layer_norm
            else:
                olin, oln = pk['img_linear'], ie.img_layer_norm
            no = blocks.layer_norm(blocks.linear(blocks.operand(o32, lowp), olin, lowp, out_dtype=F32), None, blocks.LNPack([oln]),
                                   1e-12, False).f32
            src = torch.cat([nv, no, torch.zeros((1, HIDDEN), dtype=F32, device=dev)], 0)
            a = blocks.gather_rows(src, idx.reshape(-1), B * P)
            x32 = blocks.embed(B * P, dev, a=a, feat=_f32c(loc_fts).view(B * P, -1), feat_lin=ie.loc_linear, feat_ln=ie.loc_layer_norm,
                               idx=nav_types.long().contiguous().view(-1), table=ie.nav_type_embedding.weight,
                               const_rows=(self.embeddings.token_type_embeddings.weight[1],), out_ln=ie.layer_norm, dropout=True).f32
            for lp in pk['pano']:
                x32 = blocks.pano_layer(x32, lp, B, P, km, lowp)
            y32 = blocks.layer_norm(x32, None, pk['pano_norm'], 1e-12, False).f32
        out = y32.view(B, P, HIDDEN)
        return (out if recording else out.detach()), pano_masks

    def forward_navigation_per_step(self, txt_embeds, txt_masks, gmap_img_embeds, gmap_step_ids, gmap_pos_fts,
                                    gmap_masks, gmap_pair_dists, gmap_visited_masks, gmap_vpids,
                                    vp_img_embeds, vp_pos_fts, vp_masks, vp_nav_masks, vp_obj_masks, vp_cand_vpids,
                                    imagine_embeds=None, imagine_masks=None, ctx_kv=None, defer_fuse=False):
        """'navigation'.  :1133-1235.  With autograd recording (fine-tuning, BASELINE.json cfg-4) every block records its
        node.  ``ctx_kv`` (internal, inference): context projections already looked up by the caller (VLNBert's graph path);
        txt_embeds / imagine_embeds are then not read.  ``defer_fuse`` (internal, inference): stop before the global / local
        fusion (:1198-1217) and return its operands under '_fuse' for ``fuse_logits``."""
        if vp_obj_masks is not None and not hasattr(self, 'og_head'):
            raise ValueError('vp_obj_masks given but the model has no object-grounding head (obj_feat_size = 0)')
        self._guard(gmap_img_embeds)
        lowp, pk = self.lowp, self._pk()
        dev = gmap_img_embeds.device
        B, L = txt_masks.shape
        G, P = gmap_img_embeds.shape[1], vp_img_embeds.shape[1]
        recording = ctx_kv is None and self._recording(txt_embeds, gmap_img_embeds, vp_img_embeds, imagine_embeds)
        with blocks.grad_mode(recording, self._drop() if recording else (0.0, 0.0)):
            x, row0, ends = self._branch_inputs(_f32c(gmap_img_embeds).view(B * G, HIDDEN), gmap_pos_fts, gmap_step_ids,
                                                _f32c(vp_img_embeds).view(B * P, HIDDEN), vp_pos_fts, B, G, P)
            r_g, r_l = row0
            # context = [txt ; imagine] (:1157-1158).  Inference: its K / V projections for the 4 layers are kept per episode
            # (the context never changes inside one, use_lang2visn_attn is off); training projects it in every layer
            ctx = kvs = None
            if recording:
                ctx32 = _f32c(txt_embeds)
                if self._with_imagine():
                    if imagine_embeds is None:
                        raise ValueError('navigation needs imagine_embeds and imagine_masks when imagine_enc_pano is set')
                    ctx32 = torch.cat([ctx32, _f32c(imagine_embeds)], 1)
                ctx = blocks.operand(ctx32.view(-1, HIDDEN), lowp)
            else:
                kvs = ctx_kv if ctx_kv is not None else self.context_kv(txt_embeds, imagine_embeds)
            ctx_mask, C = self.context_mask(txt_masks, imagine_masks)
            streams = self._branch_streams(B, G, P, row0, gmap_masks, vp_masks, gmap_pair_dists)
            x = self._cross_layers(x, streams, ends, C, ctx_mask, kvs=kvs, ctx=ctx)
            gmap_out = x.f32[r_g:r_g + B * G].view(B, G, HIDDEN)
            vp_out = x.f32[r_l:r_l + B * P].view(B, P, HIDDEN)
            # heads (:1182-1196) and global/local fusion (:1198-1217)
            raw, fuse_raw = self._sap_heads(x, pk['sap'], pk.get('fuse'), B, G, P, row0, ends)
            if defer_fuse:
                return {'gmap_embeds': gmap_out, 'vp_embeds': vp_out, '_g_raw': raw[r_g:], '_l_raw': raw[r_l:], '_fuse_raw': fuse_raw,
                        '_gmap_masks': blocks.mask_u8(gmap_masks), '_visited': blocks.mask_u8(gmap_visited_masks),
                        '_nav_masks': blocks.mask_u8(vp_nav_masks)}
            gmap_ids, cand_ids = self.intern_vpids(gmap_vpids, vp_cand_vpids, G, P, dev)
            gl, ll, fl = self._fuse_step(raw, fuse_raw, gmap_masks, gmap_visited_masks, vp_nav_masks, gmap_ids, cand_ids,
                                         B, G, P, row0)
            obj_logits = None
            if vp_obj_masks is not None:                       # object grounding logits (:1220-1225): -inf outside the object tokens
                obj_logits = blocks.mask_logits(blocks.cls_head(x.operand(lowp)[r_l:r_l + B * P], pk['og'], lowp), vp_obj_masks)
        return {'gmap_embeds': gmap_out, 'vp_embeds': vp_out, 'global_logits': gl, 'local_logits': ll,
                'fused_logits': fl, 'obj_logits': obj_logits}

    # -- pieces of the navigation step that pre-training (pretrain.py) runs as well --------------------------------------
    def _branch_inputs(self, gmap_img, gmap_pos_fts, gmap_step_ids, vp_img, vp_pos_fts, B, G, P):
        """input embeddings of both branches in one row-stacked activation (:1141-1152) -> (Act, row0, ends)"""
        ge, le = self.global_encoder, self.local_encoder
        row0, ends, R = blocks.stack_layout([B * G, B * P])
        x = blocks.embed_streams([
            dict(rows=B * G, a=gmap_img, feat=_f32c(gmap_pos_fts).view(B * G, -1), feat_lin=ge.gmap_pos_embeddings[0],
                 feat_ln=ge.gmap_pos_embeddings[1], idx=gmap_step_ids.long().contiguous().view(-1), table=ge.gmap_step_embeddings.weight),
            dict(rows=B * P, a=vp_img, feat=_f32c(vp_pos_fts).view(B * P, -1), feat_lin=le.vp_pos_embeddings[0],
                 feat_ln=le.vp_pos_embeddings[1])], row0, R, gmap_img.device, self.lowp)
        return x, row0, ends

    def _branch_streams(self, B, G, P, row0, gmap_masks, vp_masks, gmap_pair_dists):
        """the global (map) and local (panorama) streams; the global one carries the GASA bias (:1145-1149), applied inside the
        attention kernel"""
        sl = self.global_encoder.sprel_linear
        dist = affine = aparams = None
        if sl is not None:
            dist, affine, aparams = _f32c(gmap_pair_dists), self._pk()['sprel'].get(), (sl.weight, sl.bias)
        return [Stream(row0[0], B, G, blocks.mask_u8(gmap_masks), 0, dist, affine, aparams),
                Stream(row0[1], B, P, blocks.mask_u8(vp_masks), 1)]

    def _cross_layers(self, x, streams, ends, C, ctx_mask, kvs=None, ctx=None):
        """the graph-aware cross-modal layers, both branches per launch (:384-399, :444-453).  The context's K_g | V_g | K_l | V_l
        [B*C, 4*768] per layer: ``kvs`` when given, else projected from the context operand ``ctx`` in each layer."""
        lowp, pk = self.lowp, self._pk()
        for i, (cp, sp) in enumerate(zip(pk['x_cross'], pk['x_self'])):
            kv = kvs[i] if kvs is not None else blocks.linear(ctx, cp.kv, lowp)
            x = blocks.cross_attn(x, [(kv, 0, C, ctx_mask), (kv, 2 * HIDDEN, C, ctx_mask)], cp, streams, ends, lowp, defer=True)
            x = blocks.self_attn_ffn(x, sp, streams, ends, lowp, defer=True)
        return blocks.materialize(x, lowp, ends)

    def _sap_heads(self, x, sap, fuse, B, G, P, row0, ends):
        """(raw action logit of every token of both branches, raw fused logit of the two [stop] tokens or None) (:1182-1217)"""
        lowp = self.lowp
        r_g, r_l = row0
        fuse_raw = None
        if fuse is not None:
            if blocks.training():
                cat = blocks.operand(torch.cat([x.f32[r_g:r_g + B * G].view(B, G, HIDDEN)[:, 0],
                                                x.f32[r_l:r_l + B * P].view(B, P, HIDDEN)[:, 0]], 1), lowp)
            else:
                cat = torch.empty((B, 2 * HIDDEN), dtype=ops.h16() if lowp else F32, device=x.f32.device)
                c32, c16 = (None, cat) if lowp else (cat, None)
                ops.copy_rows(x.f32[r_g:], G * HIDDEN, HIDDEN, B, 1, c32, c16, 2 * HIDDEN, HIDDEN)
                ops.copy_rows(x.f32[r_l:], P * HIDDEN, HIDDEN, B, 1, c32[:, HIDDEN:] if c32 is not None else None,
                              c16[:, HIDDEN:] if c16 is not None else None, 2 * HIDDEN, HIDDEN)
            fuse_raw = blocks.cls_head(cat, fuse, lowp)
        return blocks.cls_head(x.operand(lowp), sap, lowp, ends), fuse_raw

    def _fuse_step(self, raw, fuse_raw, gmap_masks, visited, nav, gmap_ids, cand_ids, B, G, P, row0):
        """global / local / fused action logits from the raw head outputs (:1198-1217)"""
        args = (raw[row0[0]:row0[0] + B * G], raw[row0[1]:row0[1] + B * P], fuse_raw, blocks.mask_u8(gmap_masks),
                blocks.mask_u8(visited), blocks.mask_u8(nav), gmap_ids, cand_ids, B, G, P)
        return ag.FuseLogitsFn.apply(*args) if blocks.training() else ops.duet_fuse_logits(*args)

    def fuse_logits(self, pre: dict, gmap_vpids, vp_cand_vpids, G: int, P: int) -> dict:
        """Second half of a ``defer_fuse`` navigation call: intern the viewpoint ids (host work that then overlaps the
        encoder kernels already queued), upload them and launch the fusion kernel (:1198-1217)."""
        dev = pre['_g_raw'].device
        gmap_ids, cand_ids = self.intern_vpids(gmap_vpids, vp_cand_vpids, G, P, dev)
        B = pre['_gmap_masks'].shape[0]
        gl, ll, fl = ops.duet_fuse_logits(pre['_g_raw'], pre['_l_raw'], pre['_fuse_raw'], pre['_gmap_masks'], pre['_visited'],
                                          pre['_nav_masks'], gmap_ids, cand_ids, B, G, P)
        return {'gmap_embeds': pre['gmap_embeds'], 'vp_embeds': pre['vp_embeds'], 'global_logits': gl, 'local_logits': ll,
                'fused_logits': fl, 'obj_logits': None}

    # -- per-episode context cache ----------------------------------------------------------------------------
    def _with_imagine(self):
        cfg = self.config
        return bool(cfg.imagine_enc_pano and cfg.concat_imagine_with == 'language')

    def context_mask(self, txt_masks, imagine_masks):
        """key-padding mask and length of the [txt ; imagine] context (:1157-1158)"""
        if self._with_imagine():
            if imagine_masks is None:
                raise ValueError('navigation needs imagine_embeds and imagine_masks when imagine_enc_pano is set')
            return (blocks.mask_u8(torch.cat([txt_masks.bool(), imagine_masks.bool()], 1)),
                    txt_masks.shape[1] + imagine_masks.shape[1])
        return blocks.mask_u8(txt_masks), txt_masks.shape[1]

    def context_kv(self, txt_embeds, imagine_embeds):
        """[txt ; imagine] context (:1157-1158) projected to K | V for every cross-modal layer of both branches:
        one [B*C, 4*768] tensor (K_g | V_g | K_l | V_l) per layer.

        The reference recomputes these 8 projections per layer identically at every navigation step
        (use_lang2visn_attn=False, vlnbert_init.py:57: the context is never updated).  Here they are computed when
        the context changes and reused while the caller keeps passing the SAME txt_embeds / imagine_embeds tensor
        objects at the same version (what the agents do for the length of an episode, r2r/agent.py:409,449 -> :485-500).
        The projections live in buffers owned by the cache (one set per shape / precision), so CUDA graphs that
        captured their addresses stay valid across episodes.  ``context_cache = False`` restores per-step
        recomputation."""
        lowp, pk = self.lowp, self._pk()
        with_img = self._with_imagine()
        if with_img and imagine_embeds is None:
            raise ValueError('navigation needs imagine_embeds and imagine_masks when imagine_enc_pano is set')
        B, L, _ = txt_embeds.shape
        I = imagine_embeds.shape[1] if with_img else 0
        C = L + I
        dev = self.embeddings.LayerNorm.weight.device
        slot_key = (B, L, I, lowp, ops.h16())
        slot = self._ctx_slots.get(slot_key)
        wtok = tuple(cp.kv.get_token() for cp in pk['x_cross'])
        ident = (id(txt_embeds), txt_embeds._version, txt_embeds.data_ptr(),
                 id(imagine_embeds) if with_img else 0, imagine_embeds._version if with_img else 0,
                 imagine_embeds.data_ptr() if with_img else 0, wtok)
        if slot is not None and self.context_cache and slot['ident'] == ident:
            self.context_hits += 1
            return slot['kv']
        if slot is None:
            slot = {'ctx': torch.empty((B * C, HIDDEN), dtype=ops.h16() if lowp else F32, device=dev),
                    'kv': [torch.empty((B * C, 4 * HIDDEN), dtype=ops.h16() if lowp else F32, device=dev) for _ in pk['x_cross']]}
            self._ctx_slots[slot_key] = slot
        ctx = slot['ctx']
        c32, c16 = (None, ctx) if lowp else (ctx, None)
        txt = _f32c(txt_embeds.to(dev, non_blocking=True))
        if with_img:
            img = _f32c(imagine_embeds.to(dev, non_blocking=True))
            ops.copy_rows(txt, L * HIDDEN, HIDDEN, B, L, c32, c16, C * HIDDEN, HIDDEN)
            ops.copy_rows(img, I * HIDDEN, HIDDEN, B, I, c32[L:] if c32 is not None else None,
                          c16[L:] if c16 is not None else None, C * HIDDEN, HIDDEN)
        elif lowp:
            ops.cast_h16(txt.view(B * L, HIDDEN), ctx)
        else:
            ctx.copy_(txt.view(B * L, HIDDEN))
        for cp, kv in zip(pk['x_cross'], slot['kv']):
            w, b = cp.kv.get(lowp)
            ops.gemm(ctx, w, b, out=kv)                      # [B*C, 4*768] = K_g | V_g | K_l | V_l
        # the cache keeps the source tensors alive, so their ids / addresses cannot be recycled while it is valid
        slot['ident'], slot['refs'] = ident, (txt_embeds, imagine_embeds)
        self.context_misses += 1
        return slot['kv']

    def drop_context(self):
        """forget the cached context projections (new episode with recycled tensors, or to bound memory)"""
        for slot in self._ctx_slots.values():
            slot['ident'], slot['refs'] = None, None

    def intern_vpids(self, gmap_vpids, vp_cand_vpids, G, P, dev):
        """Viewpoint-id strings -> int32 tensors on ``dev`` (gmap padding -1, candidate padding -2).  Callers that
        already hold interned ids (a CUDA-graph replay loop, bench.py) may pass the two tensors instead of the
        lists; they are used as they are."""
        def fit(ids, n, pad):                                  # interned rows narrower than a bucketed call: pad with the padding id
            if ids.shape[1] >= n:
                return ids
            out = ids.new_full((ids.shape[0], n), pad)
            out[:, :ids.shape[1]] = ids
            return out
        if torch.is_tensor(gmap_vpids) and torch.is_tensor(vp_cand_vpids):
            return fit(gmap_vpids, G, -1), fit(vp_cand_vpids, P, -2)
        gi, ci = getattr(gmap_vpids, 'ids', None), getattr(vp_cand_vpids, 'ids', None)
        if torch.is_tensor(gi) and torch.is_tensor(ci):       # rows built by graph_map.DeviceGraphMaps: already interned
            return fit(gi, G, -1), fit(ci, P, -2)
        gmap_ids = torch.from_numpy(self._ids.encode(gmap_vpids, G, -1))
        cand_ids = torch.from_numpy(self._ids.encode(vp_cand_vpids, P, -2))
        if len(self._ids.ids) > (1 << 20):
            self._ids = _IdTable()
        if dev is not None and torch.device(dev).type == 'cuda':
            gmap_ids, cand_ids = gmap_ids.to(dev, non_blocking=True), cand_ids.to(dev, non_blocking=True)
        return gmap_ids, cand_ids

    def forward_align(self, batch):
        """'align_with_contrastive_loss'.  :1246-1262 -> AlignWithContrastiveLoss(.WithNegativeSamples) :598-779."""
        self._guard(batch['align_txt_embeds'])
        txt = batch['align_txt_embeds']
        if self.config.fix_lang_inside_cosine_model:
            txt = txt.detach()
        with blocks.grad_mode(self._recording(txt, batch['align_imagine_embeds']), self._drop()):
            if self.config.dataset == 'reverie':               # :781-888: no sub-instruction annotation, one imagination
                B, L, _ = txt.shape
                rows = reverie_align_rows(B, L, batch['align_imagine_embeds'].shape[1], batch['txt_masks'])
                return align_forward(self, txt, batch['align_imagine_embeds'], None, None, self.lowp, rows=rows)
            return align_forward(self, txt, batch['align_imagine_embeds'], batch['sub_instr_imag_flag'],
                                 batch['noun_phrase_segs'], self.lowp)

    def h16_format(self):
        """16-bit operand format of this call (blocks.operand_format)"""
        return blocks.operand_format(self, self._fmt_cache, self.operand16)

    def forward(self, mode, batch, **kwargs):
        with ops.half_format(self.h16_format()):
            return self._forward(mode, batch, **kwargs)

    def _forward(self, mode, batch, **kwargs):
        """Mode dispatch, :1237-1288."""
        if mode == 'language':
            return self.forward_text(batch['txt_ids'], batch['txt_masks'])
        if mode == 'imagine':
            assert self.config.imagine_enc_pano
            return self.forward_imagination(batch['imagine_feats'], batch['imagine_masks'])
        if mode == 'align_with_contrastive_loss':
            assert self.config.imagine_enc_pano
            return self.forward_align(batch)
        if mode == 'panorama':
            return self.forward_panorama_per_step(batch['view_img_fts'], batch['obj_img_fts'], batch['loc_fts'],
                                                  batch['nav_types'], batch['view_lens'], batch['obj_lens'])
        if mode == 'navigation':
            kw = {}
            if self.config.imagine_enc_pano:
                kw = dict(imagine_embeds=batch['imagine_embeds'], imagine_masks=batch['imagine_masks'])
            return self.forward_navigation_per_step(
                batch['txt_embeds'], batch['txt_masks'], batch['gmap_img_embeds'], batch['gmap_step_ids'],
                batch['gmap_pos_fts'], batch['gmap_masks'], batch['gmap_pair_dists'], batch['gmap_visited_masks'],
                batch['gmap_vpids'], batch['vp_img_embeds'], batch['vp_pos_fts'], batch['vp_masks'],
                batch['vp_nav_masks'], batch['vp_obj_masks'], batch['vp_cand_vpids'], **kw)
        raise NotImplementedError('wrong mode: %s' % mode)


class VLNBert(nn.Module):
    """models/model.py:12-48: mode dispatch + environment (feature) dropout on the panorama features.

    Inference calls (eval mode, autograd off) of the two per-step modes are replayed from CUDA graphs
    (graphs.GraphedCall); set ``use_cuda_graphs = False`` for plain eager launches.  Inputs may live on the host
    (pinned) or on the device."""

    NAV_TENSORS = ('txt_masks', 'gmap_img_embeds', 'gmap_step_ids', 'gmap_pos_fts', 'gmap_masks',
                   'gmap_pair_dists', 'gmap_visited_masks', 'vp_img_embeds', 'vp_pos_fts', 'vp_masks', 'vp_nav_masks',
                   'imagine_masks')

    def __init__(self, args):
        super().__init__()
        self.args = args
        self.vln_bert = GlocalTextPathNavCMT(duet_config(args))
        ckpt = getattr(args, 'bert_ckpt_file', None)
        if ckpt is not None:                                   # models/vlnbert_init.py:18-28
            sd = {}
            for k, v in torch.load(ckpt, map_location='cpu').items():
                k = k[7:] if k.startswith('module') else k
                sd[k[5:] if k.startswith('bert.') else k] = v
            self.vln_bert.load_state_dict(sd, strict=False)
        self.drop_env = nn.Dropout(p=getattr(args, 'feat_dropout', 0.0))
        self.use_cuda_graphs = os.environ.get('VLN_IMAGINE_CUDA_GRAPHS', '1') != '0'
        self._wt_cache = {}
        self._g_pano = graphs.GraphedCall(self._pano_fn)
        self._g_nav = graphs.GraphedCall(self._nav_fn)
        self._buckets = graphs.ShapeBuckets()

    def _apply(self, fn, *a, **k):
        self._wt_cache = {}
        self._g_pano.clear()
        self._g_nav.clear()
        return super()._apply(fn, *a, **k)

    # pure launch sequences over dicts of device tensors (what the graphs capture)
    def _pano_fn(self, t):
        e, m = self.vln_bert.forward_panorama_per_step(t['view_img_fts'], None, t['loc_fts'], t['nav_types'], t['view_lens'], None)
        return {'pano_embeds': e, 'pano_masks': m}

    def _nav_fn(self, t):
        kv = [t['ctx_kv%d' % i] for i in range(len(self.vln_bert.global_encoder.encoder.x_layers))]
        return self.vln_bert.forward_navigation_per_step(
            None, t['txt_masks'], t['gmap_img_embeds'], t['gmap_step_ids'], t['gmap_pos_fts'], t['gmap_masks'],
            t['gmap_pair_dists'], t['gmap_visited_masks'], None, t['vp_img_embeds'], t['vp_pos_fts'], t['vp_masks'],
            t['vp_nav_masks'], None, None, imagine_embeds=None, imagine_masks=t.get('imagine_masks'), ctx_kv=kv, defer_fuse=True)

    def _graphable(self):
        return self.use_cuda_graphs and not self.training and not torch.is_grad_enabled()

    def forward(self, mode, batch):
        with ops.half_format(self.vln_bert.h16_format()):
            return self._forward(mode, batch)

    def _forward(self, mode, batch):
        batch = collections.defaultdict(lambda: None, batch)
        m = self.vln_bert
        if mode == 'panorama':
            if self.training and self.drop_env.p > 0:                      # models/model.py:27: nn.Dropout on the view features
                batch = dict(batch)
                feats = batch['view_img_fts']
                feats = feats if feats.is_cuda else feats.to(m.embeddings.LayerNorm.weight.device, non_blocking=True)
                ops.ensure_init(feats)
                batch['view_img_fts'] = ag.dropout(feats.float(), float(self.drop_env.p))
                batch = collections.defaultdict(lambda: None, batch)
            if self._graphable() and batch['obj_img_fts'] is None:
                dev = m.embeddings.LayerNorm.weight.device
                tok = graphs.weights_token(m, self._wt_cache)
                out = self._g_pano({k: batch[k] for k in ('view_img_fts', 'loc_fts', 'nav_types', 'view_lens')}, dev,
                                   extra_key=(m.precision, ops.h16()), weights_token=tok)
                return out['pano_embeds'], out['pano_masks']
            return m(mode, batch)
        if mode == 'navigation':
            if self._graphable() and batch['vp_obj_masks'] is None:
                dev = m.embeddings.LayerNorm.weight.device
                tok = graphs.weights_token(m, self._wt_cache)
                t = {k: batch[k] for k in self.NAV_TENSORS if batch[k] is not None}
                G, P = batch['gmap_img_embeds'].shape[1], batch['vp_img_embeds'].shape[1]
                Gb, Pb = G, P
                if self._buckets.active((G, P)):
                    # a rollout's (G, P) changes every step: pad to multiples of 8 so that a handful of captured graphs serves it
                    # (graphs.ShapeBuckets); the padding is masked like the reference's own batch padding and sliced off below
                    Gb, Pb = self._buckets.up(G), self._buckets.up(P)
                    gdims = {'gmap_img_embeds': {1: Gb}, 'gmap_step_ids': {1: Gb}, 'gmap_pos_fts': {1: Gb}, 'gmap_masks': {1: Gb},
                             'gmap_pair_dists': {1: Gb, 2: Gb}, 'gmap_visited_masks': {1: Gb}, 'vp_img_embeds': {1: Pb},
                             'vp_pos_fts': {1: Pb}, 'vp_masks': {1: Pb}, 'vp_nav_masks': {1: Pb}}
                    t = {k: (graphs.pad_to(v, gdims[k], dev) if k in gdims else v) for k, v in t.items()}
                cfg = m.config
                # context projections: looked up (or recomputed, eagerly) outside the graph, which only reads them
                kv = m.context_kv(batch['txt_embeds'], batch['imagine_embeds'])
                # The graph stops before the global / local fusion: the ~1700 viewpoint-id strings of a batch are
                # interned on the host AFTER the encoder has been queued (the GPU would otherwise idle for that long),
                # then the one fusion kernel is launched eagerly on the graph's outputs.
                pre = self._g_nav(t, dev, extra_key=(m.precision, ops.h16(), cfg.imagine_enc_pano, cfg.concat_imagine_with if
                                                     cfg.imagine_enc_pano else None), weights_token=tok,
                                  borrowed={'ctx_kv%d' % i: x for i, x in enumerate(kv)}, no_clone_prefix='_')
                out = m.fuse_logits(pre, batch['gmap_vpids'], batch['vp_cand_vpids'], Gb, Pb)
                if (Gb, Pb) != (G, P):
                    cut = {'gmap_embeds': G, 'global_logits': G, 'fused_logits': G, 'vp_embeds': P, 'local_logits': P}
                    out = {k: (v[:, :cut[k]] if k in cut and v is not None else v) for k, v in out.items()}
                return out
            return m(mode, batch)
        if mode in ('language', 'imagine', 'align_with_contrastive_loss'):
            return m(mode, batch)
        raise NotImplementedError('wrong mode: %s' % mode)
