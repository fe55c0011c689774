"""HAMT-Imagine on libvlnimagine: drop-in for ``models.model_HAMT.VLNBertCMT`` / ``models.vilmodel_cmt.NavCMT``.

Same constructor (``VLNBertCMT(args)``), the reference's keyword-style ``forward(mode, ...)`` with modes
language / history / imagine / align_with_contrastive_loss / visual, same return types and parameter names
(VLN-HAMT/finetune_src/models/model_HAMT.py:13-96, models/vilmodel_cmt.py:966-1205), so the unmodified
agent (r2r/agent_cmt.py) can hold it as ``self.vln_bert``.  The released configuration is implemented:
``concat_imagine_with='language'``, ``no_lang_ca=False``, ``act_pred_token in {'ob_txt', 'ob'}``,
``bypass_imag_encoder=True``, ``num_h_layers = num_r_layers = 0``.

The two token streams of a cross-modal layer - language+imagination (C tokens) and history+observation
(Nv tokens) - live in ONE row-stacked activation; the bidirectional cross-attention, which shares its
weights between the two directions (vilmodel_cmt.py:385-397), is a single QKV GEMM / output GEMM / LayerNorm
over all rows, and the per-stream self-attention and FFN blocks are grouped launches.
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
import torch.nn as nn

from . import autograd_ops as ag
from . import blocks, graphs, ops, params
from .blocks import Stream
from .config import hamt_config
from .duet import _f32c, align_forward
from .ops import BF16, F32, HIDDEN


class NavCMT(nn.Module):
    """models/vilmodel_cmt.py:966-1205."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        c = config
        if c.num_h_layers or c.num_r_layers:
            raise NotImplementedError('num_h_layers / num_r_layers > 0 are not used by the released HAMT-Imagine runs')
        if c.no_lang_ca:
            raise NotImplementedError('no_lang_ca=True is not supported (the reference itself warns that it breaks the imagination path)')
        if c.act_pred_token not in ('ob_txt', 'ob', 'ob_hist', 'ob_txt_hist', 'ob_imagine_text'):      # H/r2r/parser.py:67
            raise NotImplementedError('act_pred_token %r' % c.act_pred_token)
        if c.act_pred_token == 'ob_imagine_text' and not c.imagine_enc_pano:
            raise NotImplementedError("act_pred_token 'ob_imagine_text' needs imagine_enc_pano")
        self.embeddings = params.BertEmbeddingsP(c)
        self.img_embeddings = params.HamtImageEmbeddingsP(c)
        self.hist_embeddings = params.HistoryEmbeddingsP(c)
        if c.imagine_enc_pano and (c.use_cosine_aux_loss or c.no_loss_test):
            if c.aux_loss_type not in ('cosine', 'contrastive-InfoNCE', 'constrastive-margin'):
                raise NotImplementedError('aux_loss_type %r' % c.aux_loss_type)
            self.contrastive_alignment_model = params.AlignModelP()
        if c.imagine_enc_pano:
            if c.concat_imagine_with not in ('language', 'visual'):
                raise NotImplementedError('concat_imagine_with=%r' % c.concat_imagine_with)
            # the released recipe: bypass + 'language' (scripts/run_r2r.sh:70-74); the parser defaults (r2r/parser.py:109,122):
            # ImagineEmbeddings encoder + 'visual' - inference only here, fine-tuning them raises NotImplementedError
            self.imagine_embeddings = params.BypassImagineEmbeddingsP() if c.bypass_imag_encoder else params.ImagineEmbeddingsP(c)
        self.encoder = params.HamtEncoderP(c)
        self.next_action = params.NextActionP(c.pred_head_dropout_prob)
        params.bert_init_(self)
        if not c.update_lang_bert:                             # H/models/vilmodel_cmt.py:461-463
            for p_ in self.encoder.layer.parameters():
                p_.requires_grad = False
        self.fix_lang_embedding = c.fix_lang_embedding
        self.fix_hist_embedding = c.fix_hist_embedding
        self.fix_obs_embedding = c.fix_obs_embedding
        if c.imagine_enc_pano:
            self.fix_imagine_embeds = c.fix_imagine_embeds
        self.precision = os.environ.get('VLN_IMAGINE_PRECISION', 'bf16')
        # 16-bit operand format of inference calls in the 'bf16' (= 16-bit tensor-core) mode: 'auto' picks fp16 when the weights
        # prove it safe (blocks.operand_format), 'bf16' / 'f16' force one
        self.operand16 = os.environ.get('VLN_IMAGINE_OPERAND16', 'auto')
        self._fmt_cache = {}
        self._packs = None
        self._mean_idx = {}

    def _pk(self):
        if self._packs is None:
            pk = {}
            pk['lang'] = [blocks.SelfFFNPack([l.attention], [l.intermediate], [l.output]) for l in self.encoder.layer]
            xs = self.encoder.x_layers
            pk['x_cross'] = []
            for x in xs:
                va = x.visual_attention
                pk['x_cross'].append({
                    'qkv': blocks.LinearPack([va.att.query.weight, va.att.key.weight, va.att.value.weight],
                                             [va.att.query.bias, va.att.key.bias, va.att.value.bias]),
                    'o': blocks.LinearPack([va.output.dense.weight], [va.output.dense.bias]),
                    'ln': blocks.LNPack([va.output.LayerNorm])})
            pk['x_self'] = [blocks.SelfFFNPack([x.lang_self_att, x.visn_self_att], [x.lang_inter, x.visn_inter],
                                               [x.lang_output, x.visn_output]) for x in xs]
            pk['ob_img'] = blocks.LinearPack([self.img_embeddings.img_linear.weight], [self.img_embeddings.img_linear.bias])
            he = self.hist_embeddings
            pk['hist_img'] = blocks.LinearPack([he.img_linear.weight], [he.img_linear.bias])
            pk['hist_ln'] = blocks.LNPack([he.layer_norm])
            if he.pano_encoder is not None:
                pk['hist_pano_img'] = blocks.LinearPack([he.pano_img_linear.weight], [he.pano_img_linear.bias])
                pk['hist_pano'] = [blocks.SelfFFNPack([l.attention], [l.intermediate], [l.output]) for l in he.pano_encoder.layer]
            if self.config.imagine_enc_pano and not self.config.bypass_imag_encoder:
                im = self.imagine_embeddings
                pk['imag_img'] = blocks.LinearPack([im.pano_img_linear.weight], [im.pano_img_linear.bias])
                pk['imag_enc'] = [blocks.SelfFFNPack([l.attention], [l.intermediate], [l.output]) for l in im.pano_encoder.layer]
                pk['imag_ln0'] = blocks.LNPack([im.pano_img_layer_norm])
                pk['imag_ln1'] = blocks.LNPack([im.layer_norm])
            pk['act'] = blocks.ClsHeadPack([self.next_action], last_index=4)
            if hasattr(self, 'contrastive_alignment_model'):
                ip = self.contrastive_alignment_model.image_proj
                pk['align'] = [blocks.LinearPack([ip.fc1.weight]), blocks.LinearPack([ip.fc2.weight]),
                               blocks.LinearPack([ip.fc3.weight])]
            self._packs = pk
        return self._packs

    def _apply(self, fn, *a, **k):
        self._packs = None
        self._mean_idx = {}
        return super()._apply(fn, *a, **k)

    @property
    def lowp(self):
        if self.precision not in ('bf16', 'fp32'):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        return self.precision == 'bf16'

    def _recording(self, *inputs) -> bool:
        if not torch.is_grad_enabled():
            return False
        return any(torch.is_tensor(t) and t.requires_grad for t in inputs) or any(p.requires_grad for p in self.parameters())

    def _drop(self):
        """(hidden, attention, prediction-head) dropout of this call: the config's probabilities in train() mode"""
        if not self.training:
            return (0.0, 0.0, 0.0)
        c = self.config
        ps = (float(c.hidden_dropout_prob), float(c.attention_probs_dropout_prob), float(c.pred_head_dropout_prob))
        if max(ps) > 0 and not self.lowp:
            raise NotImplementedError('dropout is implemented for the bf16 kernels only: use eval() or p = 0 in the fp32 check mode')
        if max(ps) > 0 and not torch.is_grad_enabled():
            raise NotImplementedError('train() mode with dropout under torch.no_grad() is not supported: call .eval() for inference')
        return ps

    # -- modes ------------------------------------------------------------------------------------
    def forward_text(self, txt_ids, txt_masks):
        """'language', :1008-1031."""
        ops.ensure_init(txt_ids)
        lowp = self.lowp
        B, L = txt_ids.shape
        e = self.embeddings
        frozen = self.fix_lang_embedding or not self.config.update_lang_bert
        with blocks.grad_mode(self._recording() and not frozen, self._drop() if not frozen else (0.0, 0.0)):
            x = blocks.embed(B * L, txt_ids.device, idx=txt_ids.long().contiguous().view(-1), table=e.word_embeddings.weight,
                             pos_table=e.position_embeddings.weight, pos_period=L,
                             const_rows=(e.token_type_embeddings.weight[0],), out_ln=e.LayerNorm, lowp=lowp, dropout=True)
            s = [Stream(0, B, L, blocks.mask_u8(txt_masks))]
            for pk in self._pk()['lang']:
                x = blocks.self_attn_ffn(x, pk, s, None, lowp, defer=True)
            x = blocks.materialize(x, lowp, want16=False)
        out = x.f32.view(B, L, HIDDEN)
        return out.detach() if frozen else out

    def _mean_rows(self, B, n, row0, per, dev):
        """(offsets, rows) index arrays of B disjoint n-row segments, segment b = rows row0 + b * per + [0, n).  Built once per
        layout: a captured graph replays the first eager call's arrays and must not create its own."""
        key = (B, n, row0, per, str(dev))
        if key not in self._mean_idx:
            idx = row0 + torch.arange(B, device=dev)[:, None] * per + torch.arange(n, device=dev)[None, :]
            self._mean_idx[key] = (torch.arange(0, B * n + 1, n, dtype=torch.int32, device=dev), idx.reshape(-1).to(torch.int32))
        return self._mean_idx[key]

    def forward_history(self, hist_img_feats, hist_ang_feats, ob_step_ids, hist_pano_img_feats, hist_pano_ang_feats):
        """'history': HistoryEmbeddings.forward, :576-618."""
        he, lowp, pk = self.hist_embeddings, self.lowp, self._pk()
        recording = not self.fix_hist_embedding and self._recording(hist_img_feats) and any(p.requires_grad for p in he.parameters())
        type_row = he.type_embedding.weight[0]
        with blocks.grad_mode(recording, self._drop() if recording else (0.0, 0.0)):
            if hist_img_feats is None:
                ops.ensure_init(he.cls_token)
                y = blocks.embed(1, he.cls_token.device, a=he.cls_token.view(1, HIDDEN), const_rows=(type_row,), out_ln=he.layer_norm,
                                 dropout=True).f32
                return y.detach() if self.fix_hist_embedding else y
            ops.ensure_init(hist_img_feats)
            dev = hist_img_feats.device
            B = hist_img_feats.shape[0]
            a = blocks.linear(blocks.operand(_f32c(hist_img_feats), lowp), pk['hist_img'], lowp, out_dtype=F32)
            # position embedding of the current step: a [B] index tensor (the same id for every episode, :597), so the
            # step never becomes a pointer baked into a captured graph
            if torch.is_tensor(ob_step_ids) and ob_step_ids.numel() == B:
                step_idx = ob_step_ids.long().contiguous().view(-1)
            else:
                step = int(ob_step_ids.view(-1)[0]) if torch.is_tensor(ob_step_ids) else int(ob_step_ids)
                step_idx = torch.full((B,), step, dtype=torch.int64, device=dev)
            e32 = blocks.embed(B, dev, a=a, a_ln=he.img_layer_norm, feat=_f32c(hist_ang_feats), feat_lin=he.ang_linear,
                               feat_ln=he.ang_layer_norm, idx=step_idx, table=he.position_embeddings.weight, const_rows=(type_row,)).f32
            pano_mean = None
            if he.pano_encoder is not None:
                V = hist_pano_img_feats.shape[1]
                pa = blocks.linear(blocks.operand(_f32c(hist_pano_img_feats).view(B * V, -1), lowp), pk['hist_pano_img'], lowp, out_dtype=F32)
                x = blocks.embed(B * V, dev, a=pa, a_ln=he.pano_img_layer_norm, feat=_f32c(hist_pano_ang_feats).view(B * V, -1),
                                 feat_lin=he.pano_ang_linear, feat_ln=he.pano_ang_layer_norm, lowp=lowp, dropout=True)
                s = [Stream(0, B, V, None)]                   # the reference's mask is all ones (:606-607)
                for lp in pk['hist_pano']:
                    x = blocks.self_attn_ffn(x, lp, s, None, lowp)
                off, idx = self._mean_rows(B, V, 0, V, dev)
                pano_mean = blocks.segment_mean(x.f32, off, idx, B, seg=V)
            y = blocks.layer_norm(e32, pano_mean, pk['hist_ln'], 1e-12, False).f32
            if blocks._Mode.p_hidden > 0:                     # nn.Dropout after the final LayerNorm (:616)
                y = ag.dropout(y, blocks._Mode.p_hidden)
        return y.detach() if self.fix_hist_embedding else y

    def forward_imagination(self, imagine_pano_img_feats, imagine_masks=None):
        """'imagine', :1040-1048: the bypass embedding (:620-631) or the ImagineEmbeddings encoder (:634-703)."""
        ops.ensure_init(imagine_pano_img_feats)
        B, I, _ = imagine_pano_img_feats.shape
        if not self.config.bypass_imag_encoder:
            return self._imagination_encoder(imagine_pano_img_feats, imagine_masks)
        with blocks.grad_mode(self._recording(imagine_pano_img_feats) and not self.fix_imagine_embeds):
            y = blocks.embed(B * I, imagine_pano_img_feats.device, a=_f32c(imagine_pano_img_feats).view(B * I, HIDDEN),
                             const_rows=(self.imagine_embeddings.type_embedding.weight[0],))
        out = y.f32.view(B, I, HIDDEN)
        return out.detach() if self.fix_imagine_embeds else out

    def _imagination_encoder(self, feats, imagine_masks):
        """ImagineEmbeddings.forward, :634-703: features + position + type embedding -> Linear + LN -> post-LN BertEncoder over
        the imaginations of an episode (additive -10000 mask) -> LN."""
        im, lowp, pk = self.imagine_embeddings, self.lowp, self._pk()
        if imagine_masks is None:
            raise ValueError("mode 'imagine' needs imagine_masks when bypass_imag_encoder is off (r2r/agent_cmt.py:413-417)")
        B, I, _ = feats.shape
        if I >= im.position_embeddings.weight.shape[0]:
            raise ValueError('imagination length %d out of bounds (max_imagination_len %d, :683)' % (I, im.position_embeddings.weight.shape[0]))
        recording = self._recording(feats) and any(p.requires_grad for p in im.parameters()) and not self.fix_imagine_embeds
        with blocks.grad_mode(recording, self._drop() if recording else (0.0, 0.0)):
            x = blocks.embed(B * I, feats.device, a=_f32c(feats).view(B * I, -1), pos_table=im.position_embeddings.weight,
                             pos_period=I, const_rows=(im.type_embedding.weight[0],), lowp=lowp, want32=not lowp)
            a = blocks.linear(x.operand(lowp), pk['imag_img'], lowp, out_dtype=F32)
            x = blocks.layer_norm(a, None, pk['imag_ln0'], 1e-12, lowp)
            if blocks._Mode.p_hidden > 0:                     # nn.Dropout after both LayerNorms (:686, :701)
                x = blocks.as_act(ag.dropout(x.f32, blocks._Mode.p_hidden), lowp)
            s = [Stream(0, B, I, blocks.mask_u8(imagine_masks))]
            for lp in pk['imag_enc']:
                x = blocks.self_attn_ffn(x, lp, s, None, lowp)
            out = blocks.layer_norm(x.f32, None, pk['imag_ln1'], 1e-12, False).f32
            if blocks._Mode.p_hidden > 0:
                out = ag.dropout(out, blocks._Mode.p_hidden)
        return out.view(B, I, HIDDEN)

    def forward_visual(self, txt_embeds, txt_masks, hist_embeds, hist_masks, ob_img_feats, ob_ang_feats, ob_nav_types,
                       ob_masks, imagine_embeds=None, imagine_masks=None):
        """'visual', :1056-1205."""
        ops.ensure_init(txt_embeds)
        cfg, lowp, pk = self.config, self.lowp, self._pk()
        dev = txt_embeds.device
        B, L, _ = txt_embeds.shape
        T, O = hist_embeds.shape[1], ob_img_feats.shape[1]
        if cfg.imagine_enc_pano:
            if imagine_embeds is None or imagine_masks is None:
                raise ValueError('visual mode needs imagine_embeds and imagine_masks when imagine_enc_pano is set')
            I = imagine_embeds.shape[1]
        else:
            I = 0
        # the imagination tokens ride on the language stream (:1109-1112) or on the vision stream (:1106-1108)
        on_visn = bool(I) and cfg.concat_imagine_with == 'visual'
        Il, Iv = (0, I) if on_visn else (I, 0)
        C, Nv = L + Il, T + O + Iv
        (r_l, r_v), ends, _ = blocks.stack_layout([B * C, B * Nv])
        recording = self._recording(txt_embeds, hist_embeds, ob_img_feats, imagine_embeds)
        with blocks.grad_mode(recording, self._drop() if recording else (0.0, 0.0)):
            # observation embedding :521-544, :1073-1077
            ie = self.img_embeddings
            a = blocks.linear(blocks.operand(_f32c(ob_img_feats).view(B * O, -1), lowp), pk['ob_img'], lowp, out_dtype=F32)
            ob = blocks.embed(B * O, dev, a=a, a_ln=ie.img_layer_norm, feat=_f32c(ob_ang_feats).view(B * O, -1), feat_lin=ie.ang_linear,
                              feat_ln=ie.ang_layer_norm, idx=ob_nav_types.long().contiguous().view(-1), table=ie.nav_type_embedding.weight,
                              const_rows=(self.embeddings.token_type_embeddings.weight[1],), out_ln=ie.layer_norm, dropout=True).f32
            if self.fix_obs_embedding:
                ob = ob.detach()
            # language stream = [txt ; imagine] (:1110), vision stream = [hist ; ob] (:1087) [; imagine] (:1106-1108)
            imag = [_f32c(imagine_embeds)] if I else []
            x = blocks.stack_segments([[_f32c(txt_embeds)] + (imag if Il else []),
                                       [_f32c(hist_embeds), ob.view(B, O, HIDDEN)] + (imag if Iv else [])], (r_l, r_v), lowp)
            lang_mask = blocks.mask_u8(torch.cat([txt_masks.bool(), imagine_masks.bool()], 1) if Il else txt_masks)
            visn_mask = blocks.mask_u8(torch.cat([hist_masks.bool(), ob_masks.bool()] + ([imagine_masks.bool()] if Iv else []), 1))
            streams = [Stream(r_l, B, C, lang_mask, 0), Stream(r_v, B, Nv, visn_mask, 1)]
            for cp, sp in zip(pk['x_cross'], pk['x_self']):
                # bidirectional cross-attention with shared weights, both directions read the layer inputs (:385-397)
                x = blocks.attn(x, cp['qkv'], cp['o'], cp['ln'], streams, ends, lowp, kv_of=(1, 0))
                x = blocks.self_attn_ffn(x, sp, streams, ends, lowp, defer=True)
            x = blocks.materialize(x, lowp, ends, want16=False)

            lang_out = x.f32[r_l:r_l + B * C].view(B, C, HIDDEN)
            visn_out = x.f32[r_v:r_v + B * Nv].view(B, Nv, HIDDEN)
            txt_out, hist_out, ob_out = lang_out[:, :L], visn_out[:, :T], visn_out[:, T:T + O]      # :1173-1182
            tok = cfg.act_pred_token                           # :1189-1199
            if tok == 'ob':
                h = blocks.take_rows(ob_out, lowp)
            else:
                if tok == 'ob_txt':
                    gate = lang_out[:, 0]
                elif tok == 'ob_hist':                         # ob * hist[:, :1]: token 0 of the vision stream
                    gate = visn_out[:, 0]
                else:                                          # ob * (txt[:, :1] + hist[:, :1] | mean over the imagination tokens)
                    t0 = blocks.take_rows(lang_out[:, :1])
                    if tok == 'ob_txt_hist':
                        other = blocks.take_rows(visn_out[:, :1])
                    else:                                      # torch.mean(imagine_embeds, 1): all I output tokens, unmasked
                        off, idx = self._mean_rows(B, I, *((r_v + T + O, Nv) if on_visn else (r_l + L, C)), dev)
                        other = blocks.segment_mean(x.f32, off, idx, B, seg=I)
                    gate = blocks.embed(B, dev, a=t0, a2=other).f32
                h = blocks.mul_bcast(ob_out, gate, lowp)
            act_logits = blocks.mask_logits(blocks.cls_head(h, pk['act'], lowp), ob_nav_types)
        return act_logits, txt_out, hist_out, ob_out

    def h16_format(self):
        """16-bit operand format of this call (blocks.operand_format)"""
        return blocks.operand_format(self, self._fmt_cache, self.operand16)

    def forward(self, mode, **kw):
        with ops.half_format(self.h16_format()):
            return self._forward(mode, **kw)

    def _forward(self, mode, txt_ids=None, txt_embeds=None, txt_masks=None, hist_img_feats=None, hist_ang_feats=None,
                hist_pano_img_feats=None, hist_pano_ang_feats=None, hist_embeds=None, ob_step_ids=None, hist_masks=None,
                ob_img_feats=None, ob_ang_feats=None, ob_nav_types=None, ob_masks=None, imagine_pano_img_feats=None,
                imagine_masks=None, imagine_embeds=None, align_txt_embeds=None, align_imagine_embeds=None,
                sub_instr_segs=None, sub_instr_imag_flag=None, noun_phrase_segs=None, obs_instr_ids=None,
                return_cross_attention_probs=False):
        """Mode dispatch, :999-1205."""
        if return_cross_attention_probs:
            raise NotImplementedError('attention scores never leave the fused attention kernel')
        if mode == 'language':
            return self.forward_text(txt_ids, txt_masks)
        if mode == 'history':
            return self.forward_history(hist_img_feats, hist_ang_feats, ob_step_ids, hist_pano_img_feats, hist_pano_ang_feats)
        if mode == 'imagine':
            assert imagine_pano_img_feats is not None
            return self.forward_imagination(imagine_pano_img_feats, imagine_masks)
        if mode == 'align_with_contrastive_loss':
            ops.ensure_init(align_txt_embeds)
            with blocks.grad_mode(self._recording(align_txt_embeds, align_imagine_embeds), self._drop()):
                return align_forward(self, align_txt_embeds, align_imagine_embeds, sub_instr_imag_flag, noun_phrase_segs, self.lowp)
        if mode == 'visual':
            return self.forward_visual(txt_embeds, txt_masks, hist_embeds, hist_masks, ob_img_feats, ob_ang_feats,
                                       ob_nav_types, ob_masks, imagine_embeds, imagine_masks)
        raise NotImplementedError('wrong mode: %s' % mode)


def length2mask(lengths, size, device):
    """utils/misc.py:12-17: True where the position is PADDING."""
    if torch.is_tensor(lengths):                 # superset of the reference: lengths may already be a tensor
        lens = lengths.to(device=device, dtype=torch.int64)
    else:
        lens = torch.as_tensor(lengths, dtype=torch.int64, device=device)
    return torch.arange(size, dtype=torch.int64, device=device)[None, :] >= lens[:, None]


class VLNBertCMT(nn.Module):
    """models/model_HAMT.py:13-96.  Inference calls of the per-step modes ('visual', 'history') are replayed from
    CUDA graphs (graphs.GraphedCall); ``use_cuda_graphs = False`` gives plain eager launches."""

    VIS_TENSORS = ('txt_embeds', 'txt_masks', 'ob_img_feats', 'ob_ang_feats', 'ob_nav_types', 'ob_masks', 'imagine_embeds',
                   'imagine_masks')
    HIST_TENSORS = ('hist_img_feats', 'hist_ang_feats', 'hist_pano_img_feats', 'hist_pano_ang_feats')

    def __init__(self, args):
        super().__init__()
        self.args = args
        self.vln_bert = NavCMT(hamt_config(args))
        ckpt = getattr(args, 'bert_ckpt_file', None)
        if ckpt is not None:                                   # models/vlnbert_init.py:20-31
            sd = {}
            for k, v in torch.load(ckpt, map_location='cpu').items():
                k = k[7:] if k.startswith('module') else k
                sd[k[5:] if k.startswith('bert.') else k] = v
            self.vln_bert.load_state_dict(sd, strict=False)
        self.drop_env = nn.Dropout(p=getattr(args, 'feat_dropout', 0.0))
        self.use_cuda_graphs = os.environ.get('VLN_IMAGINE_CUDA_GRAPHS', '1') != '0'
        self._wt_cache = {}
        self._g_vis = graphs.GraphedCall(self._vis_fn)
        self._g_hist = graphs.GraphedCall(self._hist_fn)
        self._buckets = graphs.ShapeBuckets()

    def _apply(self, fn, *a, **k):
        self._wt_cache = {}
        self._g_vis.clear()
        self._g_hist.clear()
        return super()._apply(fn, *a, **k)

    def _env_dropout(self, x):
        """models/model_HAMT.py: nn.Dropout(feat_dropout) on image features in train() mode"""
        if x is not None and self.training and self.drop_env.p > 0:
            dev = self.vln_bert.embeddings.LayerNorm.weight.device
            x = x if x.is_cuda else x.to(dev, non_blocking=True)
            ops.ensure_init(x)
            return ag.dropout(x.float(), float(self.drop_env.p))
        return x

    def _vis_fn(self, t):
        logits, txt_o, hist_o, ob_o = self.vln_bert.forward_visual(
            t['txt_embeds'], t['txt_masks'], t['hist_embeds'], t['hist_masks'], t['ob_img_feats'], t['ob_ang_feats'],
            t['ob_nav_types'], t['ob_masks'], t.get('imagine_embeds'), t.get('imagine_masks'))
        states = hist_o[:, 0] if self.args.no_lang_ca else self._states(txt_o, hist_o)
        return {'act_logits': logits, 'states': states}

    def _hist_fn(self, t):
        return {'hist': self.vln_bert.forward_history(t['hist_img_feats'], t['hist_ang_feats'], t['ob_step_ids'],
                                                      t.get('hist_pano_img_feats'), t.get('hist_pano_ang_feats'))}

    def _graphable(self):
        return self.use_cuda_graphs and not self.training and not torch.is_grad_enabled()

    def forward(self, mode, **kw):
        with ops.half_format(self.vln_bert.h16_format()):
            return self._forward(mode, **kw)

    def _forward(self, mode, txt_ids=None, txt_masks=None, txt_embeds=None, hist_img_feats=None, hist_ang_feats=None,
                 hist_pano_img_feats=None, hist_pano_ang_feats=None, hist_embeds=None, hist_lens=None, ob_step=None,
                ob_img_feats=None, ob_ang_feats=None, ob_nav_types=None, ob_masks=None, imagine_pano_img_feats=None,
                imagine_masks=None, imagine_embeds=None, align_txt_embeds=None, align_imagine_embeds=None,
                sub_instr_segs=None, sub_instr_imag_flag=None, noun_phrase_segs=None, obs_instr_ids=None,
                return_states=False, return_cross_attention_probs=False):
        m = self.vln_bert
        if mode == 'language':
            return m('language', txt_ids=txt_ids, txt_masks=txt_masks)
        if mode == 'imagine':
            return m('imagine', imagine_pano_img_feats=self._env_dropout(imagine_pano_img_feats), imagine_masks=imagine_masks)
        if mode == 'align_with_contrastive_loss':
            return m('align_with_contrastive_loss', align_txt_embeds=align_txt_embeds, txt_masks=txt_masks,
                     align_imagine_embeds=align_imagine_embeds, imagine_masks=imagine_masks, sub_instr_segs=sub_instr_segs,
                     sub_instr_imag_flag=sub_instr_imag_flag, noun_phrase_segs=noun_phrase_segs, obs_instr_ids=obs_instr_ids)
        if mode == 'history':
            if hist_img_feats is not None and self._graphable():
                dev = m.embeddings.LayerNorm.weight.device
                loc = dict(hist_img_feats=hist_img_feats, hist_ang_feats=hist_ang_feats,
                           hist_pano_img_feats=hist_pano_img_feats, hist_pano_ang_feats=hist_pano_ang_feats)
                t = {k: loc[k] for k in self.HIST_TENSORS if loc[k] is not None}
                t['ob_step_ids'] = torch.full((hist_img_feats.shape[0],), int(ob_step), dtype=torch.int64)
                return self._g_hist(t, dev, extra_key=(m.precision, ops.h16()), weights_token=graphs.weights_token(m, self._wt_cache))['hist']
            return m('history', hist_img_feats=self._env_dropout(hist_img_feats), hist_ang_feats=hist_ang_feats,
                     ob_step_ids=ob_step, hist_pano_img_feats=self._env_dropout(hist_pano_img_feats),
                     hist_pano_ang_feats=hist_pano_ang_feats)
        if mode == 'visual':
            if return_cross_attention_probs:
                raise NotImplementedError('attention scores never leave the fused attention kernel')
            hist = torch.stack(hist_embeds, 1)                                   # list of (B, 768) -> (B, T, 768)
            if self._graphable():
                dev = m.embeddings.LayerNorm.weight.device
                loc = dict(txt_embeds=txt_embeds, txt_masks=txt_masks, ob_img_feats=ob_img_feats, ob_ang_feats=ob_ang_feats,
                           ob_nav_types=ob_nav_types, ob_masks=ob_masks, imagine_embeds=imagine_embeds, imagine_masks=imagine_masks)
                t = {k: loc[k] for k in self.VIS_TENSORS if loc[k] is not None}
                t['hist_embeds'] = hist
                t['hist_masks'] = length2mask(hist_lens, hist.size(1), 'cpu').logical_not()
                T, O = hist.size(1), ob_img_feats.shape[1]
                if self._buckets.active((T, O)):
                    # the history grows by one token per step and the observation count changes with it: pad T to multiples of 4 and
                    # O to multiples of 8 (masked like the reference's batch padding) so that a few captured graphs serve a rollout
                    Tb, Ob = self._buckets.up(T, 4), self._buckets.up(O, 8)
                    dims = {'hist_embeds': {1: Tb}, 'hist_masks': {1: Tb}, 'ob_img_feats': {1: Ob}, 'ob_ang_feats': {1: Ob},
                            'ob_nav_types': {1: Ob}, 'ob_masks': {1: Ob}}
                    t = {k: (graphs.pad_to(v, dims[k], dev) if k in dims else v) for k, v in t.items()}
                out = self._g_vis(t, dev, extra_key=(m.precision, ops.h16(), m.config.imagine_enc_pano),
                                  weights_token=graphs.weights_token(m, self._wt_cache))
                logits = out['act_logits'][:, :O]
                return (logits, out['states']) if return_states else (logits,)
            hist_masks = length2mask(hist_lens, hist.size(1), hist.device).logical_not()
            act_logits, txt_o, hist_o, ob_o = m('visual', txt_embeds=txt_embeds, txt_masks=txt_masks, hist_embeds=hist,
                                                hist_masks=hist_masks, ob_img_feats=self._env_dropout(ob_img_feats),
                                                ob_ang_feats=ob_ang_feats, ob_nav_types=ob_nav_types, ob_masks=ob_masks,
                                                imagine_embeds=imagine_embeds, imagine_masks=imagine_masks)
            if return_states:
                states = hist_o[:, 0] if self.args.no_lang_ca else self._states(txt_o, hist_o)
                return act_logits, states
            return (act_logits,)
        raise NotImplementedError('wrong mode: %s' % mode)

    def _states(self, txt_o, hist_o):
        """states = txt_embeds[:, 0] * hist_embeds[:, 0]  (model_HAMT.py:86): one mul_bcast launch with
        one row per episode."""
        B = txt_o.shape[0]
        y32, _ = ops.mul_bcast(hist_o, hist_o.stride(0), txt_o, txt_o.stride(0), B, 1, want16=False)
        return y32
