"""DUET pre-training forward on libvlnimagine (SURVEY.md section 8(f), row N4): drop-in for
``GlocalTextPathCMTPreTraining`` (VLN-DUET/pretrain_src/model/pretrain_cmt.py:38-262) with the R2R proxy tasks mlm / mrc / sap
(config/r2r_pretrain.json) behind the reference's ``forward(batch, task, compute_loss)``.

The pre-training model reuses every block of the navigation model (same kernels: tcgen05 GEMMs with folded LayerNorms, fused
attention, row kernels); what it adds is
  * whole trajectories through the panorama encoder at once (vilmodel.py:484-528),
  * the per-trajectory aggregation of graph-node features (``GlobalMapEncoder._aggregate_gmap_features``, vilmodel.py:577-611:
    a Python triple loop over trajectories, steps and candidates) -> ``gmap_aggregation_rows`` turns it into ONE segment-mean
    launch (``vi_gather_mean``) over the flattened trajectory embeddings,
  * the lang2visn layers of MLM (the instruction attends to the map / the panorama, vilmodel.py:400-411, 700-747),
  * the vocabulary-wide tied MLM decoder (768 -> 30522, padded to 30528 columns for the tensor-core tiles), the MRC view
    classifier (768 -> 1000) and the per-row losses (``vi_ce_rows`` / ``vi_kl_rows``).
Parameter names equal the reference's (tests/golden/duet_pretrain_manifest.json).  Oracle: oracle/pretrain_oracle.py, pinned to
the real reference.

Training: with autograd recording (grad mode on, parameters that require grad) ``forward`` runs the same layer sequence from the
differentiable blocks (``_trunk_train``, as duet._navigation_train) and returns the per-row losses; ``loss.mean().backward()`` runs
libvlnimagine kernels only.  The padded decoder / classifier is ``autograd_ops.PaddedLinearFn`` (the tied decoder's weight gradient
adds onto the word-embedding lookup's), the losses ``CERowsFn`` / ``KLRowsFn``, whose backward kernel (vi_ce_rows_bwd /
vi_kl_rows_bwd) writes the bf16 operand of the decoder's gradient GEMMs directly.  Train-mode dropout: bf16 only, as the
navigation model.  Under torch.no_grad() the inference path below runs unchanged.
"""
from __future__ import annotations

import copy
from typing import List, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn


def gmap_aggregation_rows(traj_step_lens: Sequence[int], traj_vp_view_lens: Sequence[int], traj_vpids: List[List[str]],
                          traj_cand_vpids: List[List[List[str]]], gmap_vpids: List[list], n_views: int) -> Tuple[np.ndarray, np.ndarray, int]:
    """-> (offsets int32 [B * G + 1], row_idx int32 [n], G) for ``vi_gather_mean`` over ``src`` = the panorama-encoder output of all
    N trajectory steps flattened to [N * n_views + 1, 768] with ONE ZERO ROW appended (index N * n_views).

    Output row b * G + g is the feature of ``gmap_vpids[b][g]``:
      * g = 0 ([stop]) and the padding behind an episode's own nodes: the zero row (a unit segment - an empty segment would be 0 / 0);
      * a visited viewpoint: the mean over the valid views of its LAST panorama in the trajectory (the dict of the reference is
        overwritten by later steps, vilmodel.py:591);
      * an unvisited one: the mean over the candidate views that pointed at it while it was still unvisited (:592-595)."""
    B = len(traj_step_lens)
    G = max(len(v) for v in gmap_vpids)
    N = int(sum(traj_step_lens))
    zero_row = N * n_views
    offsets, rows = [0], []
    step0 = 0
    for b in range(B):
        visited, unvisited = {}, {}
        for t in range(traj_step_lens[b]):
            base = (step0 + t) * n_views
            visited[traj_vpids[b][t]] = [base + j for j in range(int(traj_vp_view_lens[step0 + t]))]
            for j, vp in enumerate(traj_cand_vpids[b][t]):
                if vp not in visited:
                    unvisited.setdefault(vp, []).append(base + j)
        step0 += traj_step_lens[b]
        for g in range(G):
            vp = gmap_vpids[b][g] if g < len(gmap_vpids[b]) else None
            if g == 0 or vp is None:
                rows.append(zero_row)
            elif vp in visited:
                rows.extend(visited[vp])
            else:
                rows.extend(unvisited[vp])         # KeyError: a graph node that was never seen - as in the reference
            offsets.append(len(rows))
    return np.asarray(offsets, np.int32), np.asarray(rows, np.int32), G


# ---------------------------------------------------------------------------------------------------------------------
# the module
# ---------------------------------------------------------------------------------------------------------------------
def _lazy():
    from . import blocks, duet, ops, params
    return blocks, duet, ops, params


class _MLMTransform(nn.Module):
    def __init__(self):
        super().__init__()
        self.dense = nn.Linear(768, 768)
        self.LayerNorm = nn.LayerNorm(768, eps=1e-12)


class _MLMPredictions(nn.Module):
    """BertLMPredictionHead: transform (dense -> gelu -> LayerNorm), decoder tied to the word embeddings, bias"""

    def __init__(self, vocab):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(vocab))
        self.transform = _MLMTransform()
        self.decoder = nn.Linear(768, vocab, bias=False)


class _MLMHead(nn.Module):
    def __init__(self, vocab):
        super().__init__()
        self.predictions = _MLMPredictions(vocab)


class _RegionClassification(nn.Module):
    """RegionClassification (pretrain_cmt.py:18-27): Linear -> ReLU -> LayerNorm -> Linear(768, label_dim)"""

    def __init__(self, label_dim):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(768, 768), nn.ReLU(), nn.LayerNorm(768, eps=1e-12), nn.Linear(768, label_dim))


def _make_bert(config):
    blocks, duet, ops, params = _lazy()

    class GlocalTextPathCMT(duet.GlocalTextPathNavCMT):
        """VLN-DUET/pretrain_src/model/vilmodel.py:627-747: the navigation model's encoders (with the lang2visn blocks),
        without heads and without the imagination modules.  Inherits forward_text / the panorama encoder / the weight packs."""

        def __init__(self, cfg):
            nn.Module.__init__(self)
            self.config = cfg
            self.embeddings = params.BertEmbeddingsP(cfg)
            self.lang_encoder = params.LayerStack('layer', [params.BertLayerP() for _ in range(cfg.num_l_layers)])
            self.img_embeddings = params.DuetImageEmbeddingsP(cfg)
            self.local_encoder = params.LocalVPEncoderP(cfg)
            self.global_encoder = params.GlobalMapEncoderP(cfg)
            self.sap_fuse_linear = None
            params.bert_init_(self)
            import os
            self.precision = os.environ.get('VLN_IMAGINE_PRECISION', 'bf16')
            self.operand16 = os.environ.get('VLN_IMAGINE_OPERAND16', 'auto')
            self._fmt_cache = {}
            self._packs = None
            self._ids = duet._IdTable()
            self.context_cache = False
            self._ctx_slots = {}
            self.context_hits = self.context_misses = 0

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
                # lang2visn: key | value of the map / panorama tokens per branch, the language-side blocks of both branches
                pk['l2v_kv'] = [[blocks.LinearPack([x.visual_attention.att.key.weight, x.visual_attention.att.value.weight],
                                                   [x.visual_attention.att.key.bias, x.visual_attention.att.value.bias])
                                 for x in (g, l)] for g, l in zip(gl, ll)]
                pk['l2v_self'] = [blocks.SelfFFNPack([g.lang_self_att, l.lang_self_att], [g.lang_inter, l.lang_inter],
                                                     [g.lang_output, l.lang_output]) for g, l in zip(gl, ll)]
                if self.global_encoder.sprel_linear is not None:
                    sl = self.global_encoder.sprel_linear
                    pk['sprel'] = blocks.StackPack([sl.weight, sl.bias])
                self._packs = pk
            return self._packs

    return GlocalTextPathCMT(config)


class GlocalTextPathCMTPreTraining(nn.Module):
    """pretrain_cmt.py:38-262.  ``forward(batch, task, compute_loss=True)`` with task in {'mlm', 'mrc', 'sap'}; the batch is the
    dict the reference's collate functions build (data/tasks.py; vln-imagine_b200/synth.duet_pretrain_batch has the layout)."""

    def __init__(self, config):
        super().__init__()
        blocks, duet, ops, params = _lazy()
        cfg = copy.copy(config)
        cfg.use_lang2visn_attn = True                        # model/vilmodel.py: pre-training builds the lang2visn blocks
        cfg.imagine_enc_pano = False
        cfg.obj_feat_size = 0
        self.config = cfg
        self.bert = _make_bert(cfg)
        tasks = getattr(config, 'pretrain_tasks', ['mlm', 'mrc', 'sap'])
        if 'mlm' in tasks:
            self.mlm_head = _MLMHead(cfg.vocab_size)
        if 'mrc' in tasks:
            self.image_classifier = _RegionClassification(getattr(config, 'image_prob_size', 1000))
        if 'sap' in tasks:
            self.global_sap_head = params.ClsPredictionP()
            self.local_sap_head = params.ClsPredictionP()
            self.sap_fuse_linear = params.ClsPredictionP(input_size=2 * 768) if getattr(cfg, 'glocal_fuse', True) else None
        params.bert_init_(self)
        if hasattr(self, 'mlm_head'):                        # tie_weights (pretrain_cmt.py:112-117)
            self.mlm_head.predictions.decoder.weight = self.bert.embeddings.word_embeddings.weight
        self._head_packs = None

    def _apply(self, fn, *a, **k):
        self._head_packs = None
        return super()._apply(fn, *a, **k)

    # -- derived weights of the heads ---------------------------------------------------------------------------------
    def _hp(self):
        blocks, duet, ops, params = _lazy()
        if self._head_packs is None:
            hp = {}
            if hasattr(self, 'mlm_head'):
                pr = self.mlm_head.predictions
                hp['mlm_t'] = blocks.LinearPack([pr.transform.dense.weight], [pr.transform.dense.bias])
                hp['mlm_ln'] = blocks.LNPack([pr.transform.LayerNorm])
                hp['mlm_dec'] = _PaddedLinear(pr.decoder.weight, pr.bias)
            if hasattr(self, 'image_classifier'):
                net = self.image_classifier.net
                hp['mrc0'] = blocks.LinearPack([net[0].weight], [net[0].bias])
                hp['mrc_ln'] = blocks.LNPack([net[2]])
                hp['mrc3'] = _PaddedLinear(net[3].weight, net[3].bias)
            if hasattr(self, 'global_sap_head'):
                hp['sap'] = blocks.ClsHeadPack([self.global_sap_head, self.local_sap_head])
                if self.sap_fuse_linear is not None:
                    hp['fuse'] = blocks.ClsHeadPack([self.sap_fuse_linear])
            self._head_packs = hp
        return self._head_packs

    # -- shared trunk ----------------------------------------------------------------------------------------------------
    def _trunk(self, batch, want_l2v=False):
        """GlocalTextPathCMT.forward / forward_mlm, model/vilmodel.py:660-747 -> dict of row-stacked results"""
        blocks, duet, ops, params = _lazy()
        bert = self.bert
        lowp, pk = bert.lowp, bert._pk()
        dev = bert.embeddings.LayerNorm.weight.device
        F32, HID = torch.float32, 768
        to = lambda t, dt=None: torch.as_tensor(t).to(dev, dtype=dt, non_blocking=True)     # noqa: E731
        txt_ids = to(batch['txt_ids'])
        B, L = txt_ids.shape
        txt_lens = [int(x) for x in batch['txt_lens']]
        txt_masks = torch.arange(L, device=dev)[None, :] < to(batch['txt_lens'])[:, None]
        txt = bert.forward_text(txt_ids, txt_masks)                                  # (B, L, 768) fp32
        # every panorama of every trajectory through the panorama encoder (vilmodel.py:484-528)
        step_lens = [int(x) for x in batch['traj_step_lens']]
        view_lens = to(batch['traj_vp_view_lens'])
        pano, _ = bert.forward_panorama_per_step(to(batch['traj_view_img_fts'], F32), None, to(batch['traj_loc_fts'], F32),
                                                 to(batch['traj_nav_types']), view_lens, None)
        N, V, _ = pano.shape
        vl_host = [int(x) for x in batch['traj_vp_view_lens']]
        last = np.cumsum(step_lens) - 1
        # local branch: [stop] + the LAST panorama of each trajectory (vilmodel.py:538-553)
        P = max(vl_host[i] for i in last) + 1
        src = torch.cat([pano.reshape(N * V, HID), torch.zeros((1, HID), dtype=F32, device=dev)], 0)
        zero_row = N * V
        vp_idx = np.full((B, P), zero_row, np.int32)
        for b, i in enumerate(last):
            n = min(V, P - 1)
            vp_idx[b, 1:1 + n] = i * V + np.arange(n)
        vp_lens = torch.as_tensor([vl_host[i] + 1 for i in last], device=dev)
        vp_masks = torch.arange(P, device=dev)[None, :] < vp_lens[:, None]
        unit = lambda n: torch.arange(n + 1, dtype=torch.int32, device=dev)                # noqa: E731
        vp_img, _ = ops.gather_mean(src, unit(B * P), torch.from_numpy(vp_idx.reshape(-1)).to(dev), B * P, want16=False)
        le, ge = bert.local_encoder, bert.global_encoder
        # global branch: the graph-node features aggregated from the trajectory (vilmodel.py:577-611) in one segment-mean launch
        off, rows, G = gmap_aggregation_rows(step_lens, vl_host, batch['traj_vpids'], batch['traj_cand_vpids'],
                                             batch['gmap_vpids'], V)
        gmap_img, _ = ops.gather_mean(src, torch.from_numpy(off).to(dev), torch.from_numpy(rows).to(dev), B * G, want16=False)
        gmap_masks = torch.arange(G, device=dev)[None, :] < to(batch['gmap_lens'])[:, None]
        # input embeddings of both branches into one row-stacked activation (vilmodel.py:613-625, 538-553)
        row0, ends, R = blocks.stack_layout([B * G, B * P])
        x32 = torch.zeros((R, HID), dtype=F32, device=dev)
        x16 = torch.zeros((R, HID), dtype=ops.h16(), device=dev) if lowp else None
        r_l = row0[-1]
        if True:
            ops.embed_compose(B * G, dev, a=gmap_img, feat=to(batch['gmap_pos_fts'], F32).reshape(B * G, -1).contiguous(),
                              feat_w=ge.gmap_pos_embeddings[0].weight, feat_b=ge.gmap_pos_embeddings[0].bias,
                              feat_ln=(ge.gmap_pos_embeddings[1].weight, ge.gmap_pos_embeddings[1].bias),
                              idx=to(batch['gmap_step_ids']).long().contiguous().view(-1), table=ge.gmap_step_embeddings.weight,
                              y32=x32[0:B * G], y16=x16[0:B * G] if lowp else None)
        ops.embed_compose(B * P, dev, a=vp_img, feat=to(batch['vp_pos_fts'], F32).reshape(B * P, -1).contiguous(),
                          feat_w=le.vp_pos_embeddings[0].weight, feat_b=le.vp_pos_embeddings[0].bias,
                          feat_ln=(le.vp_pos_embeddings[1].weight, le.vp_pos_embeddings[1].bias),
                          y32=x32[r_l:r_l + B * P], y16=x16[r_l:r_l + B * P] if lowp else None)
        out = dict(B=B, L=L, G=G, P=P, r_l=r_l, ends=ends, txt=txt, txt_masks=txt_masks, vp_masks=vp_masks, dev=dev,
                   last=last, vl_host=vl_host, V=V)
        x_in = blocks.Act(x32, x16)
        tmask = blocks.mask_u8(txt_masks)
        if want_l2v:
            out['l2v'] = self._lang2visn(x_in, txt, tmask, B, L, G, P, r_l, blocks.mask_u8(gmap_masks), blocks.mask_u8(vp_masks))
            return out
        # the 4 graph-aware cross-modal layers; context = the instruction (no imagination tokens in pre-training)
        ctx = blocks.operand(txt.reshape(B * L, HID), lowp)
        affine = dist = None
        if ge.sprel_linear is not None:
            affine, dist = pk['sprel'].get(), to(batch['gmap_pair_dists'], F32).contiguous()
        streams = [blocks.Stream(0, B, G, blocks.mask_u8(gmap_masks), 0, dist, affine),
                   blocks.Stream(r_l, B, P, blocks.mask_u8(vp_masks), 1)]
        x, e = x_in, ends
        for cp, sp in zip(pk['x_cross'], pk['x_self']):
            w, b = cp.kv.get(lowp)
            kv = ops.gemm(ctx, w, b)                             # [B*L, 4*768] = K_g | V_g | K_l | V_l
            x = blocks.cross_attn(x, kv, [0, 2 * HID], L, tmask, cp, streams, e, lowp, defer=True)
            x = blocks.self_attn_ffn(x, sp, streams, e, lowp, defer=True)
        out['x'] = blocks.materialize(x, lowp, e)
        return out

    def _lang2visn(self, x_in, txt, tmask, B, L, G, P, r_l, gmask, vmask):
        """GraphLXRTXLayer.forward_lang2visn x 4 for both branches (vilmodel.py:400-411, 719-735): the instruction attends to
        the (fixed) map / panorama input embeddings; two language streams (global | local weights) stacked along the rows."""
        blocks, duet, ops, params = _lazy()
        bert = self.bert
        lowp, pk = bert.lowp, bert._pk()
        HID = 768
        dev = txt.device
        (r0, r1), ends, R = blocks.stack_layout([B * L, B * L])
        t32 = txt.reshape(B * L, HID).contiguous()
        l32 = torch.zeros((R, HID), dtype=torch.float32, device=dev)
        l32[r0:r0 + B * L] = t32
        l32[r1:r1 + B * L] = t32
        lang = blocks.as_act(l32, lowp)
        streams = [blocks.Stream(r0, B, L, tmask, 0), blocks.Stream(r1, B, L, tmask, 1)]
        vg = x_in.operand(lowp)[0:B * G]
        vl = x_in.operand(lowp)[r_l:r_l + B * P]
        for cp, kvp, sp in zip(pk['x_cross'], pk['l2v_kv'], pk['l2v_self']):
            wg, bg = kvp[0].get(lowp)
            wl, bl = kvp[1].get(lowp)
            kv_g = ops.gemm(vg, wg, bg)                          # [B*G, 1536] = K | V of the map tokens (global weights)
            kv_l = ops.gemm(vl, wl, bl)                          # [B*P, 1536] of the panorama tokens (local weights)
            q = blocks.gemm_act(lang, cp.q, lowp, ends)
            ctx = blocks._ctx_buffer(R, q, streams)
            ops.attention_multi([
                dict(q=streams[0].view(q), k=kv_g[:, :HID], v=kv_g[:, HID:], out=streams[0].view(ctx), B=B, Lq=L, Lk=G, key_mask=gmask),
                dict(q=streams[1].view(q), k=kv_l[:, :HID], v=kv_l[:, HID:], out=streams[1].view(ctx), B=B, Lq=L, Lk=P, key_mask=vmask)])
            lang = blocks.linear_residual_ln(ctx, cp.o, lang, cp.ln, 1e-12, lowp, ends, defer=True)
            lang = blocks.self_attn_ffn(lang, sp, streams, ends, lowp, defer=True)
        lang = blocks.materialize(lang, lowp, ends, want16=False)
        return lang.f32[r0:r0 + B * L], lang.f32[r1:r1 + B * L]

    # -- the same trunk with autograd recording (pre-training) -------------------------------------------------------------
    def _recording(self) -> bool:
        return torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())

    def _trunk_train(self, batch, want_l2v=False):
        """_trunk with autograd recording: the same layer sequence from the differentiable blocks (as duet._navigation_train).
        The gathers of the panorama rows become autograd nodes: the vp-image gather a row gather (adjoint: scatter-add), the
        graph-node aggregation a ragged segment mean (one view row can sit in a visited and an unvisited segment)."""
        blocks, duet, ops, params = _lazy()
        from . import autograd_ops as ag
        bert = self.bert
        lowp, pk = bert.lowp, bert._pk()
        dev = bert.embeddings.LayerNorm.weight.device
        F32, HID = torch.float32, 768
        to = lambda t, dt=None: torch.as_tensor(t).to(dev, dtype=dt, non_blocking=True)     # noqa: E731
        txt_ids = to(batch['txt_ids'])
        B, L = txt_ids.shape
        txt_masks = torch.arange(L, device=dev)[None, :] < to(batch['txt_lens'])[:, None]
        txt = bert.forward_text(txt_ids, txt_masks)
        step_lens = [int(x) for x in batch['traj_step_lens']]
        pano, _ = bert.forward_panorama_per_step(to(batch['traj_view_img_fts'], F32), None, to(batch['traj_loc_fts'], F32),
                                                 to(batch['traj_nav_types']), to(batch['traj_vp_view_lens']), None)
        N, V, _ = pano.shape
        vl_host = [int(x) for x in batch['traj_vp_view_lens']]
        last = np.cumsum(step_lens) - 1
        P = max(vl_host[i] for i in last) + 1
        vp_idx = np.full((B, P), N * V, np.int64)                                       # row N * V: the appended zero row
        for b, i in enumerate(last):
            n = min(V, P - 1)
            vp_idx[b, 1:1 + n] = i * V + np.arange(n)
        vp_lens = torch.as_tensor([vl_host[i] + 1 for i in last], device=dev)
        vp_masks = torch.arange(P, device=dev)[None, :] < vp_lens[:, None]
        off, rows, G = gmap_aggregation_rows(step_lens, vl_host, batch['traj_vpids'], batch['traj_cand_vpids'],
                                             batch['gmap_vpids'], V)
        gmap_masks = torch.arange(G, device=dev)[None, :] < to(batch['gmap_lens'])[:, None]
        le, ge = bert.local_encoder, bert.global_encoder
        with blocks.grad_mode(True, bert._drop()):
            src = torch.cat([pano.reshape(N * V, HID), torch.zeros((1, HID), dtype=F32, device=dev)], 0)
            vp_img = ag.GatherRowsFn.apply(src, torch.from_numpy(vp_idx.reshape(-1)).to(dev), 0, B * P)
            gmap_img = ag.RaggedMeanFn.apply(src, torch.from_numpy(off).to(dev), torch.from_numpy(rows).to(dev), B * G)
            (r_g, r_l), ends, R = blocks.stack_layout([B * G, B * P])
            g_in = blocks.embed(B * G, dev, a=gmap_img, feat=to(batch['gmap_pos_fts'], F32).reshape(B * G, -1).contiguous(),
                                feat_lin=ge.gmap_pos_embeddings[0], feat_ln=ge.gmap_pos_embeddings[1],
                                idx=to(batch['gmap_step_ids']).long().contiguous().view(-1), table=ge.gmap_step_embeddings.weight).f32
            l_in = blocks.embed(B * P, dev, a=vp_img, feat=to(batch['vp_pos_fts'], F32).reshape(B * P, -1).contiguous(),
                                feat_lin=le.vp_pos_embeddings[0], feat_ln=le.vp_pos_embeddings[1]).f32
            parts = [g_in] + ([torch.zeros((r_l - B * G, HID), dtype=F32, device=dev)] if r_l > B * G else []) + [l_in]
            x = blocks.as_act(torch.cat(parts, 0), lowp)
            out = dict(B=B, L=L, G=G, P=P, r_l=r_l, ends=ends, dev=dev, last=last)
            tmask = blocks.mask_u8(txt_masks)
            if want_l2v:
                out['l2v'] = self._lang2visn_train(x, txt, tmask, B, L, G, P, r_l, blocks.mask_u8(gmap_masks), blocks.mask_u8(vp_masks))
                return out
            ctx = blocks.operand(txt.reshape(B * L, HID), lowp)
            affine = dist = aparams = None
            if ge.sprel_linear is not None:
                affine, dist = pk['sprel'].get(), to(batch['gmap_pair_dists'], F32).contiguous()
                aparams = (ge.sprel_linear.weight, ge.sprel_linear.bias)
            streams = [blocks.Stream(r_g, B, G, blocks.mask_u8(gmap_masks), 0, dist, affine, aparams),
                       blocks.Stream(r_l, B, P, blocks.mask_u8(vp_masks), 1)]
            for cp, sp in zip(pk['x_cross'], pk['x_self']):
                kv = blocks.linear(ctx, cp.kv, lowp)                # [B*L, 4*768] = K_g | V_g | K_l | V_l
                x = blocks.cross_attn(x, kv, [0, 2 * HID], L, tmask, cp, streams, ends, lowp)
                x = blocks.self_attn_ffn(x, sp, streams, ends, lowp)
            out['x'] = x
        return out

    def _lang2visn_train(self, x_in, txt, tmask, B, L, G, P, r_l, gmask, vmask):
        """_lang2visn with autograd recording.  Both language streams start from the same text rows, so their gradients sum
        back into the text encoder; both attention problems (text -> map, text -> panorama) run as one AttentionFn node."""
        blocks, duet, ops, params = _lazy()
        from . import autograd_ops as ag
        bert = self.bert
        lowp, pk = bert.lowp, bert._pk()
        HID = 768
        dev = txt.device
        (r0, r1), ends, R = blocks.stack_layout([B * L, B * L])
        t32 = txt.reshape(B * L, HID)
        parts = [t32] + ([torch.zeros((r1 - B * L, HID), dtype=torch.float32, device=dev)] if r1 > B * L else []) + [t32]
        lang = blocks.as_act(torch.cat(parts, 0), lowp)
        streams = [blocks.Stream(r0, B, L, tmask, 0), blocks.Stream(r1, B, L, tmask, 1)]
        vg = x_in.operand(lowp)[0:B * G]
        vl = x_in.operand(lowp)[r_l:r_l + B * P]
        for cp, kvp, sp in zip(pk['x_cross'], pk['l2v_kv'], pk['l2v_self']):
            kv_g = blocks.linear(vg, kvp[0], lowp)                  # [B*G, 1536] = K | V of the map tokens (global weights)
            kv_l = blocks.linear(vl, kvp[1], lowp)                  # [B*P, 1536] of the panorama tokens (local weights)
            q = blocks.linear(lang.operand(lowp), cp.q, lowp, ends=ends)
            spec = [dict(q=(0, r0, 0), k=(1, 0, 0), v=(1, 0, HID), B=B, Lq=L, Lk=G, key_mask=gmask, out_row0=r0,
                         drop=blocks._attn_drop(dev)),
                    dict(q=(0, r1, 0), k=(2, 0, 0), v=(2, 0, HID), B=B, Lq=L, Lk=P, key_mask=vmask, out_row0=r1,
                         drop=blocks._attn_drop(dev))]
            ctx = ag.AttentionFn.apply(spec, R, ops.MASK_ADD_NEG10000, 3, q, kv_g, kv_l)
            lang = blocks._dense_res_ln(ctx, cp.o, lang.f32, cp.ln, 1e-12, lowp, ends)
            lang = blocks.self_attn_ffn(lang, sp, streams, ends, lowp)
        return lang.f32[r0:r0 + B * L], lang.f32[r1:r1 + B * L]

    def _head_train(self, h32, lin, act, ln, dec, lowp):
        """Linear -> act -> LayerNorm(1e-12) -> padded Linear with autograd recording -> (scores, gradient handle)"""
        blocks, duet, ops, params = _lazy()
        from . import autograd_ops as ag
        with blocks.grad_mode(True, self.bert._drop()):
            hidden = ag.ActFn.apply(blocks.linear(blocks.operand(h32, lowp), lin, lowp, out_dtype=torch.float32), act)
            y = blocks.layer_norm(hidden, None, ln, 1e-12, lowp)
            return ag.padded_linear(y.operand(lowp), dec, lowp)

    # -- tasks -----------------------------------------------------------------------------------------------------------
    def forward(self, batch, task, compute_loss=True):
        """With autograd recording (parameters that require grad, grad mode on) every step records a node whose forward and
        backward are libvlnimagine kernels; ``compute_loss=True`` returns the per-row losses the reference's trainer averages.
        Under torch.no_grad() the inference path runs."""
        blocks, duet, ops, params = _lazy()
        with ops.half_format(self.bert.h16_format()):
            if task.startswith('mlm'):
                return self.forward_mlm(batch, compute_loss)
            if task.startswith('mrc'):
                return self.forward_mrc(batch, compute_loss)
            if task.startswith('sap'):
                return self.forward_sap(batch, compute_loss)
            raise ValueError('invalid task %r (the R2R recipe has mlm, mrc, sap)' % task)

    def forward_mlm(self, batch, compute_loss=True):
        """pretrain_cmt.py:128-150: prediction scores [n_masked, vocab] (or the per-token cross-entropy)"""
        blocks, duet, ops, params = _lazy()
        if self._recording():
            return self._mlm_train(batch, compute_loss)
        t = self._trunk(batch, want_l2v=True)
        lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
        gt, vt = t['l2v']
        labels = torch.as_tensor(batch['txt_labels'])
        pos = torch.nonzero(labels.reshape(-1) != -1).flatten()
        n = int(pos.numel())
        idx = pos.to(torch.int32).to(dev)
        unit = torch.arange(n + 1, dtype=torch.int32, device=dev)
        a, _ = ops.gather_mean(gt, unit, idx, n, want16=False)
        b, _ = ops.gather_mean(vt, unit, idx, n, want16=False)
        h32, h16 = ops.embed_compose(n, dev, a=a, a2=b, want16=lowp)               # (global + local) text states of the masked tokens
        w, bias = hp['mlm_t'].get(lowp)
        hidden = ops.gemm(h16 if lowp else h32, w, bias, epilogue=ops.EPI_GELU, out_dtype=torch.float32)
        pr = self.mlm_head.predictions
        y32, y16 = ops.add_ln(hidden, None, pr.transform.LayerNorm.weight, pr.transform.LayerNorm.bias, 1e-12, want16=lowp)
        w, bias, vocab = hp['mlm_dec'].get(lowp)
        scores = ops.gemm(y16 if lowp else y32, w, bias, out_dtype=torch.float32)   # [n, 30528]: the padded tail is never read
        if compute_loss:
            return ops.ce_rows(scores, labels.reshape(-1)[pos].to(dev), vocab)
        return scores[:, :vocab]

    def forward_mrc(self, batch, compute_loss=True):
        """pretrain_cmt.py:158-204 (views only): soft-label classification of the masked views of the last panorama"""
        blocks, duet, ops, params = _lazy()
        if self._recording():
            return self._mrc_train(batch, compute_loss)
        t = self._trunk(batch)          # the global branch is independent of the local one: running both changes nothing
        lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
        B, P, r_l = t['B'], t['P'], t['r_l']
        masks = torch.as_tensor(batch['vp_view_mrc_masks'])
        bi, vi = torch.nonzero(masks, as_tuple=True)
        rows = (r_l + bi * P + 1 + vi).to(torch.int32).to(dev)                      # token 0 of every episode is [stop]
        n = int(rows.numel())
        unit = torch.arange(n + 1, dtype=torch.int32, device=dev)
        h32, h16 = ops.gather_mean(t['x'].f32, unit, rows, n, want16=lowp, want32=not lowp)
        w, bias = hp['mrc0'].get(lowp)
        hidden = ops.gemm(h16 if lowp else h32, w, bias, epilogue=ops.EPI_RELU, out_dtype=torch.float32)
        net = self.image_classifier.net
        y32, y16 = ops.add_ln(hidden, None, net[2].weight, net[2].bias, 1e-12, want16=lowp)
        w, bias, n_cls = hp['mrc3'].get(lowp)
        logits = ops.gemm(y16 if lowp else y32, w, bias, out_dtype=torch.float32)
        targets = torch.as_tensor(batch['vp_view_probs'])[masks].to(dev, torch.float32).contiguous()
        if compute_loss:
            return ops.kl_rows(logits, targets, n_cls)
        return logits[:, :n_cls], targets

    def forward_sap(self, batch, compute_loss=True):
        """pretrain_cmt.py:206-262: global / local / fused action logits (or the three summed cross-entropies)"""
        blocks, duet, ops, params = _lazy()
        if self._recording():
            return self._sap_train(batch, compute_loss)
        t = self._trunk(batch)
        lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
        B, G, P, r_l, ends, x = t['B'], t['G'], t['P'], t['r_l'], t['ends'], t['x']
        fuse_raw = None
        if 'fuse' in hp:
            cat = torch.empty((B, 2 * 768), dtype=ops.h16() if lowp else torch.float32, device=dev)
            c32, c16 = (None, cat) if lowp else (cat, None)
            ops.copy_rows(x.f32, G * 768, 768, B, 1, c32, c16, 2 * 768, 768)
            ops.copy_rows(x.f32[r_l:], P * 768, 768, B, 1, c32[:, 768:] if c32 is not None else None,
                          c16[:, 768:] if c16 is not None else None, 2 * 768, 768)
            fuse_raw = blocks.cls_head(cat, hp['fuse'], lowp)
        raw = blocks.cls_head(x.operand(lowp), hp['sap'], lowp, ends)
        gmap_masks = torch.arange(G, device=dev)[None, :] < torch.as_tensor(batch['gmap_lens']).to(dev)[:, None]
        visited = torch.as_tensor(batch['gmap_visited_masks']).to(dev)
        last = t['last']
        nav_types = torch.as_tensor(batch['traj_nav_types'])[torch.as_tensor(last)]
        nav = torch.zeros((B, P), dtype=torch.bool)
        nav[:, 0] = True                                        # [stop] is always admissible (pretrain_cmt.py:231-236)
        nav[:, 1:] = nav_types[:, :P - 1] == 1
        cand = [[None] + list(c[-1]) for c in batch['traj_cand_vpids']]
        gmap_ids, cand_ids = self.bert.intern_vpids(batch['gmap_vpids'], cand, G, P, dev)
        gl, ll, fl = ops.duet_fuse_logits(raw[0:], raw[r_l:], fuse_raw, blocks.mask_u8(gmap_masks), blocks.mask_u8(visited),
                                          blocks.mask_u8(nav.to(dev)), gmap_ids, cand_ids, B, G, P)
        if compute_loss:
            ga = torch.as_tensor(batch['global_act_labels']).to(dev)
            la = torch.as_tensor(batch['local_act_labels']).to(dev)
            return ops.ce_rows(gl, ga, G) + ops.ce_rows(ll, la, P) + ops.ce_rows(fl, ga, G)
        return gl, ll, fl

    def _sap_masks(self, batch, t):
        """(gmap masks, visited masks, navigable masks of the local tokens, gmap ids, candidate ids) of forward_sap"""
        B, G, P, dev = t['B'], t['G'], t['P'], t['dev']
        gmap_masks = torch.arange(G, device=dev)[None, :] < torch.as_tensor(batch['gmap_lens']).to(dev)[:, None]
        visited = torch.as_tensor(batch['gmap_visited_masks']).to(dev)
        nav_types = torch.as_tensor(batch['traj_nav_types'])[torch.as_tensor(t['last'])]
        nav = torch.zeros((B, P), dtype=torch.bool)
        nav[:, 0] = True                                        # [stop] is always admissible (pretrain_cmt.py:231-236)
        nav[:, 1:] = nav_types[:, :P - 1] == 1
        cand = [[None] + list(c[-1]) for c in batch['traj_cand_vpids']]
        gmap_ids, cand_ids = self.bert.intern_vpids(batch['gmap_vpids'], cand, G, P, dev)
        return gmap_masks, visited, nav.to(dev), gmap_ids, cand_ids

    def _mlm_train(self, batch, compute_loss):
        blocks, duet, ops, params = _lazy()
        from . import autograd_ops as ag
        t = self._trunk_train(batch, want_l2v=True)
        lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
        gt, vt = t['l2v']
        labels = torch.as_tensor(batch['txt_labels'])
        pos = torch.nonzero(labels.reshape(-1) != -1).flatten()
        n = int(pos.numel())
        idx = pos.to(dev)
        with blocks.grad_mode(True, self.bert._drop()):
            h = ag.SumRowsFn.apply(2, ag.GatherRowsFn.apply(gt, idx, 0, n), ag.GatherRowsFn.apply(vt, idx, 0, n))
        scores, handle = self._head_train(h, hp['mlm_t'], ops.EPI_GELU, hp['mlm_ln'], hp['mlm_dec'], lowp)
        vocab = hp['mlm_dec'].n
        if compute_loss:
            return ag.CERowsFn.apply(scores, handle, labels.reshape(-1)[pos].to(dev), vocab)
        return scores[:, :vocab]

    def _mrc_train(self, batch, compute_loss):
        blocks, duet, ops, params = _lazy()
        from . import autograd_ops as ag
        t = self._trunk_train(batch)
        lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
        B, P, r_l = t['B'], t['P'], t['r_l']
        masks = torch.as_tensor(batch['vp_view_mrc_masks'])
        bi, vi = torch.nonzero(masks, as_tuple=True)
        rows = (r_l + bi * P + 1 + vi).to(dev)
        with blocks.grad_mode(True, self.bert._drop()):
            h = ag.GatherRowsFn.apply(t['x'].f32, rows, 0, int(rows.numel()))
        logits, handle = self._head_train(h, hp['mrc0'], ops.EPI_RELU, hp['mrc_ln'], hp['mrc3'], lowp)
        n_cls = hp['mrc3'].n
        targets = torch.as_tensor(batch['vp_view_probs'])[masks].to(dev, torch.float32).contiguous()
        if compute_loss:
            return ag.KLRowsFn.apply(logits, handle, targets, n_cls)
        return logits[:, :n_cls], targets

    def _sap_train(self, batch, compute_loss):
        blocks, duet, ops, params = _lazy()
        from . import autograd_ops as ag
        t = self._trunk_train(batch)
        lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
        B, G, P, r_l, ends, x = t['B'], t['G'], t['P'], t['r_l'], t['ends'], t['x']
        gmap_masks, visited, nav, gmap_ids, cand_ids = self._sap_masks(batch, t)
        with blocks.grad_mode(True, self.bert._drop()):
            fuse_raw = None
            if 'fuse' in hp:
                cat = torch.cat([x.f32[0:B * G].view(B, G, 768)[:, 0], x.f32[r_l:r_l + B * P].view(B, P, 768)[:, 0]], 1)
                fuse_raw = blocks.cls_head(blocks.operand(cat, lowp), hp['fuse'], lowp)
            raw = blocks.cls_head(x.operand(lowp), hp['sap'], lowp, ends)
            gl, ll, fl = ag.FuseLogitsFn.apply(raw[0:B * G], raw[r_l:r_l + B * P], fuse_raw, blocks.mask_u8(gmap_masks),
                                               blocks.mask_u8(visited), blocks.mask_u8(nav), gmap_ids, cand_ids, B, G, P)
        if compute_loss:
            ga = torch.as_tensor(batch['global_act_labels']).to(dev)
            la = torch.as_tensor(batch['local_act_labels']).to(dev)
            return ag.CERowsFn.apply(gl, gl, ga, G) + ag.CERowsFn.apply(ll, ll, la, P) + ag.CERowsFn.apply(fl, fl, ga, G)
        return gl, ll, fl


class _PaddedLinear:
    """A [N, 768] weight (+ bias) padded with zero rows for the tensor-core tiles, rebuilt when the parameters change.
    Inference pads the output width to a multiple of 64 (the MLM decoder: 30522 -> 30528; the MRC classifier: 1000 -> 1024);
    training to a multiple of 128 (30592 / 1024), the column granule of the weight-gradient kernel vi_wgrad16.  Also the pack
    of autograd_ops.PaddedLinearFn (weights / biases / grad_sources / get_t as blocks.LinearPack)."""

    def __init__(self, weight, bias):
        blocks, duet, ops, params = _lazy()
        self.n = weight.shape[0]
        self.weight, self.bias = weight, bias
        self.weights, self.biases = [weight], ([bias] if bias is not None else None)
        self._pack = blocks.Pack([weight] + ([bias] if bias is not None else []), self._make)

    def _padded(self, v, align):
        key = ('pad', align)
        if key not in v:
            n_pad = (self.n + align - 1) // align * align
            w = torch.zeros((n_pad, self.weight.shape[1]), dtype=torch.float32, device=self.weight.device)
            w[:self.n] = self.weight.detach()
            b = torch.zeros((n_pad,), dtype=torch.float32, device=self.weight.device)
            if self.bias is not None:
                b[:self.n] = self.bias.detach()
            v[key] = {'w32': w, 'b': b}
        return v[key]

    def _make(self):
        return {}

    def _get(self, lowp: bool, align: int, fmt=None):
        blocks, duet, ops, params = _lazy()
        v = self._padded(self._pack.get(), align)
        if not lowp:
            return v['w32'], v['b']
        key = ('w16', fmt or ops.h16())
        if key not in v:
            v[key] = ops.cast_h16(v['w32'], dtype=key[1])
        return v[key], v['b']

    def get(self, lowp: bool):
        """(weight, bias, n) of the inference GEMM"""
        w, b = self._get(lowp, 64)
        return w, b, self.n

    def get_train(self, lowp: bool):
        """(weight, bias) of the training GEMM: bf16 shadow or fp32, padded to a multiple of 128 rows"""
        blocks, duet, ops, params = _lazy()
        return self._get(lowp, 128, ops.BF16)

    def get_t(self, lowp: bool, n_groups: int = 1):
        """the transposed training weight [768, n_pad] (B operand of the input-gradient GEMM), cached with the pack"""
        from .autograd_ops import transpose
        v = self._padded(self._pack.get(), 128)
        key = ('t', lowp)
        if key not in v:
            with torch.no_grad():
                v[key] = transpose(self.get_train(lowp)[0])
        return v[key]

    def grad_sources(self):
        return self.weights + (self.biases or [])
