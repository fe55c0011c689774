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

One code path serves inference and training.  Each task runs its layer sequence from the mode-switching blocks (blocks.py) and
the navigation model's pieces (duet.GlocalTextPathNavCMT._branch_inputs / _cross_layers / _sap_heads / _fuse_step) under
``blocks.grad_mode``: under torch.no_grad() they are plain libvlnimagine launches; with autograd recording (grad mode on,
parameters that require grad) every step records a node whose backward is libvlnimagine kernels too, and ``forward`` returns the
per-row losses for ``loss.mean().backward()``.  In training the padded decoder / classifier is ``autograd_ops.PaddedLinearFn``
(the tied decoder's weight gradient adds onto the word-embedding lookup's), the losses ``CERowsFn`` / ``KLRowsFn``, whose backward
kernel (vi_ce_rows_bwd / vi_kl_rows_bwd) writes the bf16 operand of the decoder's gradient GEMMs directly.  Train-mode dropout:
bf16 only, as the navigation model.
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
    def _recording(self) -> bool:
        return torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())

    def _trunk(self, batch, want_l2v=False):
        """GlocalTextPathCMT.forward / forward_mlm, model/vilmodel.py:660-747 -> dict of row-stacked results.  In training the
        gathers of the panorama rows are autograd nodes: the vp-image gather a row gather (adjoint: scatter-add), the graph-node
        aggregation a ragged segment mean (one view row can sit in a visited and an unvisited segment)."""
        blocks, duet, ops, params = _lazy()
        bert = self.bert
        lowp = bert.lowp
        dev = bert.embeddings.LayerNorm.weight.device
        F32, HID = torch.float32, 768
        to = lambda t, dt=None: torch.as_tensor(t).to(dev, dtype=dt, non_blocking=True)     # noqa: E731
        txt_ids = to(batch['txt_ids'])
        B, L = txt_ids.shape
        txt_masks = torch.arange(L, device=dev)[None, :] < to(batch['txt_lens'])[:, None]
        txt = bert.forward_text(txt_ids, txt_masks)                                  # (B, L, 768) fp32
        # every panorama of every trajectory through the panorama encoder (vilmodel.py:484-528)
        step_lens = [int(x) for x in batch['traj_step_lens']]
        pano, _ = bert.forward_panorama_per_step(to(batch['traj_view_img_fts'], F32), None, to(batch['traj_loc_fts'], F32),
                                                 to(batch['traj_nav_types']), to(batch['traj_vp_view_lens']), None)
        N, V, _ = pano.shape
        vl_host = [int(x) for x in batch['traj_vp_view_lens']]
        last = np.cumsum(step_lens) - 1
        # local branch: [stop] + the LAST panorama of each trajectory (vilmodel.py:538-553)
        P = max(vl_host[i] for i in last) + 1
        vp_idx = np.full((B, P), N * V, np.int64)                                       # row N * V: the appended zero row
        for b, i in enumerate(last):
            n = min(V, P - 1)
            vp_idx[b, 1:1 + n] = i * V + np.arange(n)
        vp_lens = torch.as_tensor([vl_host[i] + 1 for i in last], device=dev)
        vp_masks = torch.arange(P, device=dev)[None, :] < vp_lens[:, None]
        # global branch: the graph-node features aggregated from the trajectory (vilmodel.py:577-611) in one segment mean
        off, rows, G = gmap_aggregation_rows(step_lens, vl_host, batch['traj_vpids'], batch['traj_cand_vpids'],
                                             batch['gmap_vpids'], V)
        gmap_masks = torch.arange(G, device=dev)[None, :] < to(batch['gmap_lens'])[:, None]
        src = torch.cat([pano.reshape(N * V, HID), torch.zeros((1, HID), dtype=F32, device=dev)], 0)
        vp_img = blocks.gather_rows(src, vp_idx.reshape(-1), B * P)
        gmap_img = blocks.segment_mean(src, off, rows, B * G)
        # input embeddings of both branches into one row-stacked activation (vilmodel.py:613-625, 538-553)
        x, row0, ends = bert._branch_inputs(gmap_img, to(batch['gmap_pos_fts'], F32), to(batch['gmap_step_ids']), vp_img,
                                            to(batch['vp_pos_fts'], F32), B, G, P)
        out = dict(B=B, L=L, G=G, P=P, r_l=row0[1], ends=ends, dev=dev, last=last)
        tmask = blocks.mask_u8(txt_masks)
        if want_l2v:
            out['l2v'] = self._lang2visn(x, txt, tmask, B, L, G, P, row0[1], blocks.mask_u8(gmap_masks), blocks.mask_u8(vp_masks))
            return out
        # the 4 graph-aware cross-modal layers; context = the instruction (no imagination tokens in pre-training)
        streams = bert._branch_streams(B, G, P, row0, gmap_masks, vp_masks, to(batch['gmap_pair_dists'], F32))
        out['x'] = bert._cross_layers(x, streams, ends, L, tmask, ctx=blocks.operand(txt.reshape(B * L, HID), lowp))
        return out

    def _lang2visn(self, x_in, txt, tmask, B, L, G, P, r_l, gmask, vmask):
        """GraphLXRTXLayer.forward_lang2visn x 4 for both branches (vilmodel.py:400-411, 719-735): the instruction attends to
        the (fixed) map / panorama input embeddings; two language streams (global | local weights) stacked along the rows.  In
        training both start from the same text rows, so their gradients sum back into the text encoder."""
        blocks, duet, ops, params = _lazy()
        bert = self.bert
        lowp, pk = bert.lowp, bert._pk()
        row0, ends, R = blocks.stack_layout([B * L, B * L])
        t32 = txt.reshape(B * L, 768)
        lang = blocks.as_act(blocks.stack_rows([t32, t32], row0), lowp)
        streams = [blocks.Stream(row0[0], B, L, tmask, 0), blocks.Stream(row0[1], B, L, tmask, 1)]
        vg = x_in.operand(lowp)[0:B * G]
        vl = x_in.operand(lowp)[r_l:r_l + B * P]
        for cp, kvp, sp in zip(pk['x_cross'], pk['l2v_kv'], pk['l2v_self']):
            kv_g = blocks.linear(vg, kvp[0], lowp)               # [B*G, 1536] = K | V of the map tokens (global weights)
            kv_l = blocks.linear(vl, kvp[1], lowp)               # [B*P, 1536] of the panorama tokens (local weights)
            lang = blocks.cross_attn(lang, [(kv_g, 0, G, gmask), (kv_l, 0, P, vmask)], cp, streams, ends, lowp, defer=True)
            lang = blocks.self_attn_ffn(lang, sp, streams, ends, lowp, defer=True)
        lang = blocks.materialize(lang, lowp, ends, want16=False)
        return lang.f32[row0[0]:row0[0] + B * L], lang.f32[row0[1]:row0[1] + B * L]

    def _head(self, x, lin, act, ln, dec):
        """GEMM operand -> Linear -> act -> LayerNorm(1e-12) -> padded Linear -> (scores [rows, n_pad], gradient handle)"""
        blocks, duet, ops, params = _lazy()
        lowp = self.bert.lowp
        y = blocks.layer_norm(blocks.linear(x, lin, lowp, out_dtype=torch.float32, epilogue=act), None, ln, 1e-12, lowp)
        return dec(y.operand(lowp), lowp)

    @staticmethod
    def _row_loss(kl, logits, handle, target, n_cols):
        """per-row KL (soft targets) or cross-entropy (labels) over the first n_cols columns.  Training: the loss node sends the
        logits' gradient to ``handle`` (PaddedLinearFn's, or the logits themselves when None)."""
        blocks, duet, ops, params = _lazy()
        if blocks.training():
            from . import autograd_ops as ag
            fn = ag.KLRowsFn if kl else ag.CERowsFn
            return fn.apply(logits, logits if handle is None else handle, target, n_cols)
        return (ops.kl_rows if kl else ops.ce_rows)(logits, target, n_cols)

    # -- tasks -----------------------------------------------------------------------------------------------------------
    def forward(self, batch, task, compute_loss=True):
        """With autograd recording (parameters that require grad, grad mode on) every step records a node whose forward and
        backward are libvlnimagine kernels; ``compute_loss=True`` returns the per-row losses the reference's trainer averages.
        Under torch.no_grad() the same steps run as plain launches."""
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
        with blocks.grad_mode(self._recording(), self.bert._drop()):
            t = self._trunk(batch, want_l2v=True)
            lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
            gt, vt = t['l2v']
            labels = torch.as_tensor(batch['txt_labels'])
            pos = torch.nonzero(labels.reshape(-1) != -1).flatten()
            n = int(pos.numel())
            h = blocks.embed(n, dev, a=blocks.gather_rows(gt, pos, n), a2=blocks.gather_rows(vt, pos, n), lowp=lowp)
            scores, handle = self._head(h.operand(lowp), hp['mlm_t'], ops.EPI_GELU, hp['mlm_ln'], hp['mlm_dec'])
            vocab = hp['mlm_dec'].n                     # the padded tail columns are never read
            if compute_loss:
                return self._row_loss(False, scores, handle, labels.reshape(-1)[pos].to(dev), vocab)
            return scores[:, :vocab]

    def forward_mrc(self, batch, compute_loss=True):
        """pretrain_cmt.py:158-204 (views only): soft-label classification of the masked views of the last panorama"""
        blocks, duet, ops, params = _lazy()
        with blocks.grad_mode(self._recording(), self.bert._drop()):
            t = self._trunk(batch)      # the global branch is independent of the local one: running both changes nothing
            lowp, dev, hp = self.bert.lowp, t['dev'], self._hp()
            P, r_l = t['P'], t['r_l']
            masks = torch.as_tensor(batch['vp_view_mrc_masks'])
            bi, vi = torch.nonzero(masks, as_tuple=True)
            rows = r_l + bi * P + 1 + vi                                            # token 0 of every episode is [stop]
            h = blocks.gather_rows(t['x'].f32, rows, int(rows.numel()), lowp=lowp)
            logits, handle = self._head(h, hp['mrc0'], ops.EPI_RELU, hp['mrc_ln'], hp['mrc3'])
            n_cls = hp['mrc3'].n
            targets = torch.as_tensor(batch['vp_view_probs'])[masks].to(dev, torch.float32).contiguous()
            if compute_loss:
                return self._row_loss(True, logits, handle, targets, n_cls)
            return logits[:, :n_cls], targets

    def forward_sap(self, batch, compute_loss=True):
        """pretrain_cmt.py:206-262: global / local / fused action logits (or the three summed cross-entropies)"""
        blocks, duet, ops, params = _lazy()
        with blocks.grad_mode(self._recording(), self.bert._drop()):
            t = self._trunk(batch)
            dev, hp = t['dev'], self._hp()
            B, G, P, row0 = t['B'], t['G'], t['P'], (0, t['r_l'])
            raw, fuse_raw = self.bert._sap_heads(t['x'], hp['sap'], hp.get('fuse'), B, G, P, row0, t['ends'])
            gl, ll, fl = self.bert._fuse_step(raw, fuse_raw, *self._sap_masks(batch, t), B, G, P, row0)
            if compute_loss:
                ga = torch.as_tensor(batch['global_act_labels']).to(dev)
                la = torch.as_tensor(batch['local_act_labels']).to(dev)
                return (self._row_loss(False, gl, None, ga, G) + self._row_loss(False, ll, None, la, P)
                        + self._row_loss(False, fl, None, ga, G))
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

    def __call__(self, x, lowp: bool):
        """x W^T + b -> (fp32 scores [rows, n_pad], gradient handle).  Training: autograd_ops.PaddedLinearFn over the
        128-padded weight.  Inference: one GEMM over the 64-padded weight (handle None)."""
        blocks, duet, ops, params = _lazy()
        if blocks.training():
            from .autograd_ops import padded_linear
            return padded_linear(x, self, lowp)
        w, b = self._get(lowp, 64)
        return ops.gemm(x, w, b, out_dtype=torch.float32), None

    def get_train(self, lowp: bool):
        """(weight, bias) of the training GEMM: bf16 shadow or fp32, padded to a multiple of 128 rows"""
        blocks, duet, ops, params = _lazy()
        return self._get(lowp, 128, ops.BF16)

    def get_t(self, lowp: bool, n_groups: int = 1):
        """the transposed training weight [768, n_pad] (B operand of the input-gradient GEMM), cached with the pack"""
        blocks, duet, ops, params = _lazy()
        v = self._padded(self._pack.get(), 128)
        key = ('t', lowp)
        if key not in v:
            with torch.no_grad():
                v[key] = ops.transpose(self.get_train(lowp)[0])
        return v[key]

    def grad_sources(self):
        return self.weights + (self.biases or [])
