"""TEST INFRASTRUCTURE - CPU oracle for the DUET pre-training forward (SURVEY.md section 8(f), row N4).

Functional fp32 restatement of VLN-DUET/pretrain_src/model/{vilmodel.py, pretrain_cmt.py} on top of the building blocks of
duet_oracle.py (the blocks are the same classes as in map_nav_src): whole trajectories are embedded at once, the graph-node
features are aggregated from them (``_aggregate_gmap_features``), and the three proxy tasks of the R2R recipe
(config/r2r_pretrain.json: mlm, mrc, sap) put their heads on top.  Paths below are relative to VLN-DUET/pretrain_src/.
Pinned to the real reference by ``oracle/gen_golden.py --model duet_pretrain`` (tests/golden/duet_pretrain.npz).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .duet_oracle import (bert_attention, bert_ffn, cls_prediction, cross_attention, crossmodal_encoder, forward_panorama,
                          forward_text, fuse_logits, gelu_erf, lin, lnorm, neg_mask)


def _sub(sd, prefix='bert.'):
    """the GlocalTextPathCMT tensors of the pre-training state dict under the names duet_oracle.py expects"""
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


def seq_masks(lens, width=None):
    width = int(max(lens)) if width is None else width
    return torch.arange(width)[None, :] < torch.as_tensor(lens)[:, None]


def trajectory_embeddings(bsd, ep):
    """ImageEmbeddings.forward, model/vilmodel.py:484-528: every panorama of every trajectory through the panorama encoder
    (R2R: no object features), split back per trajectory."""
    x, _ = forward_panorama(bsd, ep['traj_view_img_fts'], ep['traj_loc_fts'], ep['traj_nav_types'], ep['traj_vp_view_lens'])
    steps = list(ep['traj_step_lens'])
    return torch.split(x, steps, 0), torch.split(ep['traj_vp_view_lens'], steps, 0)


def aggregate_gmap_features(split_embeds, split_lens, traj_vpids, traj_cand_vpids, gmap_vpids):
    """GlobalMapEncoder._aggregate_gmap_features, model/vilmodel.py:577-611: a visited viewpoint = masked mean of its (last)
    panorama; an unvisited one = mean of the candidate views that pointed at it; [stop] = 0; zero padded."""
    rows = []
    for i in range(len(split_embeds)):
        visited, unvisited = {}, {}
        m = seq_masks(split_lens[i])
        e = split_embeds[i][:, :m.shape[1]] * m.unsqueeze(2)
        for t in range(e.shape[0]):
            visited[traj_vpids[i][t]] = e[t].sum(0) / split_lens[i][t]
            for j, vp in enumerate(traj_cand_vpids[i][t]):
                if vp not in visited:
                    unvisited.setdefault(vp, []).append(e[t][j])
        rows.append(torch.stack([visited[vp] if vp in visited else torch.stack(unvisited[vp], 0).mean(0)
                                 for vp in gmap_vpids[i][1:]], 0))
    G = max(r.shape[0] for r in rows) + 1
    out = torch.zeros(len(rows), G, rows[0].shape[1])
    for i, r in enumerate(rows):
        out[i, 1:1 + r.shape[0]] = r
    return out


def gmap_input_embedding(bsd, ep, split_embeds, split_lens):
    """model/vilmodel.py:613-625"""
    g = 'global_encoder'
    img = aggregate_gmap_features(split_embeds, split_lens, ep['traj_vpids'], ep['traj_cand_vpids'], ep['gmap_vpids'])
    e = (img + F.embedding(ep['gmap_step_ids'], bsd[g + '.gmap_step_embeddings.weight'])
         + lnorm(bsd, g + '.gmap_pos_embeddings.1', lin(bsd, g + '.gmap_pos_embeddings.0', ep['gmap_pos_fts']), 1e-12))
    return e, seq_masks(ep['gmap_lens'], e.shape[1])


def vp_input_embedding(bsd, ep, split_embeds, split_lens):
    """LocalVPEncoder.vp_input_embedding, model/vilmodel.py:538-553: [stop] + the LAST panorama of the trajectory"""
    lens = torch.stack([x[-1] + 1 for x in split_lens], 0)
    P = int(lens.max())
    B, H = len(split_embeds), split_embeds[0].shape[-1]
    img = torch.zeros(B, P, H)
    for i, x in enumerate(split_embeds):
        img[i, 1:] = x[-1][:P - 1]
    l = 'local_encoder'
    e = img + lnorm(bsd, l + '.vp_pos_embeddings.1', lin(bsd, l + '.vp_pos_embeddings.0', ep['vp_pos_fts']), 1e-12)
    return e, seq_masks(lens, P)


def forward_bert(sd, ep, return_gmap=True):
    """GlocalTextPathCMT.forward, model/vilmodel.py:660-698 -> (gmap_embeds or None, vp_embeds, txt_embeds, txt_masks)"""
    bsd = _sub(sd)
    txt_masks = seq_masks(ep['txt_lens'], ep['txt_ids'].shape[1])
    txt = forward_text(bsd, ep['txt_ids'], txt_masks)
    split_embeds, split_lens = trajectory_embeddings(bsd, ep)
    gmap = None
    if return_gmap:
        ge, gm = gmap_input_embedding(bsd, ep, split_embeds, split_lens)
        w, b = bsd['global_encoder.sprel_linear.weight'].reshape(()), bsd['global_encoder.sprel_linear.bias'].reshape(())
        gmap = crossmodal_encoder(bsd, 'global_encoder.encoder', 4, txt, txt_masks, ge, gm, (ep['gmap_pair_dists'] * w + b)[:, None])
    ve, vm = vp_input_embedding(bsd, ep, split_embeds, split_lens)
    vp = crossmodal_encoder(bsd, 'local_encoder.encoder', 4, txt, txt_masks, ve, vm)
    return gmap, vp, txt, txt_masks


def lang2visn_layer(bsd, p, lang, lang_add, visn, visn_add):
    """GraphLXRTXLayer.forward_lang2visn, model/vilmodel.py:400-411: the instruction attends to the map / the panorama"""
    x = cross_attention(bsd, p + '.visual_attention', lang, visn, visn_add)
    x = bert_attention(bsd, p + '.lang_self_att', x, lang_add)
    return bert_ffn(bsd, p + '.lang_inter', p + '.lang_output', x)


def forward_mlm(sd, ep):
    """GlocalTextPathCMTPreTraining.forward_mlm, model/pretrain_cmt.py:128-150 + GlocalTextPathCMT.forward_mlm
    (model/vilmodel.py:700-747): prediction scores [n_masked, vocab] through the tied BertOnlyMLMHead."""
    bsd = _sub(sd)
    txt_masks = seq_masks(ep['txt_lens'], ep['txt_ids'].shape[1])
    txt = forward_text(bsd, ep['txt_ids'], txt_masks)
    ta = neg_mask(txt_masks)
    split_embeds, split_lens = trajectory_embeddings(bsd, ep)
    ge, gm = gmap_input_embedding(bsd, ep, split_embeds, split_lens)
    ve, vm = vp_input_embedding(bsd, ep, split_embeds, split_lens)
    gt, vt = txt, txt
    for i in range(4):
        gt = lang2visn_layer(bsd, 'global_encoder.encoder.x_layers.%d' % i, gt, ta, ge, neg_mask(gm))
        vt = lang2visn_layer(bsd, 'local_encoder.encoder.x_layers.%d' % i, vt, ta, ve, neg_mask(vm))
    h = (gt + vt)[ep['txt_labels'] != -1]
    p = 'mlm_head.predictions'
    h = lnorm(sd, p + '.transform.LayerNorm', gelu_erf(lin(sd, p + '.transform.dense', h)), 1e-12)
    return F.linear(h, sd[p + '.decoder.weight'], sd[p + '.bias'])


def forward_mrc(sd, ep):
    """forward_mrc, model/pretrain_cmt.py:158-204 (views only): (prediction logits, soft-label targets) of the masked views"""
    _, vp, _, _ = forward_bert(sd, ep, return_gmap=False)
    last = torch.cumsum(torch.as_tensor(list(ep['traj_step_lens'])), 0) - 1
    view_lens = ep['traj_vp_view_lens'][last]
    V = int(view_lens.max())
    views = torch.zeros(vp.shape[0], V, vp.shape[2])
    for i in range(vp.shape[0]):
        views[i, :view_lens[i]] = vp[i, 1:view_lens[i] + 1]
    h = views[ep['vp_view_mrc_masks']]
    p = 'image_classifier.net'
    logits = lin(sd, p + '.3', lnorm(sd, p + '.2', torch.relu(lin(sd, p + '.0', h)), 1e-12))
    return logits, ep['vp_view_probs'][ep['vp_view_mrc_masks']]


def forward_sap(sd, ep):
    """forward_sap, model/pretrain_cmt.py:206-262: (global, local, fused) action logits"""
    gmap, vp, _, _ = forward_bert(sd, ep)
    fuse = torch.sigmoid(cls_prediction(sd, 'sap_fuse_linear', torch.cat([gmap[:, 0], vp[:, 0]], 1)))
    gl = cls_prediction(sd, 'global_sap_head', gmap).squeeze(2) * fuse
    gl = gl.masked_fill(ep['gmap_visited_masks'], float('-inf')).masked_fill(~seq_masks(ep['gmap_lens'], gl.shape[1]), float('-inf'))
    ll = cls_prediction(sd, 'local_sap_head', vp).squeeze(2) * (1 - fuse)
    last = torch.cumsum(torch.as_tensor(list(ep['traj_step_lens'])), 0) - 1
    not_nav = torch.cat([torch.zeros(len(last), 1, dtype=torch.bool), ep['traj_nav_types'][last][:, :ll.shape[1] - 1] != 1], 1)
    ll = ll.masked_fill(not_nav, float('-inf'))
    cand = [[None] + list(c[-1]) for c in ep['traj_cand_vpids']]
    return gl, ll, fuse_logits(gl, ll, ep['gmap_vpids'], ep['gmap_visited_masks'], cand)


def losses(sd, ep):
    """what the trainer optimises (compute_loss=True): per-token MLM cross-entropy, per-view MRC KL divergence"""
    scores = forward_mlm(sd, ep)
    mlm = F.cross_entropy(scores, ep['txt_labels'][ep['txt_labels'] != -1], reduction='none')
    logits, targets = forward_mrc(sd, ep)
    mrc = F.kl_div(F.log_softmax(logits, -1), targets, reduction='none').sum(1)
    return mlm, mrc
