"""Synthetic R2R-shaped episodes and deterministic weights for the navigation hot path.

Nothing here touches the reference or the oracle: the generators are shared by the
product benchmark (bench.py), by the parity tests and by the golden-vector script, so
that all three see bit-identical inputs on any machine (numpy PCG64 streams are
platform independent).

Input conventions follow what the reference agents collate for the model
(SURVEY.md section 8(d)):
  * DUET  : VLN-DUET/map_nav_src/r2r/agent.py:38-207 (_language_variable,
            _panorama_feature_variable, _nav_gmap_variable, _nav_vp_variable)
  * HAMT  : VLN-HAMT/finetune_src/r2r/agent_cmt.py:371-605
"""
from __future__ import annotations

import dataclasses
import zlib
from typing import Dict, List

import numpy as np
import torch


@dataclasses.dataclass(frozen=True)
class EpisodeShape:
    """Sizes of one synthetic batch of episodes (names follow the reference's domain)."""
    batch: int = 8          # episodes per rank
    instr_len: int = 80     # L: instruction tokens
    n_imagine: int = 5      # I: sub-instructions / imagination slots
    n_nodes: int = 30       # G: graph-map nodes incl. the [stop] node 0
    n_views: int = 36       # V: panorama views (vp tokens = V + 1 with [stop])
    n_hist: int = 15        # HAMT: history steps (hist tokens = n_hist + 1 with [cls])
    ragged: bool = True     # draw per-episode lengths; False = every episode at full length


CFG1 = EpisodeShape(batch=8)
CFG2 = EpisodeShape(batch=64)
CFG3 = EpisodeShape(batch=64, n_hist=15)
CFG5 = EpisodeShape(batch=256, instr_len=200, n_imagine=12, n_nodes=100)
TINY = EpisodeShape(batch=3, instr_len=24, n_imagine=3, n_nodes=7, n_views=9, n_hist=3)


def _rng(seed: int, tag: str) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64([seed, zlib.crc32(tag.encode())]))


# ----------------------------------------------------------------------------------------------
# weights
# ----------------------------------------------------------------------------------------------

def synth_state_dict(named_shapes: Dict[str, List[int]], seed: int = 0,
                     gasa_stress: bool = False) -> Dict[str, torch.Tensor]:
    """Deterministic BERT-style weights for a parameter manifest {name: shape}.

    Matrices/embeddings ~ N(0, 0.02) (transformers' BertPreTrainedModel._init_weights),
    LayerNorm gains 1 + N(0, 0.05), every bias N(0, 0.02) so that no term is trivially
    zero in a parity run.  ``gasa_stress`` sets global_encoder.sprel_linear to
    (w=-0.5, b=0) so the graph-distance bias visibly shapes the attention
    (SURVEY.md section 8(d): random init gives w~0.02 which barely exercises GASA).
    """
    out = {}
    for name in sorted(named_shapes):
        shape = tuple(named_shapes[name])
        g = _rng(seed, name)
        n = int(np.prod(shape)) if len(shape) else 1
        leaf = name.rsplit('.', 1)[-1]
        is_ln = ('LayerNorm' in name or 'layer_norm' in name or '.norm' in name
                 or name.endswith('vp_pos_embeddings.1.weight') or name.endswith('vp_pos_embeddings.1.bias')
                 or name.endswith('gmap_pos_embeddings.1.weight') or name.endswith('gmap_pos_embeddings.1.bias')
                 or '.net.2.' in name)
        if is_ln and leaf == 'weight':
            a = 1.0 + 0.05 * g.standard_normal(n, dtype=np.float32)
        elif name.endswith('sprel_linear.weight'):
            a = np.full(n, -0.5 if gasa_stress else 0.02, np.float32)
        elif name.endswith('sprel_linear.bias'):
            a = np.full(n, 0.0 if gasa_stress else -0.01, np.float32)
        else:
            a = 0.02 * g.standard_normal(n, dtype=np.float32)
        out[name] = torch.from_numpy(a.reshape(shape).copy())
    return out


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------

def _lens(g, batch, lo, hi, ragged):
    if not ragged or lo >= hi:
        return np.full(batch, hi, np.int64)
    x = g.integers(lo, hi + 1, size=batch).astype(np.int64)
    x[int(g.integers(0, batch))] = hi          # at least one episode at full length
    return x


def _mask_from_lens(lens, width):
    return np.arange(width)[None, :] < lens[:, None]


def _angle_feats(g, shape_prefix, n_angles):
    """sin/cos of uniform angles, like the reference's angle_feature (utils/data.py)."""
    ang = g.uniform(-np.pi, np.pi, size=tuple(shape_prefix) + (n_angles,)).astype(np.float32)
    return np.concatenate([np.sin(ang), np.cos(ang)], -1)


def _rel_pos7(g, shape_prefix):
    """7-d relative position: sin/cos heading, sin/cos elevation, 3 normalised distances
    (VLN-DUET/map_nav_src/models/graph_utils.py:127-148)."""
    a = _angle_feats(g, shape_prefix, 2)                       # (...,4)
    d = g.uniform(0.0, 1.0, size=tuple(shape_prefix) + (3,)).astype(np.float32)
    return np.concatenate([a, d], -1)


# ----------------------------------------------------------------------------------------------
# DUET inputs
# ----------------------------------------------------------------------------------------------

def duet_episode(shape: EpisodeShape, seed: int = 1234) -> dict:
    """One synthetic batch for every DUET mode.  Returns numpy arrays / python lists exactly
    as the reference agent would hand them to ``vln_bert(mode, batch)`` (before .cuda())."""
    B, L, I, G, V = shape.batch, shape.instr_len, shape.n_imagine, shape.n_nodes, shape.n_views
    g = _rng(seed, 'duet')
    ep = {}

    # -- language (agent.py:38-55): [CLS]=101 first, zero padded
    txt_lens = _lens(g, B, max(L // 4, 8), L, shape.ragged)
    txt_ids = g.integers(1000, 30000, size=(B, L)).astype(np.int64)
    txt_ids[:, 0] = 101
    txt_masks = _mask_from_lens(txt_lens, L)
    txt_ids[~txt_masks] = 0
    ep['txt_ids'], ep['txt_masks'], ep['txt_lens'] = txt_ids, txt_masks, txt_lens

    # -- imaginations (agent.py:317-382): slot k holds a feature iff flag k is 'True'
    flags, segs, nps = [], [], []
    n_sub = _lens(g, B, max(1, I // 2), I, shape.ragged)
    imagine_feats = np.zeros((B, I, 768), np.float32)
    imagine_masks = np.zeros((B, I), bool)
    for b in range(B):
        f = (g.uniform(size=n_sub[b]) < 0.8)
        if not f.any():
            f[int(g.integers(0, n_sub[b]))] = True
        flags.append(['True' if x else 'False' for x in f])
        imagine_masks[b, :n_sub[b]] = f
        for k in range(n_sub[b]):
            if f[k]:
                imagine_feats[b, k] = g.standard_normal(768, dtype=np.float32)
        # consecutive sub-instruction segments from token 1, all inside the valid text
        budget = int(txt_lens[b]) - 1
        seg_b, np_b, start = [], [], 1
        for k in range(n_sub[b]):
            remaining = n_sub[b] - k
            max_len = max(1, min(8, budget // remaining))
            ln = int(g.integers(min(3, max_len), max_len + 1))
            s, e = start, start + ln - 1
            seg_b.append([s, e])
            n_np = int(g.integers(0, 3)) if k % 4 == 3 else int(g.integers(1, 3))
            spans = []
            for _ in range(n_np):
                a = int(g.integers(s, e + 1))
                z = int(min(e, a + g.integers(0, 3)))
                spans.append([a, z])
            np_b.append(spans)
            start, budget = e + 1, budget - ln
        segs.append(seg_b)
        nps.append(np_b)
    ep['imagine_feats'], ep['imagine_masks'] = imagine_feats, imagine_masks
    ep['sub_instr_imag_flag'], ep['sub_instr_segs'], ep['noun_phrase_segs'] = flags, segs, nps
    ep['obs_instr_ids'] = ['%d_%d' % (1000 + b, b % 3) for b in range(B)]

    # -- panorama (agent.py:57-96): candidates first (nav_type 1), remaining views 0
    view_lens = _lens(g, B, max(V - 4, 4), V, shape.ragged)
    n_cand = g.integers(2, 7, size=B).astype(np.int64)
    n_cand = np.minimum(np.minimum(n_cand, view_lens), max(G - 2, 1))
    view_img_fts = g.standard_normal((B, V, 768), dtype=np.float32)
    loc_fts = _rel_pos7(g, (B, V))
    nav_types = (np.arange(V)[None, :] < n_cand[:, None]).astype(np.int64)
    vmask = _mask_from_lens(view_lens, V)
    view_img_fts[~vmask] = 0
    loc_fts[~vmask] = 0
    nav_types[~vmask] = 0
    ep.update(view_img_fts=view_img_fts, loc_fts=loc_fts, nav_types=nav_types,
              view_lens=view_lens, n_cand=n_cand)

    # -- graph map (agent.py:98-171)
    gmap_lens = _lens(g, B, max(5, n_cand.max() + 2), G, shape.ragged)
    gmap_lens = np.maximum(gmap_lens, n_cand + 2)
    gmap_masks = _mask_from_lens(gmap_lens, G)
    gmap_img_embeds = g.standard_normal((B, G, 768), dtype=np.float32)
    gmap_img_embeds[:, 0] = 0                      # [stop]
    gmap_img_embeds[~gmap_masks] = 0
    gmap_step_ids = g.integers(0, 15, size=(B, G)).astype(np.int64)
    gmap_step_ids[:, 0] = 0
    gmap_step_ids[~gmap_masks] = 0
    gmap_pos_fts = _rel_pos7(g, (B, G))
    gmap_pos_fts[~gmap_masks] = 0
    d = g.uniform(0.0, 20.0, size=(B, G, G)).astype(np.float32)
    d = np.triu(d, 1)
    d = d + d.transpose(0, 2, 1)
    d[:, 0, :] = 0
    d[:, :, 0] = 0
    pm = gmap_masks[:, :, None] & gmap_masks[:, None, :]
    d[~pm] = 0
    n_visited = np.array([int(g.integers(1, max(2, gmap_lens[b] - n_cand[b]))) for b in range(B)])
    gmap_visited_masks = np.zeros((B, G), bool)
    gmap_vpids, vp_cand_vpids = [], []
    for b in range(B):
        gmap_visited_masks[b, 1:1 + n_visited[b]] = True
        ids = [None] + ['vp%02d_%03d' % (b, j) for j in range(1, int(gmap_lens[b]))]
        gmap_vpids.append(ids)
        # candidates: one already-visited node + (n_cand-1) unvisited nodes that are in the graph
        unvisited = [j for j in range(1 + n_visited[b], int(gmap_lens[b]))]
        pick = [1 + int(g.integers(0, n_visited[b]))]
        perm = g.permutation(len(unvisited))[: int(n_cand[b]) - 1]
        pick += [unvisited[int(k)] for k in perm]
        order = g.permutation(len(pick))
        vp_cand_vpids.append([None] + [ids[pick[int(k)]] for k in order])
    ep.update(gmap_img_embeds=gmap_img_embeds, gmap_step_ids=gmap_step_ids, gmap_pos_fts=gmap_pos_fts,
              gmap_masks=gmap_masks, gmap_pair_dists=d, gmap_visited_masks=gmap_visited_masks,
              gmap_vpids=gmap_vpids, gmap_lens=gmap_lens)

    # -- local viewpoint tokens (agent.py:173-207): [stop] + panorama
    vp_img_embeds = g.standard_normal((B, V + 1, 768), dtype=np.float32)
    vp_img_embeds[:, 0] = 0
    vp_masks = _mask_from_lens(view_lens + 1, V + 1)
    vp_img_embeds[~vp_masks] = 0
    vp_pos_fts = np.zeros((B, V + 1, 14), np.float32)
    vp_pos_fts[:, :, :7] = _rel_pos7(g, (B, 1))
    cand7 = _rel_pos7(g, (B, V))
    for b in range(B):
        vp_pos_fts[b, 1:1 + n_cand[b], 7:] = cand7[b, :n_cand[b]]
    vp_nav_masks = np.concatenate([np.ones((B, 1), bool), nav_types == 1], 1)
    ep.update(vp_img_embeds=vp_img_embeds, vp_pos_fts=vp_pos_fts, vp_masks=vp_masks,
              vp_nav_masks=vp_nav_masks, vp_cand_vpids=vp_cand_vpids)
    return ep


def duet_reverie_episode(shape: EpisodeShape, seed: int = 1234, max_objects: int = 8, obj_dim: int = 768) -> dict:
    """duet_episode in the shape the REVERIE agent collates (VLN-DUET/map_nav_src/reverie/agent_obj.py:50-212): a ragged
    number of object boxes per panorama ([views ; objects] per episode, nav_type 2 for objects, zero padded to the longest),
    the matching local tokens with ``vp_obj_masks``, and ONE imagination per instruction (imagine tensors [B, 1, ...])."""
    ep = duet_episode(shape, seed)
    B, V = shape.batch, shape.n_views
    g = _rng(seed, 'duet_reverie')
    view_lens, n_cand = ep['view_lens'], ep['n_cand']
    obj_lens = g.integers(0, max_objects + 1, size=B).astype(np.int64)
    obj_lens[0], obj_lens[-1] = 0, max_objects                 # an episode without objects and a full one
    O = int(obj_lens.max())
    obj_img_fts = g.standard_normal((B, O, obj_dim), dtype=np.float32)     # 768: REVERIE ViT boxes; 2048: SOON butd boxes
    obj_img_fts[~_mask_from_lens(obj_lens, O)] = 0
    pano_lens = view_lens + obj_lens
    P = int(pano_lens.max())
    loc_fts = np.zeros((B, P, 7), np.float32)
    nav_types = np.zeros((B, P), np.int64)
    obj_loc = _rel_pos7(g, (B, max(O, 1)))
    for b in range(B):
        vl, ol = int(view_lens[b]), int(obj_lens[b])
        loc_fts[b, :vl] = ep['loc_fts'][b, :vl]
        loc_fts[b, vl:vl + ol] = obj_loc[b, :ol]
        nav_types[b, :vl] = ep['nav_types'][b, :vl]
        nav_types[b, vl:vl + ol] = 2
    ep.update(obj_img_fts=obj_img_fts, obj_lens=obj_lens, loc_fts=loc_fts, nav_types=nav_types)
    vp_masks = _mask_from_lens(pano_lens + 1, P + 1)
    vp_img_embeds = g.standard_normal((B, P + 1, 768), dtype=np.float32)
    vp_img_embeds[:, 0] = 0
    vp_img_embeds[~vp_masks] = 0
    vp_pos_fts = np.zeros((B, P + 1, 14), np.float32)
    vp_pos_fts[:, :, :7] = ep['vp_pos_fts'][:, :1, :7]
    for b in range(B):
        vp_pos_fts[b, 1:1 + n_cand[b], 7:] = ep['vp_pos_fts'][b, 1:1 + n_cand[b], 7:]
    ep.update(vp_img_embeds=vp_img_embeds, vp_pos_fts=vp_pos_fts, vp_masks=vp_masks,
              vp_nav_masks=np.concatenate([np.ones((B, 1), bool), nav_types == 1], 1),
              vp_obj_masks=np.concatenate([np.zeros((B, 1), bool), nav_types == 2], 1))
    ep['imagine_feats'] = g.standard_normal((B, 1, 768), dtype=np.float32)
    ep['imagine_masks'] = np.ones((B, 1), bool)
    for k in ('sub_instr_imag_flag', 'sub_instr_segs', 'noun_phrase_segs'):      # REVERIE has no sub-instruction annotation
        ep.pop(k)
    return ep


# ----------------------------------------------------------------------------------------------
# HAMT inputs
# ----------------------------------------------------------------------------------------------

def hamt_episode(shape: EpisodeShape, seed: int = 1234) -> dict:
    """One synthetic batch for every HAMT mode (agent_cmt.py:371-605).  Observation tokens are
    candidates (nav_type 1), then [stop] (nav_type 2), then the remaining views (nav_type 0)."""
    B, L, I, V, T = shape.batch, shape.instr_len, shape.n_imagine, shape.n_views, shape.n_hist
    base = duet_episode(shape, seed)            # language + imagination parts are shared
    g = _rng(seed, 'hamt')
    ep = {k: base[k] for k in ('txt_ids', 'txt_masks', 'txt_lens', 'imagine_feats', 'imagine_masks',
                               'sub_instr_imag_flag', 'sub_instr_segs', 'noun_phrase_segs', 'obs_instr_ids')}
    O = V + 1
    ob_lens = _lens(g, B, max(O - 4, 5), O, shape.ragged)
    n_cand = np.minimum(g.integers(2, 7, size=B), ob_lens - 1).astype(np.int64)
    ob_img_feats = g.standard_normal((B, O, 768), dtype=np.float32)
    ob_ang_feats = _angle_feats(g, (B, O), 2)
    ob_nav_types = np.zeros((B, O), np.int64)
    for b in range(B):
        ob_nav_types[b, :n_cand[b]] = 1
        ob_nav_types[b, n_cand[b]] = 2
        ob_img_feats[b, n_cand[b]] = 0          # the [stop] observation carries no image
    ob_masks = _mask_from_lens(ob_lens, O)
    ob_img_feats[~ob_masks] = 0
    ob_ang_feats[~ob_masks] = 0
    ob_nav_types[~ob_masks] = 0
    ep.update(ob_img_feats=ob_img_feats, ob_ang_feats=ob_ang_feats, ob_nav_types=ob_nav_types,
              ob_masks=ob_masks, ob_lens=ob_lens)
    # history: T steps already taken; hist_lens counts the [cls] slot too
    hist_lens = _lens(g, B, 1, T + 1, shape.ragged)
    ep['hist_lens'] = hist_lens
    ep['hist_embeds'] = g.standard_normal((B, T + 1, 768), dtype=np.float32) * 0.5
    ep['hist_img_feats'] = g.standard_normal((B, 768), dtype=np.float32)
    ep['hist_ang_feats'] = _angle_feats(g, (B,), 2)
    ep['hist_pano_img_feats'] = g.standard_normal((B, V, 768), dtype=np.float32)
    ep['hist_pano_ang_feats'] = _angle_feats(g, (B, V), 2)
    ep['ob_step'] = min(T, 49)
    return ep


def to_torch(ep: dict, device='cpu') -> dict:
    out = {}
    for k, v in ep.items():
        if isinstance(v, np.ndarray):
            out[k] = torch.from_numpy(v).to(device)
        else:
            out[k] = v
    return out


# ----------------------------------------------------------------------------------------------
# a synthetic navigation world for the per-step graph glue (SURVEY.md section 8(f), N1 / N2)
# ----------------------------------------------------------------------------------------------

def nav_world(seed: int = 7, n_vp: int = 24, batch: int = 4, steps: int = 6, n_views: int = 36, hidden: int = 768,
              degree: int = 3) -> List[dict]:
    """A rollout's worth of observations over a random viewpoint graph, in the shape the reference agent sees them
    (VLN-DUET/map_nav_src/r2r/env.py observations: 'viewpoint', 'position', 'heading', 'elevation',
    'candidate': [{'viewpointId', 'position'}]).  Returns one dict per step:

        obs          list[batch] of observation dicts (the state BEFORE acting at this step)
        ended        bool [batch]    episodes that stopped at an earlier step (agent.py:452, 609)
        pano_embeds  fp32 [batch, n_views, hidden]   stand-in for the panorama encoder's output of this step
        view_lens    int64 [batch]; nav_types int64 [batch, n_views] (1 for the candidate views, which come first)
    """
    g = _rng(seed, 'nav_world')
    pos = np.concatenate([g.uniform(-12, 12, (n_vp, 2)), g.uniform(-1.5, 1.5, (n_vp, 1))], 1)
    names = ['vp%03d' % i for i in range(n_vp)]
    d = np.linalg.norm(pos[:, None] - pos[None], axis=-1)
    nbr = [set() for _ in range(n_vp)]
    for i in range(n_vp):                                     # symmetric k-nearest-neighbour connectivity
        for j in np.argsort(d[i])[1:degree + 1]:
            nbr[i].add(int(j)); nbr[int(j)].add(i)
    for i in range(n_vp - 1):                                 # a spanning chain keeps the graph connected
        nbr[i].add(i + 1); nbr[i + 1].add(i)
    cur = [int(x) for x in g.integers(0, n_vp, batch)]
    seen = [{c} for c in cur]
    stop_at = [int(x) for x in g.integers(max(2, steps // 2), steps + 1, batch)]
    stop_at[0] = steps                                        # at least one episode runs the whole horizon
    out = []
    ended = np.zeros(batch, bool)
    for t in range(steps):
        obs = []
        nav_types = np.zeros((batch, n_views), np.int64)
        for b in range(batch):
            cands = sorted(nbr[cur[b]])
            order = g.permutation(len(cands))
            cands = [cands[i] for i in order]
            obs.append({'viewpoint': names[cur[b]], 'position': tuple(float(x) for x in pos[cur[b]]),
                        'heading': float(g.uniform(0, 2 * np.pi)), 'elevation': float(g.uniform(-0.5, 0.5)),
                        'candidate': [{'viewpointId': names[c], 'position': tuple(float(x) for x in pos[c])} for c in cands]})
            nav_types[b, :len(cands)] = 1
        out.append({'obs': obs, 'ended': ended.copy(),
                    'pano_embeds': g.standard_normal((batch, n_views, hidden)).astype(np.float32),
                    'view_lens': np.full((batch,), n_views, np.int64), 'nav_types': nav_types})
        for b in range(batch):                                # act: prefer an unseen neighbour, stop when scheduled
            if ended[b]:
                continue
            if t + 1 >= stop_at[b]:
                ended[b] = True
                continue
            cands = sorted(nbr[cur[b]])
            fresh = [c for c in cands if c not in seen[b]]
            pool = fresh if fresh else cands
            cur[b] = pool[int(g.integers(0, len(pool)))]
            seen[b].add(cur[b])
    return out


# ----------------------------------------------------------------------------------------------
# DUET pre-training batches (whole trajectories; VLN-DUET/pretrain_src/data/tasks.py collate functions)
# ----------------------------------------------------------------------------------------------

def duet_pretrain_batch(seed: int = 5, batch: int = 3, n_vp: int = 20, max_steps: int = 4, n_views: int = 12, instr_len: int = 24,
                        n_probs: int = 1000) -> dict:
    """One synthetic pre-training batch in the layout of the reference's mlm / mrc / sap collate functions: trajectories of
    1..max_steps panoramas flattened along dim 0 (``traj_step_lens`` splits them), the graph built from the visited viewpoints
    and every candidate seen on the way, the last panorama as the local branch.  R2R: no object features."""
    g = _rng(seed, 'duet_pretrain')
    pos = g.uniform(-10, 10, (n_vp, 3))
    d = np.linalg.norm(pos[:, None] - pos[None], axis=-1)
    nbr = [sorted(int(j) for j in np.argsort(d[i])[1:5]) for i in range(n_vp)]
    names = ['pv%02d' % i for i in range(n_vp)]
    B, V, L = batch, n_views, instr_len
    step_lens = [int(x) for x in g.integers(1, max_steps + 1, B)]
    step_lens[0] = max_steps
    traj_vpids, traj_cand_vpids, view_lens, nav_types_rows = [], [], [], []
    for b in range(B):
        cur = int(g.integers(0, n_vp))
        path, cands_b = [], []
        for t in range(step_lens[b]):
            path.append(cur)
            cands = [c for c in nbr[cur]]
            order = g.permutation(len(cands))
            cands = [cands[int(i)] for i in order]
            cands_b.append(cands)
            vl = int(g.integers(max(len(cands), V - 3), V + 1))
            view_lens.append(vl)
            nt = np.zeros(V, np.int64)
            nt[:len(cands)] = 1
            nav_types_rows.append(nt)
            fresh = [c for c in cands if c not in path]
            cur = (fresh or cands)[int(g.integers(0, len(fresh or cands)))]
        traj_vpids.append([names[i] for i in path])
        traj_cand_vpids.append([[names[c] for c in cs] for cs in cands_b])
    N = sum(step_lens)
    view_lens = np.array(view_lens, np.int64)
    vmask = _mask_from_lens(view_lens, V)
    traj_view_img_fts = g.standard_normal((N, V, 768), dtype=np.float32)
    traj_view_img_fts[~vmask] = 0
    traj_loc_fts = _rel_pos7(g, (N, V))
    traj_loc_fts[~vmask] = 0
    traj_nav_types = np.stack(nav_types_rows, 0)
    traj_nav_types[~vmask] = 0
    gmap_vpids, visited = [], []
    for b in range(B):
        vis = list(dict.fromkeys(traj_vpids[b]))
        unv = [v for v in dict.fromkeys(c for cs in traj_cand_vpids[b] for c in cs) if v not in vis]
        gmap_vpids.append([None] + vis + unv)
        visited.append([False] + [True] * len(vis) + [False] * len(unv))
    gmap_lens = np.array([len(x) for x in gmap_vpids], np.int64)
    G = int(gmap_lens.max())
    gmask = _mask_from_lens(gmap_lens, G)
    gmap_step_ids = g.integers(0, 10, (B, G)).astype(np.int64)
    gmap_step_ids[:, 0] = 0
    gmap_step_ids[~gmask] = 0
    gmap_pos_fts = _rel_pos7(g, (B, G))
    gmap_pos_fts[~gmask] = 0
    pd = np.triu(g.uniform(0, 20, (B, G, G)).astype(np.float32), 1)
    pd = pd + pd.transpose(0, 2, 1)
    pd[:, 0, :] = 0
    pd[:, :, 0] = 0
    pd[~(gmask[:, :, None] & gmask[:, None, :])] = 0
    gmap_visited_masks = np.zeros((B, G), bool)
    for b in range(B):
        gmap_visited_masks[b, :len(visited[b])] = visited[b]
    last = np.cumsum(step_lens) - 1
    P = int(view_lens[last].max()) + 1
    vp_pos_fts = np.zeros((B, P, 14), np.float32)
    vp_pos_fts[:, :, :7] = _rel_pos7(g, (B, 1))
    c7 = _rel_pos7(g, (B, V))
    for b in range(B):
        nc = len(traj_cand_vpids[b][-1])
        vp_pos_fts[b, 1:1 + nc, 7:] = c7[b, :nc]
    txt_lens = _lens(g, B, max(L // 3, 6), L, True)
    txt_ids = g.integers(1000, 30000, (B, L)).astype(np.int64)
    txt_ids[:, 0] = 101
    tmask = _mask_from_lens(txt_lens, L)
    txt_ids[~tmask] = 0
    txt_labels = np.full((B, L), -1, np.int64)
    for b in range(B):                                        # a few masked tokens per instruction (103 = [MASK])
        for j in g.choice(np.arange(1, txt_lens[b]), size=min(3, int(txt_lens[b]) - 1), replace=False):
            txt_labels[b, j] = txt_ids[b, j]
            txt_ids[b, j] = 103
    Vl = int(view_lens[last].max())
    vp_view_mrc_masks = np.zeros((B, Vl), bool)
    for b in range(B):
        k = g.choice(np.arange(view_lens[last[b]]), size=2, replace=False)
        vp_view_mrc_masks[b, k] = True
    probs = g.gamma(0.3, size=(B, Vl, n_probs)).astype(np.float32) + 1e-6
    vp_view_probs = probs / probs.sum(-1, keepdims=True)
    return dict(txt_ids=txt_ids, txt_lens=txt_lens, txt_labels=txt_labels, traj_view_img_fts=traj_view_img_fts,
                traj_obj_img_fts=None, traj_loc_fts=traj_loc_fts, traj_nav_types=traj_nav_types, traj_step_lens=step_lens,
                traj_vp_view_lens=view_lens, traj_vp_obj_lens=None, traj_vpids=traj_vpids, traj_cand_vpids=traj_cand_vpids,
                gmap_lens=gmap_lens, gmap_step_ids=gmap_step_ids, gmap_pos_fts=gmap_pos_fts, gmap_pair_dists=pd,
                gmap_vpids=gmap_vpids, vp_pos_fts=vp_pos_fts, gmap_visited_masks=gmap_visited_masks,
                vp_view_mrc_masks=vp_view_mrc_masks, vp_view_probs=vp_view_probs)


def duet_pretrain_sap_labels(batch: dict) -> dict:
    """``global_act_labels`` / ``local_act_labels`` of the sap collate function (data/tasks.py) for a duet_pretrain_batch: the
    last admissible graph node (valid, unvisited) and the last navigable candidate of the last panorama ([stop] = 0 when there
    is none), so both targets have finite logits.  Returns the batch with the two labels added."""
    B = len(batch['traj_step_lens'])
    last = np.cumsum(np.asarray(batch['traj_step_lens'])) - 1
    nav = np.asarray(batch['traj_nav_types'])[last]
    visited = np.asarray(batch['gmap_visited_masks'])
    gl, ll = np.zeros(B, np.int64), np.zeros(B, np.int64)
    for b in range(B):
        ok = [g for g in range(1, int(batch['gmap_lens'][b])) if not visited[b, g]]
        gl[b] = ok[-1] if ok else 0
        cand = [j + 1 for j in range(len(batch['traj_cand_vpids'][b][-1])) if nav[b, j] == 1]
        ll[b] = cand[-1] if cand else 0
    return dict(batch, global_act_labels=gl, local_act_labels=ll)
