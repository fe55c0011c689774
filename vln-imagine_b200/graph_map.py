"""Device-resident graph maps for a DUET rollout (SURVEY.md section 8(f), rows N1 and N2).

The reference agent keeps one Python ``GraphMap`` per episode (VLN-DUET/map_nav_src/models/graph_utils.py:96-148) and
rebuilds the navigation inputs from it at every step with per-node Python loops and per-episode host->device copies
(r2r/agent.py:98-207, 466-479).  ``DeviceGraphMaps`` is the batch of those objects with the state in HBM: the host
only interns viewpoint-id strings into node indices and ships ONE small packed buffer per call; distances, running
mean embeddings, position features and the padded batch tensors are produced by three libvlnimagine kernels
(csrc/vi_graph.cu).  Method names and the returned dict keys are the reference's, so the rollout loop reads the same:

    gmaps = DeviceGraphMaps(obs, device)                          # agent.py:395-398  GraphMap(...) + update_graph
    gmaps.set_step_ids(obs, t, ended)                             # agent.py:461-464
    nav_inputs = gmaps.nav_inputs(obs, pano_embeds, pano_masks, pano_inputs, ended)   # agent.py:466-493
    gmaps.update_graph(obs, ended)                                # agent.py:599-604

No CPU path: every array below is computed on the GPU; the oracle (oracle/graph_oracle.py) is only used by tests.
"""
from __future__ import annotations

import collections.abc
from typing import Dict, List, Sequence

import numpy as np
import torch

from . import _lib, ops

lib = ops.lib           # checked and traced like every library call

MAX_NODES = 128


class _Staging:
    """A small ring of pinned host buffers: one packed host->device copy per call.  Every slot carries the CUDA event of its
    last copy; a slot is rewritten only after that copy has completed (the wait is free unless the caller runs more than
    ``slots`` calls ahead of the device)."""

    def __init__(self, slots: int = 4):
        self.bufs = [None] * slots
        self.events = [None] * slots
        self.i = 0

    def get(self, nbytes: int) -> torch.Tensor:
        self.i = (self.i + 1) % len(self.bufs)
        ev = self.events[self.i]
        if ev is not None:
            ev.synchronize()                     # the H2D copy that last read this slot has finished
        b = self.bufs[self.i]
        if b is None or b.numel() < nbytes:
            b = self.bufs[self.i] = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8).pin_memory()
        return b

    def copied(self):
        """record the copy just queued from the current slot on the current stream"""
        ev = self.events[self.i]
        if ev is None:
            ev = self.events[self.i] = torch.cuda.Event()
        ev.record()


_TORCH_DTYPE = {np.dtype(k).char: v for k, v in (('float64', torch.float64), ('float32', torch.float32), ('int64', torch.int64),
                                                 ('int32', torch.int32), ('uint8', torch.uint8))}


def _pack(staging: _Staging, device, arrays: Dict[str, np.ndarray]) -> Dict[str, torch.Tensor]:
    """Concatenate numpy arrays (8-byte aligned each) into one pinned buffer, copy once, return device views."""
    offs, total = {}, 0
    for k, a in arrays.items():
        offs[k] = total
        total += (a.nbytes + 7) & ~7
    host = staging.get(total)
    hv = host.numpy()
    for k, a in arrays.items():
        hv[offs[k]:offs[k] + a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    dev = host[:total].to(device, non_blocking=True)
    if dev.is_cuda:
        staging.copied()
    out = {}
    for k, a in arrays.items():
        out[k] = dev[offs[k]:offs[k] + a.nbytes].view(_TORCH_DTYPE[a.dtype.char]).view(a.shape)
    return out


STOP_ID = 1 << 20      # id of the [stop] slot (None) in the interned-id tensors handed to the fusion kernel


class VpidRows(collections.abc.Sequence):
    """``gmap_vpids`` / ``vp_cand_vpids`` of a step as the agent reads them (a list of per-episode lists of viewpoint-id
    strings, None for [stop]: r2r/agent.py:113-118, 205), materialised row by row on first access, plus the same rows as an
    int32 device tensor (``ids``: node indices, [stop] = STOP_ID, padding = ``pad``) which the navigation call uses instead of
    interning ~1700 strings per step (duet.GlocalTextPathNavCMT.intern_vpids)."""

    def __init__(self, names, nodes: np.ndarray, lens: np.ndarray, ids: torch.Tensor, pad: int):
        self._names, self._nodes, self._lens, self.ids, self.pad = names, nodes, lens, ids, pad
        self._rows = [None] * len(lens)

    def __len__(self):
        return len(self._rows)

    def __getitem__(self, b):
        if isinstance(b, slice):
            return [self[i] for i in range(*b.indices(len(self)))]
        row = self._rows[b]
        if row is None:
            names = self._names[b]
            row = self._rows[b] = [None] + [names[i] for i in self._nodes[b, 1:self._lens[b]]]
        return row

    def __eq__(self, other):
        return list(self) == list(other)


class _CandRows(list):
    """vp_cand_vpids (agent.py:205) with the same rows as interned ids on the device (``ids``, padding -2)"""

    def __init__(self, rows, ids: torch.Tensor):
        super().__init__(rows)
        self.ids = ids


class DeviceGraphMaps:
    def __init__(self, obs: Sequence[dict], device, hidden: int = 768, max_nodes: int = MAX_NODES):
        self.device = torch.device(device)
        self.B, self.N, self.H = len(obs), int(max_nodes), int(hidden)
        B, N = self.B, self.N
        ops.ensure_init(torch.zeros(1, device=self.device))
        self.pos = torch.zeros((B, N, 3), dtype=torch.float64, device=self.device)
        self.dis = torch.empty((B, N, N), dtype=torch.float64, device=self.device)
        self.point = torch.empty((B, N, N), dtype=torch.int32, device=self.device)
        self.visited_dev = torch.empty((B, N), dtype=torch.uint8, device=self.device)
        self.esum = torch.zeros((B, N, hidden), dtype=torch.float32, device=self.device)
        self.ecnt = torch.empty((B, N), dtype=torch.float32, device=self.device)
        lib.vi_graph_init(self.dis.data_ptr(), self.point.data_ptr(), self.visited_dev.data_ptr(), self.ecnt.data_ptr(),
                          B, N, ops._stream())
        # host mirror of what only needs strings / small ints
        self.start_vps = [ob['viewpoint'] for ob in obs]            # GraphMap.start_vp
        self.index: List[Dict[str, int]] = [dict() for _ in obs]    # viewpoint id -> node index (node_positions order)
        self.names: List[List[str]] = [[] for _ in obs]
        self.visited = np.zeros((B, N), bool)                       # FloydGraph._visited
        self.step_ids = np.zeros((B, N), np.int64)                  # GraphMap.node_step_ids, by node index
        self.n_nodes = np.zeros((B,), np.int32)
        self._ar = np.arange(N)
        self._staging = _Staging()
        self.update_graph(obs)

    # ------------------------------------------------------------------ graph_utils.py:109-115
    def _node(self, b: int, vp: str) -> int:
        idx = self.index[b]
        i = idx.get(vp)
        if i is None:
            i = idx[vp] = len(self.names[b])
            if i >= self.N:
                raise _lib.VlnImagineError('episode %d exceeds max_nodes=%d graph nodes' % (b, self.N))
            self.names[b].append(vp)
            self.n_nodes[b] = i + 1
        return i

    def update_graph(self, obs: Sequence[dict], ended=None):
        """GraphMap.update_graph(ob) for every episode that has not ended (agent.py:396-398, 599-604)."""
        B = self.B
        C = max(1, max(len(ob['candidate']) for ob in obs))
        cur = np.full((B,), -1, np.int32)
        cur_pos = np.zeros((B, 3), np.float64)
        cand = np.full((B, C), -1, np.int32)
        cand_pos = np.zeros((B, C, 3), np.float64)
        node = self._node
        for b, ob in enumerate(obs):
            if ended is not None and ended[b]:
                continue
            cur[b] = node(b, ob['viewpoint'])
            cur_pos[b] = ob['position']
            cc = ob['candidate']
            if cc:
                n = len(cc)
                cand[b, :n] = [node(b, c['viewpointId']) for c in cc]
                cand_pos[b, :n] = [c['position'] for c in cc]
        act = cur >= 0
        self.visited[act, cur[act]] = True
        n_nodes = self.n_nodes.copy()
        d = _pack(self._staging, self.device, dict(cur_pos=cur_pos, cand_pos=cand_pos, cur=cur, cand=cand, n_nodes=n_nodes))
        lib.vi_graph_update(self.pos.data_ptr(), self.dis.data_ptr(), self.point.data_ptr(), self.visited_dev.data_ptr(),
                            B, self.N, d['cur'].data_ptr(), d['cur_pos'].data_ptr(), d['cand'].data_ptr(),
                            d['cand_pos'].data_ptr(), C, d['n_nodes'].data_ptr(), ops._stream())

    def set_step_ids(self, obs: Sequence[dict], t: int, ended):
        for b, ob in enumerate(obs):                                 # agent.py:461-464
            if not ended[b]:
                self.step_ids[b, self.index[b][ob['viewpoint']]] = t + 1

    # ------------------------------------------------------------------ agent.py:466-493
    def nav_inputs(self, obs: Sequence[dict], pano_embeds: torch.Tensor, pano_masks: torch.Tensor, pano_inputs: dict,
                   ended) -> dict:
        """Node-embedding update (agent.py:466-479) + _nav_gmap_variable (:98-171, enc_full_graph) + _nav_vp_variable
        (:173-207).  pano_inputs: the dict _panorama_feature_variable returned ('cand_vpids', 'view_lens', 'nav_types')."""
        B, V, H = pano_embeds.shape
        if H != self.H or B != self.B:
            raise _lib.VlnImagineError('pano_embeds of shape %s does not match the graph memory (B=%d, H=%d)'
                                       % (tuple(pano_embeds.shape), self.B, self.H))
        cand_vpids = pano_inputs['cand_vpids']
        C = max(1, max(len(c) for c in cand_vpids))
        N, ar = self.N, self._ar
        # [stop] + visited + unvisited nodes, each group in node_positions order (agent.py:103-118): one stable sort
        n = self.n_nodes
        known = ar[None, :] < n[:, None]
        order = np.argsort(np.where(known, np.where(self.visited, 0, 1), 2).astype(np.int8), axis=1, kind='stable')
        lens = (n + 1).astype(np.int32)
        G = int(lens.max())
        col = ar[None, :G]
        live = col < lens[:, None]
        gnode = np.full((B, G), -1, np.int32)
        gnode[:, 1:] = order[:, :G - 1]
        gnode[~live] = -1
        gnode[:, 0] = -1
        step_ids = np.zeros((B, G), np.int64)
        step_ids[:, 1:] = np.take_along_axis(self.step_ids, order[:, :G - 1], 1)
        step_ids[~live] = 0
        n_vis = self.visited.sum(1)
        vmask = (col >= 1) & (col < 1 + n_vis[:, None])
        no_vp_left = (n_vis == n).tolist()
        cur_all = np.fromiter((idx[ob['viewpoint']] for idx, ob in zip(self.index, obs)), np.int32, B)
        cur = np.where(np.asarray(ended, bool), -1, cur_all).astype(np.int32)        # -1: no embedding update (ended)
        start = np.fromiter((idx[s] for idx, s in zip(self.index, self.start_vps)), np.int32, B)
        heading = np.fromiter((ob['heading'] for ob in obs), np.float64, B)
        elevation = np.fromiter((ob['elevation'] for ob in obs), np.float64, B)
        cand = np.full((B, C), -1, np.int32)
        for b, vps in enumerate(cand_vpids):
            if vps:
                cand[b, :len(vps)] = [self.index[b][v] for v in vps]
        gids = np.where(live, gnode, -1).astype(np.int32)
        gids[:, 0] = STOP_ID
        cids = np.full((B, V + 1), -2, np.int32)
        cids[:, 0] = STOP_ID
        cids[:, 1:C + 1] = np.where(cand >= 0, cand, -2)[:, :V]
        d = _pack(self._staging, self.device, dict(heading=heading, elevation=elevation, step_ids=step_ids, cur=cur, cur_all=cur_all,
                                                   cand=cand, start=start, gnode=gnode, lens=lens, vmask=vmask.view(np.uint8),
                                                   gids=gids, cids=cids))
        pano_embeds = pano_embeds.float().contiguous()
        pm = pano_masks.to(torch.uint8).contiguous()
        dev = self.device
        gmap_img = torch.empty((B, G, H), dtype=torch.float32, device=dev)
        vp_img = torch.empty((B, V + 1, H), dtype=torch.float32, device=dev)
        lib.vi_graph_embed_step(pano_embeds.data_ptr(), pm.data_ptr(), B, V, H, d['cur'].data_ptr(), d['cand'].data_ptr(), C,
                                self.visited_dev.data_ptr(), self.esum.data_ptr(), self.ecnt.data_ptr(), self.N,
                                d['gnode'].data_ptr(), G, gmap_img.data_ptr(), vp_img.data_ptr(), ops._stream())
        gmap_pos = torch.empty((B, G, 7), dtype=torch.float32, device=dev)
        pair = torch.empty((B, G, G), dtype=torch.float32, device=dev)
        vp_pos = torch.empty((B, V + 1, 14), dtype=torch.float32, device=dev)
        lib.vi_graph_features(self.pos.data_ptr(), self.dis.data_ptr(), self.point.data_ptr(), B, self.N,
                              d['cur_all'].data_ptr(), d['heading'].data_ptr(), d['elevation'].data_ptr(),
                              d['gnode'].data_ptr(), d['lens'].data_ptr(), G, gmap_pos.data_ptr(), pair.data_ptr(),
                              d['cand'].data_ptr(), C, d['start'].data_ptr(), V + 1, vp_pos.data_ptr(), ops._stream())
        view_lens = pano_inputs['view_lens']
        nav_types = pano_inputs['nav_types']
        ar = torch.arange(max(G, V + 1), device=dev)
        gmap_masks = ar[None, :G] < d['lens'][:, None]
        vp_masks = ar[None, :V + 1] < (view_lens.to(dev)[:, None] + 1)
        vp_nav_masks = torch.cat([torch.ones((B, 1), dtype=torch.bool, device=dev), nav_types.to(dev) == 1], 1)
        return {
            'gmap_vpids': VpidRows(self.names, gnode, lens, d['gids'], -1), 'gmap_img_embeds': gmap_img, 'gmap_step_ids': d['step_ids'], 'gmap_pos_fts': gmap_pos,
            'gmap_visited_masks': d['vmask'].bool(), 'gmap_pair_dists': pair, 'gmap_masks': gmap_masks, 'no_vp_left': no_vp_left,
            'vp_img_embeds': vp_img, 'vp_pos_fts': vp_pos, 'vp_masks': vp_masks, 'vp_nav_masks': vp_nav_masks,
            'vp_cand_vpids': _CandRows([[None] + list(x) for x in cand_vpids], d['cids']),
        }

    # ------------------------------------------------------------------ reads used by the agent after acting
    def distance(self, b: int, x: str, y: str) -> float:
        """FloydGraph.distance (graph_utils.py:47-51); a device read (synchronises) - the rollout itself never needs it."""
        if x == y:
            return 0.0
        return float(self.dis[b, self.index[b][x], self.index[b][y]])
