"""Image feature databases kept in HBM: per-step model inputs become row indices instead of feature tensors.

The reference agents read their image features from read-only databases for the whole run - ``ImageFeaturesDB``
(VLN-DUET/map_nav_src/r2r/data_utils.py, key ``"<scan>_<viewpoint>"``, (36, F) arrays) and ``ImaginationImageFeaturesDB``
(imagine_db.py, key ``"<path_id>_<instr_idx>"``) - and collate a float tensor on the host at every step
(64 x 37 x 768 fp32 = 6.9 MB per DUET step).  ``DeviceFeatureStore`` holds those arrays in one device tensor once;
``FeatureRows`` names rows of it ([B, N] int32 indices, -1 = a zero row) and is accepted by the modes wherever the agents
pass per-step or per-episode image features.  The first operand is then gathered from the store by one kernel
(vi_gather_rows, blocks.feature_operand) that takes the place of the fp32 -> 16-bit cast of the dense path, with the same
values bit for bit.

The collation helpers below build the indices in exactly the row order of the reference's agent functions and return what
those functions return, with ``FeatureRows`` in place of the image-feature tensor.
"""
from __future__ import annotations

from typing import Dict, List, Mapping, Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops
from .imagine_db import open_source

_STORE_DTYPES = (torch.float32, torch.float16, torch.bfloat16)


class DeviceFeatureStore:
    """Feature arrays ``key -> (n, >= feat_dim)`` in one device tensor [n_rows, feat_dim] of ``dtype``; every key owns a
    contiguous block of rows (row ``start + k`` = its k-th array row, sliced to ``feat_dim`` columns as the reference DBs do).

    ``dtype=torch.float16`` (default) halves the footprint: the host-side float -> fp16 conversion at load time is a storage
    cast, like the 16-bit weight shadows.  ``dtype=torch.float32`` is exact with respect to the fp32 features the agent would
    have uploaded.  ``add`` may reallocate the tensor (one reallocation per call); captured CUDA graphs key on its address."""

    def __init__(self, device, feat_dim: int, dtype=torch.float16):
        if dtype not in _STORE_DTYPES:
            raise ValueError('store dtype must be torch.float32, torch.float16 or torch.bfloat16')
        if feat_dim <= 0 or feat_dim % 8:
            raise ValueError('feat_dim must be a positive multiple of 8 (got %d)' % feat_dim)
        self.device = torch.device(device)
        self.feat_dim = int(feat_dim)
        self.dtype = dtype
        self.spans: Dict[str, Tuple[int, int]] = {}        # key -> (first row, number of rows)
        self.tensor = torch.empty((0, self.feat_dim), dtype=dtype, device=self.device)

    @classmethod
    def load(cls, source, device, feat_dim: int, dtype=torch.float16, keys: Optional[Sequence[str]] = None):
        """a store holding ``keys`` (default: every key) of ``source``: a mapping, an .npz path or an HDF5 path (h5py)"""
        return cls(device, feat_dim, dtype).add(source, keys)

    @property
    def n_rows(self) -> int:
        return self.tensor.shape[0]

    def __len__(self) -> int:
        return len(self.spans)

    def __contains__(self, key) -> bool:
        return key in self.spans

    def add(self, source, keys: Optional[Sequence[str]] = None) -> 'DeviceFeatureStore':
        """append the arrays of ``keys`` (default: all) of ``source`` that the store does not hold yet"""
        src = open_source(source)
        try:
            keys = list(src.keys()) if keys is None else list(keys)
            arrays, seen = [], set()
            for k in keys:
                if k in self.spans or k in seen:
                    continue
                a = np.asarray(src[k][...])
                if a.ndim != 2 or a.shape[1] < self.feat_dim:
                    raise ValueError('%s: feature array of shape %s has fewer than %d columns' % (k, a.shape, self.feat_dim))
                arrays.append((k, a[:, :self.feat_dim]))
                seen.add(k)
        finally:
            if src is not source and hasattr(src, 'close'):
                src.close()
        n_new = sum(a.shape[0] for _, a in arrays)
        if n_new == 0:
            return self
        host = torch.empty((n_new, self.feat_dim), dtype=self.dtype)
        row, n_old = 0, self.n_rows
        for k, a in arrays:
            host[row:row + a.shape[0]] = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
            self.spans[k] = (n_old + row, a.shape[0])
            row += a.shape[0]
        grown = torch.empty((n_old + n_new, self.feat_dim), dtype=self.dtype, device=self.device)
        grown[:n_old].copy_(self.tensor)
        grown[n_old:].copy_(host)
        self.tensor = grown
        return self

    def span(self, key) -> Tuple[int, int]:
        """(first row, number of rows) of ``key``; KeyError for an unknown key"""
        s = self.spans.get(key)
        if s is None:
            raise KeyError(key)
        return s

    def row(self, key, k: int = 0) -> int:
        """store row of the k-th array row of ``key``"""
        start, n = self.span(key)
        if not 0 <= k < n:
            raise IndexError('%s has %d feature rows, asked for row %d' % (key, n, k))
        return start + k


class FeatureRows:
    """Image features named by rows of a feature store: ``idx`` int32 [B, N] or [B], host (pinned) or device, -1 = a zero row.
    ``shape`` is ``idx.shape + (feat_dim,)``, so the modes read their sizes as from the dense tensor.  Host indices are
    range-checked here; device indices outside the store give zero rows in the kernel."""

    def __init__(self, store, idx: torch.Tensor, drop=None):
        self.table = store.tensor if isinstance(store, DeviceFeatureStore) else store
        if not torch.is_tensor(idx) or idx.dtype != torch.int32 or idx.dim() not in (1, 2):
            raise ValueError('feature row indices must be an int32 tensor of shape [B] or [B, N]')
        if self.table.dim() != 2 or self.table.dtype not in _STORE_DTYPES:
            raise ValueError('a feature store is a 2-D fp32 / fp16 / bf16 tensor')
        if not idx.is_cuda and idx.numel() and (int(idx.min()) < -1 or int(idx.max()) >= self.table.shape[0]):
            raise IndexError('feature row indices must lie in [-1, %d) (got [%d, %d])'
                             % (self.table.shape[0], int(idx.min()), int(idx.max())))
        self.idx = idx
        self.drop = drop                                      # (p, site) of the environment dropout, set by the host module

    @property
    def shape(self) -> torch.Size:
        return torch.Size(tuple(self.idx.shape) + (self.table.shape[1],))

    @property
    def device(self) -> torch.device:
        return self.table.device

    @property
    def is_cuda(self) -> bool:
        return self.table.is_cuda

    def with_dropout(self, p: float, site: int) -> 'FeatureRows':
        """the same rows with nn.Dropout(p) applied at dropout site ``site`` (autograd_ops.next_site) when gathered"""
        return FeatureRows(self.table, self.idx, (float(p), int(site)))

    def gather(self, dtype, seed: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[rows, feat_dim] of ``dtype`` (vi_gather_rows); ``seed``: the device dropout seed when ``drop`` is set"""
        drop = (self.drop[0], seed, self.drop[1]) if self.drop is not None and self.drop[0] > 0 else None
        return ops.gather_rows(self.table, self.idx.reshape(-1), dtype, drop)

    def dense(self) -> torch.Tensor:
        """the fp32 tensor the dense path would have received (no environment dropout)"""
        return FeatureRows(self.table, self.idx).gather(torch.float32).view(self.shape)


# ----------------------------------------------------------------------------------------------
# CUDA-graph plumbing: the indices are an ordinary graph input, the store is borrowed (read in place, address in the signature)
# ----------------------------------------------------------------------------------------------
def graph_args(name: str, x):
    """(inputs, borrowed) entries of a graphs.GraphedCall for the feature argument ``name``"""
    if isinstance(x, FeatureRows):
        return {name + ':idx': x.idx}, {name + ':store': x.table}
    return ({name: x} if x is not None else {}), {}


def from_graph(t: dict, name: str):
    """the feature argument ``name`` inside a graphed function: a dense tensor or FeatureRows over the borrowed store"""
    if name + ':idx' in t:
        return FeatureRows(t[name + ':store'], t[name + ':idx'])
    return t.get(name)


# ----------------------------------------------------------------------------------------------
# collation: the reference agents' functions with row indices in place of the image features
# ----------------------------------------------------------------------------------------------
def _host(a: np.ndarray, store: DeviceFeatureStore) -> torch.Tensor:
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.pin_memory() if store.device.type == 'cuda' else t


def view_key(ob: dict) -> str:
    """ImageFeaturesDB key of an observation's viewpoint"""
    return '%s_%s' % (ob['scan'], ob['viewpoint'])


def duet_panorama_inputs(store: DeviceFeatureStore, obs: Sequence[dict], n_views: int = 36) -> dict:
    """DUET ``_panorama_feature_variable`` (VLN-DUET/map_nav_src/r2r/agent.py:57-96): candidate views by ``pointId`` first, then
    the remaining of the 36 views in order, padded to the longest panorama.  Same dict, ``view_img_fts`` = FeatureRows; the
    location features are the angle part of the observations' 'feature' arrays (columns feat_dim:) plus the box [1, 1, 1]."""
    F = store.feat_dim
    rows, locs, navs, cand_vpids = [], [], [], []
    for ob in obs:
        base = store.row(view_key(ob))
        used = set()
        r, ang, nav, cv = [], [], [], []
        for cc in ob['candidate']:
            r.append(base + cc['pointId'])
            ang.append(np.asarray(cc['feature'])[F:])
            nav.append(1)
            cv.append(cc['viewpointId'])
            used.add(cc['pointId'])
        feat = ob['feature']
        for k in range(n_views):
            if k not in used:
                r.append(base + k)
                ang.append(np.asarray(feat[k])[F:])
                nav.append(0)
        ang = np.stack(ang, 0).astype(np.float32)
        locs.append(np.concatenate([ang, np.ones((len(r), 3), np.float32)], 1))
        rows.append(r)
        navs.append(nav)
        cand_vpids.append(cv)
    B, V = len(obs), max(len(r) for r in rows)
    idx = np.full((B, V), -1, np.int32)
    loc = np.zeros((B, V, locs[0].shape[1]), np.float32)
    nav_types = np.zeros((B, V), np.int64)
    for b in range(B):
        n = len(rows[b])
        idx[b, :n], loc[b, :n], nav_types[b, :n] = rows[b], locs[b], navs[b]
    return {'view_img_fts': FeatureRows(store, _host(idx, store)), 'loc_fts': _host(loc, store),
            'nav_types': _host(nav_types, store), 'view_lens': _host(np.array([len(r) for r in rows], np.int64), store),
            'cand_vpids': cand_vpids}


def hamt_cand_pano_inputs(store: DeviceFeatureStore, obs: Sequence[dict], n_views: int = 36):
    """HAMT ``_cand_pano_feature_variable`` (VLN-HAMT/finetune_src/r2r/agent_cmt.py): the candidates, the zero [STOP] row (-1),
    then the views no candidate points at, padded to the longest.  Same tuple (ob_img_fts, ob_ang_fts, ob_nav_types, ob_lens,
    ob_cand_lens), ob_img_fts = FeatureRows."""
    F = store.feat_dim
    rows, angs, navs = [], [], []
    for ob in obs:
        base = store.row(view_key(ob))
        cand = np.zeros(n_views, bool)
        r = [base + cc['pointId'] for cc in ob['candidate']]
        ang = [np.asarray(cc['feature'])[F:] for cc in ob['candidate']]
        for cc in ob['candidate']:
            cand[cc['pointId']] = True
        feat = np.asarray(ob['feature'])
        ang_w = feat.shape[1] - F
        r.append(-1)                                          # [STOP]
        ang.append(np.zeros(ang_w, np.float32))
        nav = [1] * len(ob['candidate']) + [2]
        r.extend(base + k for k in range(n_views) if not cand[k])
        ang.extend(feat[~cand][:, F:])
        nav.extend([0] * (n_views - int(cand.sum())))
        rows.append(r)
        angs.append(np.stack(ang, 0).astype(np.float32))
        navs.append(nav)
    B, O = len(obs), max(len(r) for r in rows)
    idx = np.full((B, O), -1, np.int32)
    ang = np.zeros((B, O, angs[0].shape[1]), np.float32)
    nav_types = np.zeros((B, O), np.int64)
    for b in range(B):
        n = len(rows[b])
        idx[b, :n], ang[b, :n], nav_types[b, :n] = rows[b], angs[b], navs[b]
    ob_lens = [len(r) for r in rows]
    ob_cand_lens = [len(ob['candidate']) + 1 for ob in obs]
    return FeatureRows(store, _host(idx, store)), _host(ang, store), _host(nav_types, store), ob_lens, ob_cand_lens


def hamt_history_inputs(store: DeviceFeatureStore, obs: Sequence[dict], actions, n_views: int = 36) -> dict:
    """HAMT's per-step 'history' inputs after choosing ``actions`` (int per episode, an index into the candidates; anything
    else - [STOP], an ended episode, -1 - is no move): ``hist_img_feats`` [B] = the view of the chosen candidate (zero row
    without a move), ``hist_ang_feats`` = its angle features, ``hist_pano_img_feats`` [B, 36] = all views of the viewpoint,
    ``hist_pano_ang_feats`` = their angle features.  Keyword arguments of the 'history' mode, ``ob_step`` aside."""
    F = store.feat_dim
    B = len(obs)
    hist = np.full((B,), -1, np.int32)
    pano = np.empty((B, n_views), np.int32)
    feats = [np.asarray(ob['feature']) for ob in obs]
    ang_w = feats[0].shape[1] - F
    hist_ang = np.zeros((B, ang_w), np.float32)
    pano_ang = np.zeros((B, n_views, ang_w), np.float32)
    for b, ob in enumerate(obs):
        base = store.row(view_key(ob))
        a = int(actions[b])
        if 0 <= a < len(ob['candidate']):
            cc = ob['candidate'][a]
            hist[b] = base + cc['pointId']
            hist_ang[b] = np.asarray(cc['feature'])[F:]
        pano[b] = base + np.arange(n_views)
        pano_ang[b] = feats[b][:n_views, F:]
    return {'hist_img_feats': FeatureRows(store, _host(hist, store)), 'hist_ang_feats': _host(hist_ang, store),
            'hist_pano_img_feats': FeatureRows(store, _host(pano, store)), 'hist_pano_ang_feats': _host(pano_ang, store)}


def imagination_inputs(store: DeviceFeatureStore, instr_ids: Sequence[str], generated_flags: Mapping[str, List[str]]):
    """imagine_db.collate_imaginations with rows of ``store`` (keys = instruction ids): slot k of episode i is the next unread
    row of its key iff flag k is 'True' (holes are -1), the slot count is the number of sub-instructions, an instruction whose
    flags are all 'False' has length 0.  Returns (FeatureRows [B, max_subinstr], imagine_mask bool [B, max_subinstr])."""
    lens = []
    for iid in instr_ids:
        flags = generated_flags[iid]
        lens.append(0 if flags.count('False') == len(flags) else len(flags))
    width = max(lens) if lens else 0
    idx = np.full((len(instr_ids), width), -1, np.int32)
    mask = np.zeros((len(instr_ids), width), dtype=bool)
    for i, iid in enumerate(instr_ids):
        if lens[i] == 0:
            continue
        flags = [f == 'True' for f in generated_flags[iid]]
        mask[i, :len(flags)] = flags
        start, n = store.span(iid)
        if n != sum(flags):
            raise AssertionError('%s: %d feature rows for %d generated imaginations' % (iid, n, sum(flags)))
        k = 0
        for slot, f in enumerate(flags):
            if f:
                idx[i, slot] = start + k
                k += 1
    return FeatureRows(store, _host(idx, store)), mask
