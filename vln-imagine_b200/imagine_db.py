"""Imagination feature loader with the reference's key / shape / slot semantics.

Reference: ``ImaginationImageFeaturesDB.get_image_feature`` (VLN-DUET/map_nav_src/r2r/data_utils.py:52-67, the
byte-identical copy in VLN-HAMT/finetune_src/r2r/data_utils.py:32-47) and the agent-side collation
``_create_diffusion_imaginations_v2`` (VLN-DUET/map_nav_src/r2r/agent.py:317-382).

The reference reads an HDF5 file through h5py (not installed here, SURVEY.md section 8 A12); the store is therefore
pluggable: any mapping ``key -> (n_valid_imaginations, >= image_feat_size) array`` - an ``h5py.File`` when h5py is
available, an ``.npz`` archive, or a dict.  Key = ``"<path_id>_<instr_idx>"``; rows are sliced to
``image_feat_size`` columns, cast to float32 and cached, exactly like the reference.
"""
from __future__ import annotations

from typing import Dict, List, Mapping, Sequence, Tuple

import numpy as np


def open_source(src) -> Mapping:
    """a mapping ``key -> array`` for a dict (returned as is), an .npz path or an HDF5 path (needs h5py); the caller closes
    what it opened"""
    if isinstance(src, Mapping):
        return src
    if isinstance(src, str) and src.endswith('.npz'):
        return np.load(src)
    try:
        import h5py
    except ImportError as e:                                      # pragma: no cover
        raise ImportError('reading %r needs h5py; pass a dict or an .npz archive instead' % (src,)) from e
    return h5py.File(src, 'r')


class ImaginationImageFeaturesDB(object):
    def __init__(self, img_ft_file, image_feat_size: int):
        self.image_feat_size = image_feat_size
        self.img_ft_file = img_ft_file
        self._feature_store: Dict[str, np.ndarray] = {}

    def _open(self) -> Mapping:
        return open_source(self.img_ft_file)

    def get_image_feature(self, path_id_instr_idx: str) -> np.ndarray:
        key = path_id_instr_idx
        ft = self._feature_store.get(key)
        if ft is None:
            store = self._open()
            try:
                ft = np.asarray(store[key][...])[:, :self.image_feat_size].astype(np.float32)
            finally:
                if hasattr(store, 'close') and not isinstance(self.img_ft_file, Mapping):
                    store.close()
            self._feature_store[key] = ft
        return ft


def collate_imaginations(db: ImaginationImageFeaturesDB, instr_ids: Sequence[str],
                         generated_flags: Mapping[str, List[str]], image_feat_size: int) -> Tuple[np.ndarray, np.ndarray]:
    """(imagined_diff_img_feats (B, max_subinstr, F) f32, imagine_mask (B, max_subinstr) bool).

    Slot k of episode i holds the next unread feature row iff flag k is 'True'; the slot count is the number of
    SUB-INSTRUCTIONS (so the mask can have 'False' holes), and an instruction whose flags are all 'False'
    contributes length 0 and all-zero rows (agent.py:334-371)."""
    lens = []
    for iid in instr_ids:
        flags = generated_flags[iid]
        lens.append(0 if flags.count('False') == len(flags) else len(flags))
    width = max(lens) if lens else 0
    feats = np.zeros((len(instr_ids), width, image_feat_size), np.float32)
    mask = np.zeros((len(instr_ids), width), dtype=bool)
    for i, iid in enumerate(instr_ids):
        if lens[i] == 0:
            continue
        flags = [f == 'True' for f in generated_flags[iid]]
        mask[i, :len(flags)] = flags
        rows = db.get_image_feature(iid)
        if rows.shape[0] != sum(flags):
            raise AssertionError('%s: %d feature rows for %d generated imaginations' % (iid, rows.shape[0], sum(flags)))
        k = 0
        for slot, f in enumerate(flags):
            if f:
                feats[i, slot] = rows[k]
                k += 1
    return feats, mask
