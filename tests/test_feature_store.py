"""Host side of the device-resident feature store (vln-imagine_b200/feature_store.py): key -> row mapping, loading, index checks,
and the collation helpers against restatements of the reference agents' functions on synth.nav_world observations (store on
the CPU; the gather kernel itself is tested in test_feature_store_gpu.py)."""
import importlib

import numpy as np
import pytest
import torch

fs = importlib.import_module('vln_imagine_b200.feature_store')
synth = importlib.import_module('vln_imagine_b200.synth')
imagine_db = importlib.import_module('vln_imagine_b200.imagine_db')

F, A, V = 16, 4, 36              # image feature size, angle feature size, views


def _db(names, seed=0, width=F + 8):
    g = np.random.default_rng(seed)
    return {'scan0_%s' % n: g.standard_normal((V, width)).astype(np.float32) for n in names}


def _obs(seed=3, steps=3, batch=5):
    """nav_world observations with what the reference env adds: scan, per-candidate pointId (two candidates may share one),
    the (36, F + 4) 'feature' array of the viewpoint and each candidate's (F + 4) 'feature'"""
    world = synth.nav_world(seed=seed, batch=batch, steps=steps)
    names = sorted({ob['viewpoint'] for st in world for ob in st['obs']} |
                   {c['viewpointId'] for st in world for ob in st['obs'] for c in ob['candidate']})
    db = _db(names)
    g = np.random.default_rng(seed)
    out = []
    for st in world:
        obs = []
        for ob in st['obs']:
            feat = np.concatenate([db['scan0_' + ob['viewpoint']][:, :F], g.standard_normal((V, A)).astype(np.float32)], 1)
            cands = []
            for c in ob['candidate']:
                pid = int(g.integers(0, V))
                cands.append(dict(c, pointId=pid, feature=np.concatenate([feat[pid, :F], g.standard_normal(A).astype(np.float32)])))
            if len(cands) > 1:
                cands[-1]['pointId'] = cands[0]['pointId']          # a shared pointId
                cands[-1]['feature'] = np.concatenate([feat[cands[0]['pointId'], :F], cands[-1]['feature'][F:]])
            obs.append(dict(ob, scan='scan0', feature=feat, candidate=cands))
        out.append(obs)
    return out, db


def _rows(store, idx):
    t = store.tensor.numpy()
    idx = idx.numpy()
    return np.where((idx >= 0)[..., None], t[np.maximum(idx, 0)], 0)


# ---- restatements of the reference agents (VLN-DUET r2r/agent.py:57-96, VLN-HAMT r2r/agent_cmt.py) ----------------------
def _ref_duet_pano(obs):
    img, loc, nav, lens, cvp = [], [], [], [], []
    for ob in obs:
        vi, va, nt, cv, used = [], [], [], [], set()
        for cc in ob['candidate']:
            vi.append(cc['feature'][:F]); va.append(cc['feature'][F:]); nt.append(1); cv.append(cc['viewpointId'])
            used.add(cc['pointId'])
        vi.extend([x[:F] for k, x in enumerate(ob['feature']) if k not in used])
        va.extend([x[F:] for k, x in enumerate(ob['feature']) if k not in used])
        nt.extend([0] * (36 - len(used)))
        vi, va = np.stack(vi, 0), np.stack(va, 0)
        img.append(vi); loc.append(np.concatenate([va, np.ones((len(vi), 3), np.float32)], 1)); nav.append(nt)
        lens.append(len(vi)); cvp.append(cv)
    n = max(lens)
    pad = lambda a: np.concatenate([a, np.zeros((n - len(a),) + a.shape[1:], a.dtype)], 0)   # noqa: E731
    return {'view_img_fts': np.stack([pad(a) for a in img]), 'loc_fts': np.stack([pad(a) for a in loc]),
            'nav_types': np.stack([pad(np.array(t, np.int64)) for t in nav]), 'view_lens': np.array(lens), 'cand_vpids': cvp}


def _ref_hamt_cand_pano(obs):
    img, ang, nav, lens = [], [], [], []
    for ob in obs:
        ci, ca, cn = [], [], []
        cp = np.zeros((36,), dtype=bool)
        for cc in ob['candidate']:
            ci.append(cc['feature'][:F]); ca.append(cc['feature'][F:]); cp[cc['pointId']] = True; cn.append(1)
        ci.append(np.zeros((F,), np.float32)); ca.append(np.zeros((A,), np.float32)); cn.append(2)
        pano = ob['feature'][~cp]
        img.append(np.concatenate([np.vstack(ci), pano[:, :F]], 0)); ang.append(np.concatenate([np.vstack(ca), pano[:, F:]], 0))
        cn.extend([0] * (36 - np.sum(cp))); nav.append(cn); lens.append(len(cn))
    n = max(lens)
    pad = lambda a: np.concatenate([a, np.zeros((n - len(a),) + a.shape[1:], a.dtype)], 0)   # noqa: E731
    return (np.stack([pad(a) for a in img]), np.stack([pad(a) for a in ang]), np.stack([pad(np.array(t, np.int64)) for t in nav]),
            lens, [len(ob['candidate']) + 1 for ob in obs])


# ---- tests --------------------------------------------------------------------------------------------------------------
def test_key_rows_slicing_and_growth():
    a = np.arange(36 * 20, dtype=np.float32).reshape(36, 20)
    b = np.full((3, 17), 2.5, np.float32)
    s = fs.DeviceFeatureStore('cpu', F, torch.float32).add({'a': a})
    assert (s.n_rows, s.span('a'), s.row('a', 5)) == (36, (0, 36), 5)
    t0 = s.tensor
    s.add({'a': a * 0, 'b': b})                                    # a known key is kept, a new one appended
    assert s.tensor is not t0 and s.n_rows == 39 and s.span('b') == (36, 3) and len(s) == 2 and 'b' in s
    np.testing.assert_array_equal(s.tensor[:36].numpy(), a[:, :F])
    np.testing.assert_array_equal(s.tensor[36:].numpy(), b[:, :F])
    with pytest.raises(KeyError):
        s.row('nope')
    with pytest.raises(IndexError):
        s.row('b', 3)
    with pytest.raises(ValueError):
        s.add({'c': np.zeros((2, F - 8), np.float32)})             # fewer columns than feat_dim


def test_npz_source_and_half_storage(tmp_path):
    g = np.random.default_rng(1)
    arrs = {'k%d' % i: g.standard_normal((4, 24)).astype(np.float32) for i in range(3)}
    np.savez(tmp_path / 'f.npz', **arrs)
    s = fs.DeviceFeatureStore.load(str(tmp_path / 'f.npz'), 'cpu', F, torch.float16, keys=['k2', 'k0'])
    assert s.dtype == torch.float16 and s.span('k2') == (0, 4) and s.span('k0') == (4, 4) and 'k1' not in s
    np.testing.assert_array_equal(s.tensor[4:8].numpy(), arrs['k0'][:, :F].astype(np.float16))


def test_feature_rows_shape_and_range_check():
    s = fs.DeviceFeatureStore('cpu', F, torch.float32).add({'a': np.zeros((5, F), np.float32)})
    r = fs.FeatureRows(s, torch.tensor([[0, 4, -1]], dtype=torch.int32))
    assert r.shape == (1, 3, F) and fs.FeatureRows(s, torch.zeros(7, dtype=torch.int32)).shape == (7, F)
    for bad in ([5], [-2]):
        with pytest.raises(IndexError):
            fs.FeatureRows(s, torch.tensor(bad, dtype=torch.int32))
    with pytest.raises(ValueError):
        fs.FeatureRows(s, torch.tensor([0], dtype=torch.int64))


def test_duet_panorama_rows_follow_the_agent():
    steps, db = _obs()
    s = fs.DeviceFeatureStore('cpu', F, torch.float32).add(db)
    for obs in steps:
        got, ref = fs.duet_panorama_inputs(s, obs), _ref_duet_pano(obs)
        assert isinstance(got['view_img_fts'], fs.FeatureRows)
        np.testing.assert_array_equal(_rows(s, got['view_img_fts'].idx), ref['view_img_fts'])
        np.testing.assert_array_equal(got['loc_fts'].numpy(), ref['loc_fts'])
        np.testing.assert_array_equal(got['nav_types'].numpy(), ref['nav_types'])
        np.testing.assert_array_equal(got['view_lens'].numpy(), ref['view_lens'])
        assert got['cand_vpids'] == ref['cand_vpids']
        assert (got['view_img_fts'].idx.numpy()[np.arange(ref['view_img_fts'].shape[1])[None] >= ref['view_lens'][:, None]] == -1).all()


def test_hamt_cand_pano_and_history_rows_follow_the_agent():
    steps, db = _obs(seed=4)
    s = fs.DeviceFeatureStore('cpu', F, torch.float32).add(db)
    g = np.random.default_rng(0)
    for obs in steps:
        rows, ang, nav, lens, clens = fs.hamt_cand_pano_inputs(s, obs)
        r_img, r_ang, r_nav, r_lens, r_clens = _ref_hamt_cand_pano(obs)
        np.testing.assert_array_equal(_rows(s, rows.idx), r_img)
        np.testing.assert_array_equal(ang.numpy(), r_ang)
        np.testing.assert_array_equal(nav.numpy(), r_nav)
        assert (lens, clens) == (r_lens, r_clens)
        # history after acting: the chosen candidate's view (zero row for [STOP] / no move), all 36 views of the viewpoint
        a_t = [int(g.integers(-1, len(ob['candidate']) + 1)) for ob in obs]
        h = fs.hamt_history_inputs(s, obs, a_t)
        ref_hist = np.stack([r_img[b, a] if 0 <= a < len(obs[b]['candidate']) else np.zeros(F, np.float32) for b, a in enumerate(a_t)])
        np.testing.assert_array_equal(_rows(s, h['hist_img_feats'].idx), ref_hist)
        np.testing.assert_array_equal(_rows(s, h['hist_pano_img_feats'].idx), np.stack([ob['feature'][:, :F] for ob in obs]))
        np.testing.assert_array_equal(h['hist_pano_ang_feats'].numpy(), np.stack([ob['feature'][:, F:] for ob in obs]))
        ref_ang = np.stack([obs[b]['candidate'][a]['feature'][F:] if 0 <= a < len(obs[b]['candidate']) else np.zeros(A, np.float32)
                            for b, a in enumerate(a_t)])
        np.testing.assert_array_equal(h['hist_ang_feats'].numpy(), ref_ang)


def test_imagination_slots_match_collate_imaginations():
    g = np.random.default_rng(2)
    flags = {'p0_0': ['True', 'False', 'True'], 'p1_0': ['False', 'False'], 'p2_1': ['True'], 'p3_2': ['False', 'True', 'True', 'False']}
    feats = {k: g.standard_normal((v.count('True'), F + 4)).astype(np.float32) for k, v in flags.items() if v.count('True')}
    db = imagine_db.ImaginationImageFeaturesDB(feats, F)
    s = fs.DeviceFeatureStore('cpu', F, torch.float32).add(feats)
    for ids in (['p0_0', 'p1_0', 'p2_1', 'p3_2'], ['p1_0'], ['p2_1', 'p0_0']):
        ref, ref_mask = imagine_db.collate_imaginations(db, ids, flags, F)
        rows, mask = fs.imagination_inputs(s, ids, flags)
        assert rows.shape == ref.shape
        np.testing.assert_array_equal(mask, ref_mask)
        np.testing.assert_array_equal(_rows(s, rows.idx), ref)
    with pytest.raises(AssertionError):
        fs.imagination_inputs(s, ['p0_0'], {'p0_0': ['True', 'True', 'True']})
