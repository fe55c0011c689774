"""Per-step graph glue (SURVEY.md section 8(f), N1 / N2).

CPU: oracle/graph_oracle.py replayed on the synthetic rollout against tests/golden/graph_world.npz, which holds the
outputs of the REAL reference GraphMap / FloydGraph (oracle/gen_graph_golden.py).
GPU: vln_imagine_b200.graph_map.DeviceGraphMaps (csrc/vi_graph.cu through the C ABI) against the same fixture and,
at hidden size 768 and a larger world, against the oracle.  Integer outputs, distances, path-length and distance
features are bit-exact; sin / cos of the fp32-cast angles within 1e-6 (numpy and CUDA round differently); the masked
panorama mean within 1e-6 relative (summation order)."""
import importlib
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

synth = importlib.import_module('vln_imagine_b200.synth')
ANGLE_TOL = 1e-6


def _world():
    meta = json.load(open(os.path.join(GOLDEN, 'graph_oracle_vs_reference.json')))
    assert meta['max_abs_diff_oracle_vs_reference'] == 0.0
    return synth.nav_world(**meta['world']), np.load(os.path.join(GOLDEN, 'graph_world.npz'))


def _cands(ob):
    return [(c['viewpointId'], c['position']) for c in ob['candidate']]


def _oracle_rollout(world, hidden):
    """yields (t, step, gmap dict, vp dict) exactly as oracle/gen_graph_golden.py drives the reference"""
    from oracle import graph_oracle as GO
    obs0 = world[0]['obs']
    B = len(obs0)
    states = [GO.GraphState(ob['viewpoint'], hidden) for ob in obs0]
    for b, ob in enumerate(obs0):
        states[b].update_graph(ob['viewpoint'], ob['position'], _cands(ob))
    for t, step in enumerate(world):
        obs, ended = step['obs'], step['ended']
        cur = [st.index[ob['viewpoint']] for st, ob in zip(states, obs)]
        cands = [[st.index[c['viewpointId']] for c in ob['candidate']] for st, ob in zip(states, obs)]
        for b, st in enumerate(states):
            if not ended[b]:
                st.step_id[cur[b]] = t + 1
        V = step['pano_embeds'].shape[1]
        GO.update_node_embeds(states, cur, cands, step['pano_embeds'], np.ones((B, V), bool), ended)
        heads, elevs = [ob['heading'] for ob in obs], [ob['elevation'] for ob in obs]
        og = GO.nav_gmap_variable(states, cur, heads, elevs)
        ov = GO.nav_vp_variable(states, cur, heads, elevs, step['pano_embeds'], cands, step['view_lens'], step['nav_types'])
        og['names'] = [[None if v < 0 else states[b].names[v] for v in og['gmap_nodes'][b, :og['gmap_lens'][b]]] for b in range(B)]
        yield t, step, og, ov
        if t + 1 < len(world):
            for b, ob in enumerate(world[t + 1]['obs']):
                if not ended[b]:
                    states[b].update_graph(ob['viewpoint'], ob['position'], _cands(ob))


def test_graph_oracle_matches_reference_golden():
    world, gold = _world()
    for t, step, og, ov in _oracle_rollout(world, hidden=8):
        for k_o, k_e in (('gmap_nodes', 'nodes'), ('gmap_img_embeds', 'emb'), ('gmap_pos_fts', 'pos'), ('gmap_pair_dists', 'pair'),
                         ('gmap_step_ids', 'step_ids'), ('gmap_visited_masks', 'visited'), ('gmap_lens', 'lens')):
            assert np.array_equal(og[k_o], gold['t%d_%s' % (t, k_e)]), (t, k_o)
        assert np.array_equal(ov['vp_pos_fts'], gold['t%d_vp_pos' % t]), t


def test_graph_oracle_edge_cases():
    """unreached pairs keep the reference's sentinel, a start viewpoint seen from itself, an episode with one node"""
    from oracle import graph_oracle as GO
    st = GO.GraphState('a', 4)
    st.update_graph('a', (0.0, 0.0, 0.0), [])
    f = st.pos_fts(0, [-1, 0], 0.3, -0.1)
    assert np.array_equal(f[0], np.array([0, 1, 0, 1, 0, 0, 0], np.float32))
    assert f[1, 5] == 0 and f[1, 6] == 0 and abs(f[1, 4] - 1e-8 / 30) < 1e-12
    st.update_graph('a', (0.0, 0.0, 0.0), [('b', (3.0, 4.0, 0.0))])
    st.node('c', (9.0, 9.0, 9.0))                              # known position, no edge: never reached
    assert st.distance(0, 1) == 5.0 and st.distance(1, 2) == GO.UNREACHED and st.path_len(1, 2) == 1


def test_device_graph_maps_host_bookkeeping_without_a_gpu(monkeypatch):
    """The host side of DeviceGraphMaps (viewpoint interning, [stop] + visited + unvisited ordering, step ids, masks, the id
    tensors handed to the fusion kernel, the index arrays the kernels receive) against the oracle, with the library calls
    stubbed out: everything that is NOT arithmetic is checked on the CPU."""
    from oracle import graph_oracle as GO
    gm_mod = importlib.import_module('vln_imagine_b200.graph_map')
    ops = importlib.import_module('vln_imagine_b200.ops')

    calls = []

    class FakeLib:
        def __getattr__(self, name):
            def f(*a):
                calls.append(name)
                return 0
            return f
    monkeypatch.setattr(gm_mod, 'lib', FakeLib())
    monkeypatch.setattr(ops, 'ensure_init', lambda t: None)
    monkeypatch.setattr(ops, '_stream', lambda: 0)
    monkeypatch.setattr(torch.Tensor, 'pin_memory', lambda self: self)
    packed = {}
    real_pack = gm_mod._pack

    def spy_pack(staging, device, arrays):
        packed.update({k: np.array(v) for k, v in arrays.items()})
        return real_pack(staging, device, arrays)
    monkeypatch.setattr(gm_mod, '_pack', spy_pack)

    world = synth.nav_world(seed=31, n_vp=40, batch=5, steps=6, hidden=8)
    gm = gm_mod.DeviceGraphMaps(world[0]['obs'], 'cpu', hidden=8)
    for t, step, og, ov in _oracle_rollout(world, 8):
        obs, ended = step['obs'], step['ended']
        gm.set_step_ids(obs, t, ended)
        pano = torch.from_numpy(step['pano_embeds'])
        pin = {'cand_vpids': [[c['viewpointId'] for c in ob['candidate']] for ob in obs],
               'view_lens': torch.from_numpy(step['view_lens']), 'nav_types': torch.from_numpy(step['nav_types'])}
        out = gm.nav_inputs(obs, pano, torch.ones(pano.shape[:2], dtype=torch.bool), pin, ended)
        B, G = og['gmap_masks'].shape
        assert out['gmap_vpids'] == og['names'] and out['no_vp_left'] == og['no_vp_left'], t
        assert np.array_equal(out['gmap_step_ids'].numpy(), og['gmap_step_ids']), t
        assert np.array_equal(out['gmap_visited_masks'].numpy(), og['gmap_visited_masks']), t
        assert np.array_equal(out['gmap_masks'].numpy(), og['gmap_masks']), t
        assert np.array_equal(out['vp_masks'].numpy(), ov['vp_masks']) and np.array_equal(out['vp_nav_masks'].numpy(), ov['vp_nav_masks']), t
        assert out['vp_cand_vpids'] == [[None] + c for c in pin['cand_vpids']], t
        # index arrays the kernels receive: node order, candidates, current / start nodes, lengths
        assert np.array_equal(packed['gnode'], og['gmap_nodes']) and np.array_equal(packed['lens'], og['gmap_lens']), t
        assert packed['cur'].tolist() == [(-1 if e else gm.index[b][ob['viewpoint']]) for b, (ob, e) in enumerate(zip(obs, ended))], t
        assert packed['start'].tolist() == [gm.index[b][gm.start_vps[b]] for b in range(B)], t
        for b, vps in enumerate(pin['cand_vpids']):
            assert packed['cand'][b, :len(vps)].tolist() == [gm.index[b][v] for v in vps] and (packed['cand'][b, len(vps):] == -1).all(), t
        # interned ids for the fusion kernel: equal strings <-> equal ids inside an episode, [stop] and padding as documented
        gids, cids = out['gmap_vpids'].ids.numpy(), out['vp_cand_vpids'].ids.numpy()
        assert (gids[:, 0] == gm_mod.STOP_ID).all() and (cids[:, 0] == gm_mod.STOP_ID).all()
        for b in range(B):
            row = og['names'][b]
            assert (gids[b, len(row):] == -1).all() and (cids[b, 1 + len(pin['cand_vpids'][b]):] == -2).all()
            for j, vp in enumerate(row[1:], 1):
                for k, cvp in enumerate(pin['cand_vpids'][b], 1):
                    assert (gids[b, j] == cids[b, k]) == (vp == cvp)
        if t + 1 < len(world):
            gm.update_graph(world[t + 1]['obs'], ended)
            nxt = world[t + 1]['obs']
            assert packed['cur'].tolist() == [(-1 if e else gm.index[b][ob['viewpoint']]) for b, (ob, e) in enumerate(zip(nxt, ended))]
            assert packed['n_nodes'].tolist() == [len(n) for n in gm.names]
    assert {'vi_graph_init', 'vi_graph_update', 'vi_graph_embed_step', 'vi_graph_features'} <= set(calls)


def _run_device(world, hidden, check):
    from vln_imagine_b200 import graph_map
    dev = torch.device('cuda')
    obs0 = world[0]['obs']
    gm = graph_map.DeviceGraphMaps(obs0, dev, hidden=hidden)
    for t, step, og, ov in _oracle_rollout(world, hidden):
        obs, ended = step['obs'], step['ended']
        gm.set_step_ids(obs, t, ended)
        pano = torch.from_numpy(step['pano_embeds']).to(dev)
        masks = torch.ones(pano.shape[:2], dtype=torch.bool, device=dev)
        pin = {'cand_vpids': [[c['viewpointId'] for c in ob['candidate']] for ob in obs],
               'view_lens': torch.from_numpy(step['view_lens']).to(dev), 'nav_types': torch.from_numpy(step['nav_types']).to(dev)}
        out = gm.nav_inputs(obs, pano, masks, pin, ended)
        check(t, out, og, ov)
        if t + 1 < len(world):
            gm.update_graph(world[t + 1]['obs'], ended)
    return gm


def _compare(t, out, og, ov):
    assert out['gmap_vpids'] == og['names'], t
    c = {k: v.cpu().numpy() for k, v in out.items() if torch.is_tensor(v)}
    assert np.array_equal(c['gmap_step_ids'], og['gmap_step_ids']), t
    assert np.array_equal(c['gmap_visited_masks'], og['gmap_visited_masks']), t
    assert np.array_equal(c['gmap_masks'], og['gmap_masks']), t
    assert out['no_vp_left'] == og['no_vp_left'], t
    assert np.array_equal(c['gmap_pair_dists'], og['gmap_pair_dists']), t          # fp64 relax, one cast: bit-exact
    assert np.array_equal(c['gmap_pos_fts'][..., 4:], og['gmap_pos_fts'][..., 4:]), t
    assert np.abs(c['gmap_pos_fts'][..., :4] - og['gmap_pos_fts'][..., :4]).max() <= ANGLE_TOL, t
    assert np.array_equal(c['vp_pos_fts'][..., [4, 5, 6, 11, 12, 13]], ov['vp_pos_fts'][..., [4, 5, 6, 11, 12, 13]]), t
    assert np.abs(c['vp_pos_fts'] - ov['vp_pos_fts']).max() <= ANGLE_TOL, t
    assert np.array_equal(c['vp_img_embeds'], ov['vp_img_embeds']), t
    assert np.array_equal(c['vp_masks'], ov['vp_masks']) and np.array_equal(c['vp_nav_masks'], ov['vp_nav_masks']), t
    ref = og['gmap_img_embeds']
    assert np.abs(c['gmap_img_embeds'] - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max()), t


@pytest.mark.gpu
def test_device_graph_maps_match_reference_golden(lib_built):
    """hidden = 8 world of the fixture: the kernels against the REAL reference's outputs"""
    world, gold = _world()

    def check(t, out, og, ov):
        _compare(t, out, og, ov)
        c = out['gmap_pair_dists'].cpu().numpy()
        assert np.array_equal(c, gold['t%d_pair' % t]), t
        assert np.array_equal(out['gmap_pos_fts'].cpu().numpy()[..., 4:], gold['t%d_pos' % t][..., 4:]), t
        assert np.abs(out['gmap_pos_fts'].cpu().numpy() - gold['t%d_pos' % t]).max() <= ANGLE_TOL, t
        assert np.abs(out['vp_pos_fts'].cpu().numpy() - gold['t%d_vp_pos' % t]).max() <= ANGLE_TOL, t
        assert np.abs(out['gmap_img_embeds'].cpu().numpy() - gold['t%d_emb' % t]).max() <= 1e-6 * 4, t
    _run_device(world, 8, check)


@pytest.mark.gpu
@pytest.mark.parametrize('seed,n_vp,batch,steps', [(11, 60, 16, 10), (12, 100, 8, 15)])
def test_device_graph_maps_match_oracle_hidden768(lib_built, seed, n_vp, batch, steps):
    """batch of long rollouts over larger graphs (up to ~60 known nodes per episode) at the model's hidden size"""
    world = synth.nav_world(seed=seed, n_vp=n_vp, batch=batch, steps=steps, hidden=768, degree=4)
    gm = _run_device(world, 768, _compare)
    # distances are symmetric and every visited node is at distance > 0 from every other known node
    n = len(gm.names[0])
    d = gm.dis[0, :n, :n].cpu().numpy()
    assert np.array_equal(d, d.T) and (d[~np.eye(n, dtype=bool)] > 0).all()


@pytest.mark.gpu
def test_rollout_glue_feeds_the_navigation_call(lib_built):
    """The dict DeviceGraphMaps.nav_inputs returns goes straight into model('navigation', ...) - device tensors plus the
    pre-interned viewpoint ids - and must score actions exactly like the inputs the reference agent would have collated
    on the host (oracle arrays, lists of id strings interned by the model)."""
    import dataclasses
    from parity_utils import manifest, max_rel
    duet = importlib.import_module('vln_imagine_b200.duet')
    config = importlib.import_module('vln_imagine_b200.config')
    graph_map = importlib.import_module('vln_imagine_b200.graph_map')
    B = 6
    world = synth.nav_world(seed=5, n_vp=30, batch=B, steps=4, hidden=768)
    model = duet.VLNBert(config.default_duet_args()).cuda().eval()
    model.vln_bert.load_state_dict(synth.synth_state_dict(manifest('duet'), seed=0, gasa_stress=True))
    model.vln_bert.precision = 'fp32'      # the two input sets differ by ~1e-6 (sin / cos, mean order): fp32 mode keeps it visible
    ep = synth.to_torch(synth.duet_episode(dataclasses.replace(synth.TINY, batch=B), 3))
    dev = torch.device('cuda')
    with torch.no_grad():
        txt = model('language', {'txt_ids': ep['txt_ids'].to(dev), 'txt_masks': ep['txt_masks'].to(dev)})
        img = model('imagine', {'imagine_feats': ep['imagine_feats'].to(dev), 'imagine_masks': None})
        common = {'txt_embeds': txt, 'txt_masks': ep['txt_masks'].to(dev), 'imagine_embeds': img,
                  'imagine_masks': ep['imagine_masks'].to(dev)}
        gm = graph_map.DeviceGraphMaps(world[0]['obs'], dev)
        for t, step, og, ov in _oracle_rollout(world, 768):
            obs, ended = step['obs'], step['ended']
            gm.set_step_ids(obs, t, ended)
            pano = torch.from_numpy(step['pano_embeds']).to(dev)
            pin = {'cand_vpids': [[c['viewpointId'] for c in ob['candidate']] for ob in obs],
                   'view_lens': torch.from_numpy(step['view_lens']).to(dev), 'nav_types': torch.from_numpy(step['nav_types']).to(dev)}
            a = gm.nav_inputs(obs, pano, torch.ones(pano.shape[:2], dtype=torch.bool, device=dev), pin, ended)
            assert torch.is_tensor(a['gmap_vpids'].ids) and torch.is_tensor(a['vp_cand_vpids'].ids)
            out_a = model('navigation', {**common, **{k: v for k, v in a.items() if k != 'no_vp_left'}})
            host = {'gmap_vpids': og['names'], 'vp_cand_vpids': [[None] + c for c in pin['cand_vpids']]}
            for k in ('gmap_img_embeds', 'gmap_step_ids', 'gmap_pos_fts', 'gmap_masks', 'gmap_pair_dists', 'gmap_visited_masks'):
                host[k] = torch.from_numpy(og[k]).to(dev)
            for k in ('vp_img_embeds', 'vp_pos_fts', 'vp_masks', 'vp_nav_masks'):
                host[k] = torch.from_numpy(ov[k]).to(dev)
            out_b = model('navigation', {**common, **host})
            for k in ('global_logits', 'local_logits', 'fused_logits'):
                assert max_rel(out_a[k], out_b[k]) < 1e-4, (t, k)
            assert torch.equal(out_a['fused_logits'].argmax(-1), out_b['fused_logits'].argmax(-1)), t
            if t + 1 < len(world):
                gm.update_graph(world[t + 1]['obs'], ended)
