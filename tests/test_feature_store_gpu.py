"""The device-resident feature store on the GPU: vi_gather_rows bit for bit against torch indexing + vi_dropout + vi_cast_h16, and
every mode that takes image features giving bit-identical outputs with FeatureRows and with the dense tensor rows.dense() -
eager, graph-replayed (new indices, a store that grew), in the fp32 / fp16 / bf16 operand formats, and in training with the
environment dropout on (the loss and every parameter gradient bit for bit, except the gradients that the dense path itself sums
in a run-dependent order - see _compare_training)."""
import importlib

import numpy as np
import pytest
import torch

from parity_utils import manifest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mods(lib_built):
    m = {n: importlib.import_module('vln_imagine_b200.' + n) for n in ('ops', 'feature_store', 'synth', 'config', 'duet', 'hamt',
                                                                       'autograd_ops')}
    m['ops'].ensure_init(torch.zeros(1, device='cuda'))
    return m


def _bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _store(fs, n_rows, F, dtype, seed=0):
    g = np.random.default_rng(seed)
    a = (g.standard_normal((n_rows, F)) * 3).astype(np.float32)
    a[0, :8] = [70000.0, -70000.0, 1e-8, -0.0, 65504.0, 3e38, -3e38, 0.5]     # saturation / subnormal / signed-zero columns
    return fs.DeviceFeatureStore('cuda', F, dtype).add({'k%d' % i: a[i * 16:(i + 1) * 16] for i in range((n_rows + 15) // 16)})


@pytest.mark.parametrize('F', [512, 768, 2048])
@pytest.mark.parametrize('store_dtype', [torch.float32, torch.float16, torch.bfloat16])
def test_gather_rows_kernel_bitwise(mods, F, store_dtype):
    ops, fs, ag = mods['ops'], mods['feature_store'], mods['autograd_ops']
    s = _store(fs, 96, F, store_dtype, seed=F)
    n = s.n_rows
    g = torch.Generator().manual_seed(F)
    for rows in (1, 37, 2367):
        idx = torch.randint(0, n, (rows,), generator=g, dtype=torch.int32)
        idx[::5] = -1
        idx[1::7] = n + 3                                          # out of range: zero rows as well
        idx[2::11] = -1000
        if rows > 2:
            idx[-1] = 0                                            # the saturating row
        d_idx = idx.cuda()
        valid = ((idx >= 0) & (idx < n)).cuda()[:, None]
        ref32 = torch.where(valid, s.tensor[d_idx.clamp(0, n - 1).long()].float(), torch.zeros((), device='cuda'))
        seed = ag.dropout_seed(torch.device('cuda'))
        for drop in (None, (0.3, seed, 77)):
            ref = ops.dropout(ref32, drop[0], seed, drop[2]) if drop else ref32
            assert _same(ops.gather_rows(s.tensor, d_idx, torch.float32, drop), ref), (rows, drop)
            for out in (torch.float16, torch.bfloat16):
                assert _same(ops.gather_rows(s.tensor, d_idx, out, drop), ops.cast_h16(ref, dtype=out)), (rows, drop, out)


def test_empty_selection_gathers_nothing(mods):
    """imagination slots of width 0 (every instruction's flags 'False') and an empty store: no rows, no error"""
    ops, fs = mods['ops'], mods['feature_store']
    s = _store(fs, 32, 768, torch.float16)
    rows, mask = fs.imagination_inputs(s, ['a', 'b'], {'a': ['False', 'False'], 'b': ['False']})
    assert rows.shape == (2, 0, 768) and mask.shape == (2, 0)
    assert rows.dense().shape == (2, 0, 768)
    for dtype in (torch.float32, torch.float16, torch.bfloat16):
        assert ops.gather_rows(s.tensor, torch.empty(0, dtype=torch.int32, device='cuda'), dtype).shape == (0, 768)
    empty = fs.DeviceFeatureStore('cuda', 768, torch.float16)
    out = ops.gather_rows(empty.tensor, torch.tensor([-1, 0, 5], dtype=torch.int32, device='cuda'), torch.float32)
    assert torch.equal(out, torch.zeros((3, 768), device='cuda'))


# ---------------------------------------------------------------------------------------------------------------------------
def _duet(mods):
    m = mods['duet'].VLNBert(mods['config'].default_duet_args()).cuda().eval()
    m.vln_bert.load_state_dict(mods['synth'].synth_state_dict(manifest('duet'), seed=0, gasa_stress=True))
    return m


def _hamt(mods):
    m = mods['hamt'].VLNBertCMT(mods['config'].default_hamt_args()).cuda().eval()
    m.vln_bert.load_state_dict(mods['synth'].synth_state_dict(manifest('hamt'), seed=0))
    return m


def _rows_like(fs, store, shape, masked=None, seed=0):
    """FeatureRows of ``shape`` (host int32 indices) with -1 where ``masked`` (bool array) is True"""
    g = np.random.default_rng(seed)
    idx = g.integers(0, store.n_rows, shape).astype(np.int32)
    if masked is not None:
        idx[masked] = -1
    return fs.FeatureRows(store, torch.from_numpy(idx).pin_memory())


FORMATS = [('fp32', 'auto'), ('bf16', 'f16'), ('bf16', 'bf16')]


def _set_format(model, fmt):
    model.vln_bert.precision, model.vln_bert.operand16 = fmt


def _duet_calls(mods, model, ep):
    d = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in ep.items()}
    pano = lambda x: model('panorama', {'view_img_fts': x, 'loc_fts': d['loc_fts'], 'nav_types': d['nav_types'],   # noqa: E731
                                        'view_lens': d['view_lens']})[0]
    imag = lambda x: model('imagine', {'imagine_feats': x, 'imagine_masks': None})                                   # noqa: E731
    return pano, imag


def _hamt_calls(mods, model, ep):
    d = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in ep.items()}
    with torch.no_grad():
        txt = model('language', txt_ids=d['txt_ids'], txt_masks=d['txt_masks'])
        img = model('imagine', imagine_pano_img_feats=d['imagine_feats'], imagine_masks=None)
    hist = [d['hist_embeds'][:, t] for t in range(d['hist_embeds'].shape[1])]
    visual = lambda x: model('visual', txt_embeds=txt, txt_masks=d['txt_masks'], hist_embeds=hist,                   # noqa: E731
                             hist_lens=[int(v) for v in ep['hist_lens']], ob_img_feats=x, ob_ang_feats=d['ob_ang_feats'],
                             ob_nav_types=d['ob_nav_types'], ob_masks=d['ob_masks'], imagine_embeds=img,
                             imagine_masks=d['imagine_masks'], return_states=True)
    history = lambda x, xp: model('history', hist_img_feats=x, hist_ang_feats=d['hist_ang_feats'], ob_step=ep['ob_step'],  # noqa: E731
                                  hist_pano_img_feats=xp, hist_pano_ang_feats=d['hist_pano_ang_feats'])
    imag = lambda x: model('imagine', imagine_pano_img_feats=x, imagine_masks=None)                                  # noqa: E731
    return visual, history, imag


def _check(call, rows_list, tag):
    """call(*FeatureRows) against call(*dense tensors), bit for bit, for every output"""
    got = call(*rows_list)
    ref = call(*[r.dense() for r in rows_list])
    got = got if isinstance(got, (tuple, list)) else (got,)
    ref = ref if isinstance(ref, (tuple, list)) else (ref,)
    for i, (a, b) in enumerate(zip(got, ref)):
        if torch.is_tensor(a):
            assert _same(a, b), (tag, i)


@pytest.mark.parametrize('fmt', FORMATS, ids=['fp32', 'f16', 'bf16'])
@pytest.mark.parametrize('graphs', [False, True], ids=['eager', 'graph'])
def test_duet_modes_rows_equal_dense(mods, fmt, graphs):
    fs, synth = mods['feature_store'], mods['synth']
    model = _duet(mods)
    _set_format(model, fmt)
    model.use_cuda_graphs = graphs
    ep = synth.to_torch(synth.duet_episode(synth.TINY, 7))
    B, V, _ = ep['view_img_fts'].shape
    store = _store(fs, 200, 768, torch.float16)
    vmask = ~(np.arange(V)[None] < ep['view_lens'].numpy()[:, None])
    pano, imag = _duet_calls(mods, model, ep)
    with torch.no_grad():
        # three calls with one set of indices (eager, capture, replay), a replay with new indices, then the store grows
        for i, seed in enumerate((1, 1, 1, 2)):
            _check(pano, [_rows_like(fs, store, (B, V), vmask, seed)], ('pano', i))
        store.add({'extra': np.ones((40, 768), np.float32)})
        for i in range(3):
            _check(pano, [_rows_like(fs, store, (B, V), vmask, 3 + i)], ('pano after growth', i))
        I = ep['imagine_feats'].shape[1]
        _check(imag, [_rows_like(fs, store, (B, I), ~ep['imagine_masks'].numpy(), 9)], 'imagine')


@pytest.mark.parametrize('fmt', FORMATS, ids=['fp32', 'f16', 'bf16'])
@pytest.mark.parametrize('graphs', [False, True], ids=['eager', 'graph'])
def test_hamt_modes_rows_equal_dense(mods, fmt, graphs):
    fs, synth = mods['feature_store'], mods['synth']
    model = _hamt(mods)
    _set_format(model, fmt)
    model.use_cuda_graphs = graphs
    ep = synth.to_torch(synth.hamt_episode(synth.TINY, 7))
    B, O, _ = ep['ob_img_feats'].shape
    V = ep['hist_pano_img_feats'].shape[1]
    store = _store(fs, 300, 768, torch.bfloat16, seed=5)
    omask = ~ep['ob_masks'].numpy()
    visual, history, imag = _hamt_calls(mods, model, ep)
    with torch.no_grad():
        for i, seed in enumerate((1, 1, 1, 2)):
            _check(visual, [_rows_like(fs, store, (B, O), omask, seed)], ('visual', i))
            _check(history, [_rows_like(fs, store, (B,), None, seed), _rows_like(fs, store, (B, V), None, seed + 10)], ('history', i))
        store.add({'extra': np.ones((24, 768), np.float32)})
        for i in range(3):
            _check(visual, [_rows_like(fs, store, (B, O), omask, 5 + i)], ('visual after growth', i))
            _check(history, [_rows_like(fs, store, (B,), None, 5 + i), _rows_like(fs, store, (B, V), None, 15 + i)],
                   ('history after growth', i))
        I = ep['imagine_feats'].shape[1]
        _check(imag, [_rows_like(fs, store, (B, I), ~ep['imagine_masks'].numpy(), 9)], 'imagine')


def _train_step(model, ag, call, x, w):
    ag._DropState.site = 1000                                      # the same dropout site sequence for both paths
    model.zero_grad(set_to_none=True)
    out = call(x)
    loss = (out * w).sum()
    loss.backward()
    return loss.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}


def _compare_training(model, ag, call, rows, w):
    """loss and gradients with FeatureRows against the dense rows.  The loss and every gradient the dense path computes
    reproducibly must be identical bit for bit.  This is weaker than bitwise equality of EVERY gradient: the library sums some
    gradients with atomics (embedding-table rows in vi_scatter_add_rows, attention key / value gradients) and offers no ordered
    variant, so two runs of the dense path itself differ there.  Those parameters - the ones whose gradient differs between two
    dense runs - are only held to 4x the spread of the dense path."""
    l_r, g_r = _train_step(model, ag, call, rows, w)
    l_d, g_d = _train_step(model, ag, call, rows.dense(), w)
    _, g_d2 = _train_step(model, ag, call, rows.dense(), w)
    assert _same(l_r, l_d) and g_r.keys() == g_d.keys() and len(g_r) > 10
    unordered = {n for n in g_d if not _same(g_d[n], g_d2[n])}
    assert len(unordered) < len(g_d) // 4, unordered
    for n in g_r:
        if n in unordered:
            spread = float((g_d[n] - g_d2[n]).abs().max())
            assert float((g_r[n] - g_d[n]).abs().max()) <= 4 * spread + 1e-6 * float(g_d[n].abs().max()), n
        else:
            assert _same(g_r[n], g_d[n]), n


def test_training_with_env_dropout_rows_equal_dense(mods):
    fs, synth, ag = mods['feature_store'], mods['synth'], mods['autograd_ops']
    store = _store(fs, 200, 768, torch.float16, seed=3)
    # DUET panorama
    model = _duet(mods).train()
    assert model.drop_env.p > 0
    ep = synth.to_torch(synth.duet_episode(synth.TINY, 7))
    B, V, _ = ep['view_img_fts'].shape
    pano, _ = _duet_calls(mods, model, ep)
    rows = _rows_like(fs, store, (B, V), ~(np.arange(V)[None] < ep['view_lens'].numpy()[:, None]), 4)
    w = torch.randn((B, V, 768), generator=torch.Generator().manual_seed(0)).cuda()
    _compare_training(model, ag, pano, rows, w)
    # HAMT visual (ob_img_feats)
    model = _hamt(mods).train()
    assert model.drop_env.p > 0
    ep = synth.to_torch(synth.hamt_episode(synth.TINY, 7))
    B, O, _ = ep['ob_img_feats'].shape
    visual, _, _ = _hamt_calls(mods, model, ep)
    rows = _rows_like(fs, store, (B, O), ~ep['ob_masks'].numpy(), 6)
    logits = visual(rows.dense())[0]
    w = torch.randn(logits.shape, generator=torch.Generator().manual_seed(1)).cuda()
    fin = torch.isfinite(logits)
    call = lambda x: torch.where(fin, visual(x)[0], torch.zeros((), device='cuda'))            # noqa: E731
    _compare_training(model, ag, call, rows, w)


def test_graphed_panorama_launches_the_same_library_kernels(mods):
    ops, fs, synth = mods['ops'], mods['feature_store'], mods['synth']
    model = _duet(mods)
    model.use_cuda_graphs = True
    ep = synth.to_torch(synth.duet_episode(synth.TINY, 7))
    B, V, _ = ep['view_img_fts'].shape
    store = _store(fs, 200, 768, torch.float16)
    rows = _rows_like(fs, store, (B, V), None, 1)
    pano, _ = _duet_calls(mods, model, ep)
    counts = {}
    with torch.no_grad():
        model.use_cuda_graphs = False                             # builds the weight shadows outside the counted calls
        pano(rows.dense())
        model.use_cuda_graphs = True
        for name, x in (('dense', rows.dense()), ('rows', rows)):
            per_call = []
            for _ in range(3):                                    # eager, capture (a warm-up run + the captured one), replay
                torch.cuda.synchronize()
                n0 = ops.lib.vi_launch_count()
                pano(x)
                torch.cuda.synchronize()
                per_call.append(ops.lib.vi_launch_count() - n0)
            counts[name] = per_call
    assert counts['rows'] == counts['dense'] and counts['dense'][0] > 0 and counts['dense'][2] == 0, counts
