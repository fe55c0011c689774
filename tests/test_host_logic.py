"""CPU: host-side logic of the product (no kernel launches): the C ABI surface, parameter trees, configuration,
ragged-input flattening, id interning, row stacking, synthetic generators, algorithmic FLOP counts."""
import ctypes
import importlib
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from parity_utils import manifest

synth = importlib.import_module('vln_imagine_b200.synth')
config = importlib.import_module('vln_imagine_b200.config')


def header_symbols():
    text = open(os.path.join(ROOT, 'include', 'vlnimagine.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(vi_[a-z0-9_]+)\s*\(', text)))


def test_library_builds_loads_and_exports_every_declared_symbol(lib_built):
    lib = ctypes.CDLL(lib_built)
    syms = header_symbols()
    assert len(syms) >= 18
    for name in syms:
        assert hasattr(lib, name), '%s is declared in include/vlnimagine.h but not exported' % name
    lib.vi_version.restype = ctypes.c_int
    assert lib.vi_version() >= 100


def test_ctypes_prototypes_cover_the_header(lib_built):
    _lib = importlib.import_module('vln_imagine_b200._lib')
    declared = set(header_symbols()) - {'vi_last_error'}
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    assert _lib.QUERIES <= declared | {'vi_last_error'}


def test_library_contains_blackwell_tensor_core_and_tma_code(lib_built):
    """SASS evidence: UTCHMMA (tcgen05.mma), LDTM (tcgen05.ld), UTMALDG / UTMASTG (TMA load / store)"""
    try:
        sass = subprocess.run(['cuobjdump', '-sass', lib_built], capture_output=True, text=True, timeout=300).stdout
    except FileNotFoundError:
        pytest.skip('cuobjdump not installed')
    for mnemonic in ('UTCHMMA', 'LDTM', 'UTMALDG', 'UTMASTG'):
        assert mnemonic in sass, mnemonic
    assert 'HGMMA' not in sass


def test_no_cpu_fallback(lib_built):
    ops = importlib.import_module('vln_imagine_b200.ops')
    _lib = importlib.import_module('vln_imagine_b200._lib')
    with pytest.raises(_lib.VlnImagineError):
        ops.ensure_init(torch.zeros(4))
    duet = importlib.import_module('vln_imagine_b200.duet')
    model = duet.VLNBert(config.default_duet_args())
    with pytest.raises(_lib.VlnImagineError):
        model('language', {'txt_ids': torch.zeros(2, 8, dtype=torch.long), 'txt_masks': torch.ones(2, 8, dtype=torch.bool)})


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'vln-imagine_b200')
    for fn in os.listdir(pkg):
        if fn.endswith('.py'):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r'^\s*(from|import)\s+oracle', src, flags=re.M), fn


@pytest.mark.parametrize('kind', ['duet', 'hamt'])
def test_parameter_tree_matches_the_reference_state_dict(kind):
    if kind == 'duet':
        m = importlib.import_module('vln_imagine_b200.duet').VLNBert(config.default_duet_args())
    else:
        m = importlib.import_module('vln_imagine_b200.hamt').VLNBertCMT(config.default_hamt_args())
    man = manifest(kind)
    sd = m.vln_bert.state_dict()
    assert set(sd) == set(man)
    assert all(list(sd[k].shape) == man[k] for k in man)
    assert sum(v.numel() for v in sd.values()) == {'duet': 181538565, 'hamt': 171442433}[kind]
    m.vln_bert.load_state_dict(synth.synth_state_dict(man, seed=0))            # reference-layout dict loads verbatim
    names = [n for n, _ in m.named_parameters()]
    assert any(n.startswith('vln_bert.contrastive_alignment_model') for n in names)     # agent optimiser groups
    assert any(n.startswith('vln_bert.imagine_embeddings') for n in names)


def test_parameter_tree_of_the_hamt_imagination_encoder_variant():
    """bypass_imag_encoder=False (the HAMT parser default): imagine_embeddings.* are the ImagineEmbeddings tensors of the reference"""
    m = importlib.import_module('vln_imagine_b200.hamt').VLNBertCMT(
        config.default_hamt_args(bypass_imag_encoder=False, concat_imagine_with='visual'))
    man = manifest('hamt_encvis')
    sd = m.vln_bert.state_dict()
    assert set(sd) == set(man) and all(list(sd[k].shape) == man[k] for k in man)
    assert 'imagine_embeddings.pano_encoder.layer.1.output.LayerNorm.weight' in sd
    m.vln_bert.load_state_dict(synth.synth_state_dict(man, seed=0))


def test_parameter_tree_of_the_duet_reverie_recipe():
    """dataset 'reverie', obj_feat_size 768 (scripts/run_reverie.sh): og_head.* joins the tree, objects share img_linear"""
    m = importlib.import_module('vln_imagine_b200.duet').VLNBert(config.default_duet_args(dataset='reverie', obj_feat_size=768))
    man = manifest('duet_reverie')
    sd = m.vln_bert.state_dict()
    assert set(sd) == set(man) and all(list(sd[k].shape) == man[k] for k in man)
    assert 'og_head.net.3.weight' in sd and not any(k.startswith('img_embeddings.obj_linear') for k in sd)
    m2 = importlib.import_module('vln_imagine_b200.duet').VLNBert(
        config.default_duet_args(dataset='soon', obj_feat_size=2048, imagine_enc_pano=False))       # scripts/run_soon.sh
    man2 = manifest('duet_soon')
    sd2 = m2.vln_bert.state_dict()
    assert set(sd2) == set(man2) and all(list(sd2[k].shape) == man2[k] for k in man2)
    assert list(sd2['img_embeddings.obj_linear.weight'].shape) == [768, 2048] and not any('imagine' in k for k in sd2)


def test_reverie_align_rows_and_lazy_vpid_rows():
    """host-side index builders: REVERIE alignment rows (all valid instruction tokens, slot 0, other episodes as negatives) and the
    lazily materialised viewpoint-id rows DeviceGraphMaps hands to the agent"""
    import numpy as np
    duet = importlib.import_module('vln_imagine_b200.duet')
    masks = torch.tensor([[1, 1, 1, 0, 0], [1, 1, 1, 1, 1], [1, 0, 1, 0, 0]], dtype=torch.bool)
    r = duet.reverie_align_rows(3, 5, 1, masks)
    assert r.R == 3 and r.n_negs == 3 and r.slot.tolist() == [0, 1, 2] and r.ep.tolist() == r.np_ep.tolist() == [0, 1, 2]
    assert r.tok_off.tolist() == [0, 3, 8, 10] and r.tok_rows.tolist() == [0, 1, 2, 5, 6, 7, 8, 9, 10, 12]
    assert r.np_rows.tolist() == r.tok_rows.tolist() and r.np_off.tolist() == r.tok_off.tolist()
    with pytest.raises(ValueError):
        duet.reverie_align_rows(1, 3, 1, torch.zeros(1, 3, dtype=torch.bool))
    gm = importlib.import_module('vln_imagine_b200.graph_map')
    names = [['a', 'b', 'c'], ['x', 'y']]
    nodes = np.array([[-1, 1, 0, 2], [-1, 0, 1, -1]], np.int32)
    rows = gm.VpidRows(names, nodes, np.array([4, 3], np.int32), torch.zeros(2, 4, dtype=torch.int32), -1)
    assert len(rows) == 2 and rows[0] == [None, 'b', 'a', 'c'] and rows[1] == [None, 'x', 'y']
    assert rows == [[None, 'b', 'a', 'c'], [None, 'x', 'y']] and list(rows)[1][2] == 'y' and rows[0] is rows[0]


def test_pretraining_gmap_aggregation_rows_match_the_oracle():
    """N4 groundwork: the segment-mean index arrays for GlobalMapEncoder._aggregate_gmap_features against the oracle's loop"""
    import numpy as np
    from oracle import pretrain_oracle as P
    pre = importlib.import_module('vln_imagine_b200.pretrain')
    ep = synth.duet_pretrain_batch(seed=9, batch=4, max_steps=5)
    N, V = ep['traj_view_img_fts'].shape[:2]
    emb = np.random.default_rng(0).standard_normal((N, V, 16)).astype(np.float32)
    t = torch.from_numpy(emb)
    steps = list(ep['traj_step_lens'])
    ref = P.aggregate_gmap_features(torch.split(t, steps, 0), torch.split(torch.from_numpy(ep['traj_vp_view_lens']), steps, 0),
                                    ep['traj_vpids'], ep['traj_cand_vpids'], ep['gmap_vpids']).numpy()
    off, rows, G = pre.gmap_aggregation_rows(steps, ep['traj_vp_view_lens'], ep['traj_vpids'], ep['traj_cand_vpids'], ep['gmap_vpids'], V)
    src = np.concatenate([emb.reshape(N * V, 16), np.zeros((1, 16), np.float32)], 0)
    got = np.stack([src[rows[off[r]:off[r + 1]]].mean(0) for r in range(len(off) - 1)]).reshape(len(steps), G, 16)
    assert G == ref.shape[1] and np.abs(got - ref).max() < 1e-6
    assert (got[:, 0] == 0).all()


def test_freeze_flags_follow_the_reference():
    duet = importlib.import_module('vln_imagine_b200.duet')
    m = duet.VLNBert(config.default_duet_args(fix_lang_embedding=True, fix_pano_embedding=True)).vln_bert
    assert not any(p.requires_grad for p in m.lang_encoder.parameters())
    assert not any(p.requires_grad for p in m.img_embeddings.parameters())
    assert all(p.requires_grad for p in m.global_encoder.parameters())


def test_config_mirrors_get_vlnbert_models():
    c = config.duet_config(config.default_duet_args(fusion='avg', graph_sprels=False))
    assert c.glocal_fuse is False and c.graph_sprels is False and c.max_action_steps == 100 and c.layer_norm_eps == 1e-12
    h = config.hamt_config(config.default_hamt_args())
    assert h.max_action_steps == 50 and h.num_h_pano_layers == 2 and h.num_r_layers == 0
    with pytest.raises(NotImplementedError):
        importlib.import_module('vln_imagine_b200.hamt').NavCMT(config.hamt_config(config.default_hamt_args(no_lang_ca=True)))


def test_align_rows_flattening():
    duet = importlib.import_module('vln_imagine_b200.duet')
    flags = [['True', 'False', 'True'], ['True']]
    nps = [[[[2, 3], [5, 5]], [[7, 8]], []], [[[1, 1]]]]
    r = duet.AlignRows(2, 10, 3, flags, nps)
    assert r.R == 2                                       # (0,0) and (1,0); (0,2) has no noun phrase, (0,1) is not flagged
    assert r.slot.tolist() == [0, 3]
    assert r.tok_off.tolist() == [0, 3, 4] and r.tok_rows.tolist() == [2, 3, 5, 11]
    assert r.n_negs == 3 and r.np_ep.tolist() == [0, 0, 1] and r.np_off.tolist() == [0, 2, 3, 4]
    with pytest.raises(ValueError):
        duet.AlignRows(1, 4, 1, [['True']], [[[[2, 9]]]])


def test_id_table_padding_and_consistency():
    duet = importlib.import_module('vln_imagine_b200.duet')
    t = duet._IdTable()
    g = t.encode([[None, 'a', 'b'], [None, 'c']], 4, -1)
    c = t.encode([[None, 'b'], [None, 'c', 'a']], 3, -2)
    assert g[0, 3] == -1 and g[1, 2] == -1 and c[0, 2] == -2
    assert g[0, 2] == c[0, 1] and g[1, 1] == c[1, 1] and g[0, 1] == c[1, 2] and g[0, 0] == c[0, 0]


def test_stack_layout_and_pair_alignment():
    blocks = importlib.import_module('vln_imagine_b200.blocks')
    row0, ends, total = blocks.stack_layout([1920, 2368])
    assert row0 == [0, 2048] and ends == [2048, 4416] and total == 4416
    assert all(e % 256 == 0 for e in ends[:-1])            # a 256-row CTA-pair tile never straddles two groups


def test_synthetic_generators_are_deterministic_and_well_formed():
    a, b = synth.duet_episode(synth.CFG1, 5), synth.duet_episode(synth.CFG1, 5)
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert np.array_equal(a[k], b[k]), k
    assert a['txt_ids'][:, 0].tolist() == [101] * 8 and (a['txt_ids'][~a['txt_masks']] == 0).all()
    assert (a['gmap_pair_dists'] == a['gmap_pair_dists'].transpose(0, 2, 1)).all()
    assert (a['gmap_pair_dists'][:, 0] == 0).all() and a['gmap_lens'].max() == 30
    for i in range(8):
        segs, nps, flags = a['sub_instr_segs'][i], a['noun_phrase_segs'][i], a['sub_instr_imag_flag'][i]
        assert len(segs) == len(nps) == len(flags) and 'True' in flags
        for (s, e), spans in zip(segs, nps):
            assert 1 <= s <= e < a['txt_lens'][i] and all(s <= x <= y <= e for x, y in spans)
    h = synth.hamt_episode(synth.CFG1, 5)
    assert ((h['ob_nav_types'] == 2).sum(1) == 1).all() and h['hist_embeds'].shape == (8, 16, 768)
    sd = synth.synth_state_dict(manifest('duet'), seed=0, gasa_stress=True)
    assert float(sd['global_encoder.sprel_linear.weight']) == -0.5


def test_algorithmic_flops_match_the_survey():
    sys.path.insert(0, ROOT)
    bench = importlib.import_module('bench')
    assert abs(bench.flops_per_decision('duet', synth.CFG2) / 1e9 - 7.281) < 2e-3
    assert abs(bench.flops_per_decision('hamt', synth.CFG3) / 1e9 - 11.811) < 2e-3
    assert abs(bench.flops_per_decision('duet', synth.CFG5) / 1e9 - 14.784) < 2e-3


def test_imagination_feature_loader_semantics(tmp_path):
    db_mod = importlib.import_module('vln_imagine_b200.imagine_db')
    rng = np.random.default_rng(0)
    store = {'10_0': rng.standard_normal((2, 1000)), '11_2': rng.standard_normal((3, 1000)), '12_1': np.zeros((0, 1000))}
    np.savez(tmp_path / 'feats.npz', **store)
    for src in (store, str(tmp_path / 'feats.npz')):
        db = db_mod.ImaginationImageFeaturesDB(src, 768)
        ft = db.get_image_feature('10_0')
        assert ft.shape == (2, 768) and ft.dtype == np.float32 and db.get_image_feature('10_0') is ft      # cached
        flags = {'10_0': ['True', 'False', 'True'], '11_2': ['True', 'True', 'False', 'True'], '12_1': ['False', 'False']}
        feats, mask = db_mod.collate_imaginations(db, ['10_0', '11_2', '12_1'], flags, 768)
        assert feats.shape == (3, 4, 768) and mask.tolist() == [[True, False, True, False], [True, True, False, True],
                                                                 [False] * 4]
        assert np.array_equal(feats[0, 2], store['10_0'][1, :768].astype(np.float32)) and not feats[0, 1].any()
        assert np.array_equal(feats[1, 3], store['11_2'][2, :768].astype(np.float32)) and not feats[2].any()
    with pytest.raises(AssertionError):
        db_mod.collate_imaginations(db_mod.ImaginationImageFeaturesDB(store, 768), ['10_0'], {'10_0': ['True']}, 768)


def test_derived_weights_follow_fused_optimizers():
    """torch.optim.AdamW(fused=True) updates parameters in place WITHOUT bumping their version counters; the derived
    weight copies (blocks.Pack) must still be rebuilt after such a step (global optimizer-step hook)."""
    import importlib
    blocks = importlib.import_module('vln_imagine_b200.blocks')
    p = torch.nn.Parameter(torch.randn(8))
    p.grad = torch.randn(8)
    builds = {'n': 0}

    def build():
        builds['n'] += 1
        return p.detach().clone()
    pk = blocks.Pack([p], build)
    pk.get(); pk.get()
    assert builds['n'] == 1
    try:
        opt = torch.optim.AdamW([p], lr=1e-2, fused=True)
    except (RuntimeError, TypeError):                    # no fused CPU implementation in this torch build
        opt = torch.optim.AdamW([p], lr=1e-2)
    opt.step()
    assert torch.equal(pk.get(), p.detach())
    assert builds['n'] == 2
    pk.get()
    assert builds['n'] == 2


def test_16bit_gelu_formula_is_below_bf16_rounding():
    """act_fwd / act_bwd on 16-bit tensors (vln-imagine_b200/csrc/vi_bwd.cu: gelu_terms) replace erff + expf by Abramowitz & Stegun
    7.1.26 with the exponential shared between erf and the density.  The same arithmetic in fp32 numpy, with the constants READ FROM
    THE SOURCE, against the fp64 definition (D/models/vilmodel.py:32-38): both GELU and its derivative within 1e-6 absolute, three
    orders below the 2^-9 relative rounding of the bf16 result."""
    from math import sqrt, pi
    from scipy.special import erf
    src = open(os.path.join(ROOT, 'vln-imagine_b200', 'csrc', 'vi_bwd.cu')).read()
    body = src[src.index('void gelu_terms('):src.index('float gelu_fast(')]
    consts = [float(c) for c in re.findall(r'(-?\d+\.\d+)f', body)]
    assert len(consts) == 12, consts
    ex_scale, _, p, inv_sqrt2, _, a5, a4, a3, a2, a1, half, _ = consts
    assert abs(ex_scale + 0.5 / np.log(2.0)) < 1e-7 and abs(inv_sqrt2 - 1 / sqrt(2)) < 1e-7 and half == 0.5
    f = np.float32
    x = np.linspace(-12, 12, 400001).astype(f)
    ex = np.exp2((x * x * f(ex_scale)).astype(f)).astype(f)
    t = (f(1) / (np.abs(x) * f(p * inv_sqrt2) + f(1))).astype(f)
    q = t * f(a5) + f(a4)
    for a in (a3, a2, a1):
        q = q * t + f(a)
    h = (f(half) * q * t * ex).astype(f)
    cdf = np.where(x >= 0, f(1) - h, h)
    gelu, grad = x * cdf, x * f(0.39894228040143267794) * ex + cdf
    xd = x.astype(np.float64)
    cdf64 = 0.5 * (1 + erf(xd / sqrt(2)))
    assert np.abs(gelu - xd * cdf64).max() < 1e-6
    assert np.abs(grad - (cdf64 + xd * np.exp(-xd * xd / 2) / sqrt(2 * pi))).max() < 1e-6
