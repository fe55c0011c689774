"""The text encoder trained through the InfoNCE and margin forms of the imagination <-> noun-phrase alignment loss.

* vi_infonce_loss_bwd / vi_margin_loss_bwd with their text outputs (dtgt: the row's own noun-phrase mean, dnegs: the noun-phrase
  means of the other episodes) against torch autograd in fp64, fp32 within 1e-4; two calls bit-identical; dproj the same bits
  whether or not the text outputs are asked for;
* the language encoder + the alignment step through the module API against torch autograd of the CPU oracle (forward_text + its
  align function; oracle/gen_golden: _grad_fixture + autocast_noise, built in memory): DUET InfoNCE with
  fix_lang_inside_cosine_model off, DUET REVERIE InfoNCE, HAMT margin and HAMT InfoNCE with fix_lang_embedding off.  fp32 within
  1e-3, bf16 within 1.5 x the oracle's own autocast(bfloat16) noise (parity_utils.check_gradients);
* the same configurations with the text frozen (the released recipes): no gradient reaches the language encoder, and the
  projection head gets the same gradient as with the text trainable (DUET: bit for bit);
* a DUET fine-tuning iteration with InfoNCE and trainable text: fused accumulation, the split language backward and a CUDA-graph
  replay agree with the plain eager pass.

The negatives are built from the same text tensor as the positives (D/models/vilmodel.py:689-779 via :1249-1262), so they carry
gradients exactly when the positives do."""
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from parity_utils import LOSS_TOL, check_gradients, manifest, max_rel, to_dev

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ag(lib_built):
    ops = importlib.import_module('vln_imagine_b200.ops')
    ops.ensure_init(torch.zeros(1, device='cuda'))
    return importlib.import_module('vln_imagine_b200.autograd_ops')


def _rand(*shape, seed=0):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return torch.randn(*shape, generator=g).cuda()


def relerr(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


# ---- kernels ------------------------------------------------------------------------------------------------------------------
def _operands(R, Nn, seed, close):
    """proj, tgt, negs and the episode ids (sorted, 8 episodes); ``close``: half the targets and a third of the negatives near
    their projection rows, so that both hinge states of the margin form occur"""
    p, t = _rand(R, 768, seed=seed), _rand(R, 768, seed=seed + 1)
    negs = _rand(Nn, 768, seed=seed + 2) if Nn else None
    if close:
        t[::2] = p[::2] + 0.3 * t[::2]
        k = negs[::3].shape[0]
        negs[::3] = p[torch.arange(k, device='cuda') % R] + 0.3 * negs[::3]
    g = torch.Generator().manual_seed(seed + 3)
    row_ep = torch.sort(torch.randint(0, 8, (R,), generator=g)).values.int().cuda()
    neg_ep = torch.sort(torch.randint(0, 8, (Nn,), generator=g)).values.int().cuda() if Nn else None
    return p, t, negs, row_ep, neg_ep


def _reference(form, param, p, t, negs, row_ep, neg_ep):
    """torch autograd in fp64 of F.cosine_similarity + F.cross_entropy (InfoNCE) or of the margin form; -> (loss, dp, dt, dn, active)"""
    pr, tr = p.double().requires_grad_(), t.double().requires_grad_()
    nr = negs.double().requires_grad_() if negs is not None else None
    losses, active = [], 0
    for r in range(p.shape[0]):
        ng = nr[neg_ep != row_ep[r]] if nr is not None else pr.new_zeros((0, 768))
        if form == 'infonce':
            sim = F.cosine_similarity(pr[r:r + 1], torch.cat([tr[r:r + 1], ng], 0)) / param
            losses.append(F.cross_entropy(sim[None], torch.zeros(1, dtype=torch.long, device='cuda')))
        else:
            pos = F.cosine_similarity(pr[r:r + 1], tr[r:r + 1]).squeeze()
            hinge = F.relu(param + F.cosine_similarity(pr[r:r + 1], ng) - pos)
            active += int((hinge > 0).sum())
            losses.append((1 - pos) + hinge.mean())
    loss = torch.stack(losses).mean()
    (loss * 0.7).backward()
    return loss, pr.grad, tr.grad, (nr.grad if nr is not None else None), active


def _product(ag, form, param, p, t, negs, row_ep, neg_ep, text_grads=(True, True)):
    fn = ag.InfoNCELossFn if form == 'infonce' else ag.MarginLossFn
    pl = p.clone().requires_grad_()
    tl = t.clone().requires_grad_(text_grads[0])
    nl = negs.clone().requires_grad_(text_grads[1]) if negs is not None else None
    loss = fn.apply(pl, tl, nl, row_ep, neg_ep, param, p.shape[0], 0 if negs is None else negs.shape[0])
    (loss * 0.7).backward()
    torch.cuda.synchronize()
    return loss, pl.grad, tl.grad, (nl.grad if nl is not None else None)


KERNEL_CASES = ([('infonce', T, R, Nn) for T in (0.007, 0.07, 0.3) for R, Nn in ((41, 57), (1, 57), (41, 0))]
                + [('margin', m, R, 57) for m in (0.1, 0.5) for R in (41, 1)])


@pytest.mark.parametrize('form,param,R,Nn', KERNEL_CASES)
def test_text_adjoints_vs_torch(ag, form, param, R, Nn):
    p, t, negs, row_ep, neg_ep = _operands(R, Nn, seed=60 + R, close=form == 'margin')
    loss, dp, dt, dn = _product(ag, form, param, p, t, negs, row_ep, neg_ep)
    ref_loss, rp, rt, rn, active = _reference(form, param, p, t, negs, row_ep, neg_ep)
    loss = float(loss.detach())
    assert abs(loss - float(ref_loss)) < 1e-4 * max(1.0, abs(float(ref_loss)))
    assert relerr(dp, rp) < 1e-4
    if Nn == 0:                                   # InfoNCE over the positive alone: log 1, no gradient anywhere
        assert float(ref_loss) == 0.0 and float(dt.abs().max()) == 0.0 and float(dp.abs().max()) < 1e-6
    else:
        assert relerr(dt, rt) < 1e-4
        assert relerr(dn, rn) < 1e-4
        if R == 1:                                # the negatives of the row's own episode take no part
            own = neg_ep == row_ep[0]
            assert bool(own.any()) and float(dn[own].abs().max()) == 0.0 and float(dn[~own].abs().max()) > 0.0
    if form == 'margin':
        assert 0 < active < int((neg_ep[None, :] != row_ep[:, None]).sum()), 'both hinge states must occur'
    # a second call: the same bits
    _, dp2, dt2, dn2 = _product(ag, form, param, p, t, negs, row_ep, neg_ep)
    assert torch.equal(dp, dp2) and torch.equal(dt, dt2) and (dn is None or torch.equal(dn, dn2))
    # the text outputs do not touch dproj, and each one is independent of the other
    _, dp0, dt0, dn0 = _product(ag, form, param, p, t, negs, row_ep, neg_ep, text_grads=(False, False))
    assert dt0 is None and dn0 is None and torch.equal(dp0, dp)
    _, dp1, dt1, _ = _product(ag, form, param, p, t, negs, row_ep, neg_ep, text_grads=(True, False))
    assert torch.equal(dp1, dp) and torch.equal(dt1, dt)
    if negs is not None:
        _, dp3, dt3, dn3 = _product(ag, form, param, p, t, negs, row_ep, neg_ep, text_grads=(False, True))
        assert dt3 is None and torch.equal(dp3, dp) and torch.equal(dn3, dn)


# ---- modules against torch autograd of the oracle ------------------------------------------------------------------------------
CONFIGS = {
    # name: (model, constructor overrides with the text trainable, the same with the text frozen, manifest)
    'duet_infonce': ('duet', dict(aux_loss_type='contrastive-InfoNCE', fix_lang_inside_cosine_model=False),
                     dict(aux_loss_type='contrastive-InfoNCE'), 'duet'),
    'duet_reverie_infonce': ('duet', dict(dataset='reverie', obj_feat_size=768, aux_loss_type='contrastive-InfoNCE',
                                          fix_lang_inside_cosine_model=False),
                             dict(dataset='reverie', obj_feat_size=768, aux_loss_type='contrastive-InfoNCE'), 'duet_reverie'),
    'hamt_margin': ('hamt', dict(aux_loss_type='constrastive-margin', contrastive_margin_value=0.5, fix_lang_embedding=False),
                    dict(aux_loss_type='constrastive-margin', contrastive_margin_value=0.5), 'hamt'),
    'hamt_infonce': ('hamt', dict(aux_loss_type='contrastive-InfoNCE', fix_lang_embedding=False),
                     dict(aux_loss_type='contrastive-InfoNCE'), 'hamt'),
}
TEXT_PREFIXES = ('embeddings.', 'lang_encoder.', 'encoder.layer.')


def _is_text(name):
    return any(name.startswith(p) for p in TEXT_PREFIXES)


def _episode(cfg_name, shape):
    synth = importlib.import_module('vln_imagine_b200.synth')
    shp, seed = (synth.TINY, 7) if shape == 'tiny' else (synth.CFG1, 1234)
    if cfg_name == 'duet_reverie_infonce':
        return synth.to_torch(synth.duet_reverie_episode(shp, seed))
    if cfg_name.startswith('duet'):
        return synth.to_torch(synth.duet_episode(shp, seed))
    return synth.to_torch(synth.hamt_episode(shp, seed))


_MODELS = {}


def _model(cfg_name, trainable):
    key = (cfg_name, trainable)
    if key not in _MODELS:
        synth = importlib.import_module('vln_imagine_b200.synth')
        config = importlib.import_module('vln_imagine_b200.config')
        kind, over_train, over_frozen, man = CONFIGS[cfg_name]
        over = over_train if trainable else over_frozen
        if kind == 'duet':
            model = importlib.import_module('vln_imagine_b200.duet').VLNBert(config.default_duet_args(**over)).cuda().eval()
        else:
            model = importlib.import_module('vln_imagine_b200.hamt').VLNBertCMT(config.default_hamt_args(**over)).cuda().eval()
        sd = synth.synth_state_dict(manifest(man), seed=0)
        model.vln_bert.load_state_dict(sd)
        _MODELS[key] = (model, sd)
    return _MODELS[key]


def _product_step(cfg_name, model, ep):
    """language -> imagine -> align_with_contrastive_loss; -> the alignment loss"""
    if cfg_name.startswith('duet'):
        txt = model('language', {'txt_ids': ep['txt_ids'], 'txt_masks': ep['txt_masks']})
        img = model('imagine', {'imagine_feats': ep['imagine_feats'], 'imagine_masks': None})
        batch = {'align_txt_embeds': txt, 'txt_masks': ep['txt_masks'], 'align_imagine_embeds': img,
                 'imagine_masks': ep['imagine_masks'], 'obs_instr_ids': ep['obs_instr_ids']}
        if cfg_name != 'duet_reverie_infonce':
            batch.update({k: ep[k] for k in ('sub_instr_segs', 'sub_instr_imag_flag', 'noun_phrase_segs')})
        return model('align_with_contrastive_loss', batch)[0]
    net = model.vln_bert
    txt = net('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
    img = net('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
    return net('align_with_contrastive_loss', align_txt_embeds=txt, align_imagine_embeds=img,
               sub_instr_imag_flag=ep['sub_instr_imag_flag'], noun_phrase_segs=ep['noun_phrase_segs'])[0]


def _oracle_step(cfg_name, cfg, sd, ep, trainable):
    from oracle import duet_oracle as D, hamt_oracle as H
    O = D if cfg_name.startswith('duet') else H
    txt = O.forward_text(sd, ep['txt_ids'], ep['txt_masks'])
    if not trainable:
        txt = txt.detach()
    img = D.forward_imagination(sd, ep['imagine_feats'])
    flags, segs = ep.get('sub_instr_imag_flag'), ep.get('noun_phrase_segs')
    if cfg_name == 'duet_reverie_infonce':
        return D.forward_align_reverie(sd, txt, ep['txt_masks'].bool(), img, 'contrastive-InfoNCE', cfg.infonce_temperature)[0]
    if cfg.aux_loss_type == 'constrastive-margin':
        return D.forward_align_margin(sd, txt, img, flags, segs, cfg.contrastive_margin_value)[0]
    return D.forward_align_infonce(sd, txt, img, flags, segs, cfg.infonce_temperature)[0]


class _OracleParams(torch.nn.Module):
    """the oracle's state dict as leaf tensors, listed in the product's parameter order"""

    def __init__(self, sd, product_names):
        super().__init__()
        self.sd = {k: (v.clone().requires_grad_() if v.is_floating_point() else v) for k, v in sd.items()}
        self.names = [n for n in product_names if n in self.sd]

    def named_parameters(self, *a, **k):
        for n in self.names:
            yield n, self.sd[n]


_FIXTURES = {}


def _fixture(cfg_name, shape, trainable):
    """gradient fixture of one oracle step built in memory (oracle/gen_golden: _grad_fixture + autocast_noise)"""
    key = (cfg_name, shape, trainable)
    if key not in _FIXTURES:
        from oracle.gen_golden import _grad_fixture, autocast_noise
        model, sd = _model(cfg_name, trainable)
        cfg = model.vln_bert.config
        ep = _episode(cfg_name, shape)
        ref = _OracleParams(sd, [n for n, _ in model.vln_bert.named_parameters()])
        loss = _oracle_step(cfg_name, cfg, ref.sd, ep, trainable)
        loss.backward()
        out = {'loss': loss.detach()}
        autocast_noise(ref, lambda: _oracle_step(cfg_name, cfg, ref.sd, ep, trainable), out)
        names = _grad_fixture(ref, out)
        gold = {k: torch.as_tensor(np.asarray(v.detach().numpy() if torch.is_tensor(v) else v)) for k, v in out.items()}
        _FIXTURES[key] = (gold, names)
    return _FIXTURES[key]


def _run(cfg_name, shape, precision, trainable):
    model, _ = _model(cfg_name, trainable)
    net = model.vln_bert
    net.precision = precision
    net.zero_grad(set_to_none=True)
    loss = _product_step(cfg_name, model, to_dev(_episode(cfg_name, shape)))
    loss.backward()
    torch.cuda.synchronize()
    return model, loss


@pytest.mark.parametrize('shape', ['tiny', 'cfg1'])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('cfg_name', list(CONFIGS))
def test_text_encoder_gradients_vs_oracle(lib_built, cfg_name, precision, shape):
    gold, names = _fixture(cfg_name, shape, True)
    model, loss = _run(cfg_name, shape, precision, True)
    assert abs(float(loss) - float(gold['loss'])) < LOSS_TOL[precision] * abs(float(gold['loss']))
    assert sum(_is_text(n) for n in names) > 100, 'the oracle must train the language encoder in this configuration'
    check_gradients(model.vln_bert, gold, names, precision, '%s %s trainable text' % (cfg_name, shape))


@pytest.mark.parametrize('shape', ['tiny', 'cfg1'])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('cfg_name', list(CONFIGS))
def test_frozen_text_gradients(lib_built, cfg_name, precision, shape):
    """the released recipes: the language encoder gets no gradient; the projection head gets the oracle's gradient, and (DUET,
    where freezing only detaches the text at the alignment step) the very bits of the trainable-text run"""
    gold, names = _fixture(cfg_name, shape, False)
    model, loss = _run(cfg_name, shape, precision, False)
    assert abs(float(loss) - float(gold['loss'])) < LOSS_TOL[precision] * abs(float(gold['loss']))
    params = dict(model.vln_bert.named_parameters())
    assert not any(_is_text(n) for n in names)
    assert all(p.grad is None for n, p in params.items() if _is_text(n))
    check_gradients(model.vln_bert, gold, names, precision, '%s %s frozen text' % (cfg_name, shape))
    head = {n: p.grad.clone() for n, p in params.items() if n.startswith('contrastive_alignment_model.')}
    assert head
    model_t, loss_t = _run(cfg_name, shape, precision, True)
    params_t = dict(model_t.vln_bert.named_parameters())
    for n, g in head.items():
        if cfg_name.startswith('duet'):
            assert torch.equal(g, params_t[n].grad), n
        else:                         # HAMT runs the frozen text encoder as an inference call: the same values up to its kernels
            assert max_rel(g, params_t[n].grad) < (1e-4 if precision == 'fp32' else 2e-2), n


# ---- a fine-tuning iteration ---------------------------------------------------------------------------------------------------
def test_finetune_iteration_variants_agree(lib_built):
    """train.duet_finetune_iteration with InfoNCE and trainable text: fused gradient accumulation, the split language backward
    with finish() and a train.GraphedIteration replay against the plain eager pass (the checks of the cosine form)"""
    train = importlib.import_module('vln_imagine_b200.train')
    synth = importlib.import_module('vln_imagine_b200.synth')
    config = importlib.import_module('vln_imagine_b200.config')
    duet = importlib.import_module('vln_imagine_b200.duet')
    model = duet.VLNBert(config.default_duet_args(aux_loss_type='contrastive-InfoNCE', fix_lang_inside_cosine_model=False)).cuda().eval()
    net = model.vln_bert
    net.load_state_dict(synth.synth_state_dict(manifest('duet'), seed=0, gasa_stress=True))
    net.precision = 'bf16'
    ep = to_dev(synth.to_torch(synth.duet_episode(synth.CFG1, 1234)))

    def grads():
        torch.cuda.synchronize()
        return {n: p.grad.detach().clone() for n, p in net.named_parameters()}

    def close(g, ref, what):
        assert set(g) == set(ref), what
        for n in ref:
            assert float((g[n] - ref[n]).abs().max()) <= 1e-4 * float(ref[n].abs().max()) + 1e-12, (what, n)

    net.zero_grad(set_to_none=True)
    l0 = float(train.duet_finetune_iteration(model, ep, n_steps=2)[0])
    ref = grads()
    assert float(ref['lang_encoder.layer.0.attention.self.query.weight'].abs().max()) > 0
    net.zero_grad(set_to_none=True)
    l1 = float(train.duet_finetune_iteration(model, ep, n_steps=2, fused_accumulation=True)[0])
    assert l1 == l0
    close(grads(), ref, 'fused')
    net.zero_grad(set_to_none=True)
    out = train.duet_finetune_iteration(model, ep, n_steps=2, split_language_backward=True)
    params = dict(net.named_parameters())
    assert all(p.grad is None or float(p.grad.abs().max()) == 0.0 for n, p in params.items() if n.startswith('lang_encoder.'))
    out[4]()
    close(grads(), ref, 'split')
    # the returned loss and finish() keep that iteration's autograd graph alive, and with it AccumulateGrad nodes bound to the
    # default stream: a graph captured on a side stream while they live would accumulate outside the capture
    del out

    net.zero_grad(set_to_none=True)
    flat = train.FlatGradients(net)

    def grad_fn(d):
        flat.zero()
        return train.duet_finetune_iteration(model, d, n_steps=2, fused_accumulation=True)[0].detach()

    holder = {}

    def update_fn():
        holder['grads'] = flat.buffer.clone()             # no optimiser step: every replay sees the same weights

    d = dict(ep)                                           # a replayed graph takes interned viewpoint ids
    G, P = ep['gmap_img_embeds'].shape[1], ep['vp_img_embeds'].shape[1]
    d['gmap_vpids'], d['vp_cand_vpids'] = net.intern_vpids(ep['gmap_vpids'], ep['vp_cand_vpids'], G, P, torch.device('cuda'))
    it = train.GraphedIteration(net, grad_fn, update_fn, d, warmup=1)
    try:
        it.load(d)
        loss = float(it.replay())
        torch.cuda.synchronize()
        assert abs(loss - l0) < 1e-5 * abs(l0)
        names = {id(p): n for n, p in net.named_parameters()}
        g = {names[id(p)]: holder['grads'][off:off + p.numel()].view_as(p) for p, off in zip(flat.params, flat.offsets)}
        close(g, ref, 'graph replay')
    finally:
        it.finish()
        net.zero_grad(set_to_none=True)
