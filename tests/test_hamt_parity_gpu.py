"""HAMT-Imagine module-level parity on the GPU: product vs golden vectors of the real reference and vs the
CPU oracle, shared weights, both precisions; called through the reference's VLNBertCMT keyword API."""
import dataclasses
import importlib
import os

import pytest
import torch

from parity_utils import TOL, argmax_report, golden, manifest, max_rel, sub16, to_dev

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def env(lib_built):
    synth = importlib.import_module('vln_imagine_b200.synth')
    hamt = importlib.import_module('vln_imagine_b200.hamt')
    config = importlib.import_module('vln_imagine_b200.config')
    from oracle import hamt_oracle
    model = hamt.VLNBertCMT(config.default_hamt_args()).cuda().eval()
    sd = synth.synth_state_dict(manifest('hamt'), seed=0)
    model.vln_bert.load_state_dict(sd)
    return synth, model, hamt_oracle, sd


def run_product(model, ep):
    inner = model.vln_bert
    with torch.no_grad():
        txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
        img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
        loss, img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=ep['txt_masks'],
                           align_imagine_embeds=img.clone(), imagine_masks=ep['imagine_masks'],
                           sub_instr_segs=ep['sub_instr_segs'], sub_instr_imag_flag=ep['sub_instr_imag_flag'],
                           noun_phrase_segs=ep['noun_phrase_segs'], obs_instr_ids=ep['obs_instr_ids'])
        hist_list = [ep['hist_embeds'][:, t] for t in range(ep['hist_embeds'].shape[1])]
        hist_lens = [int(x) for x in ep['hist_lens']]
        kw = dict(txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=hist_list, hist_lens=hist_lens,
                  ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'],
                  ob_masks=ep['ob_masks'], imagine_embeds=img2, imagine_masks=ep['imagine_masks'])
        (logits,) = model('visual', **kw)
        logits2, states = model('visual', return_states=True, **kw)
        # the inner module also returns the refreshed token streams (used for parity only)
        hm = torch.arange(ep['hist_embeds'].shape[1], device='cuda')[None] < torch.as_tensor(hist_lens, device='cuda')[:, None]
        _, txt_o, hist_o, ob_o = inner('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=ep['hist_embeds'],
                                       hist_masks=hm, ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'],
                                       ob_nav_types=ep['ob_nav_types'], ob_masks=ep['ob_masks'], imagine_embeds=img2,
                                       imagine_masks=ep['imagine_masks'])
        hist = model('history', hist_img_feats=ep['hist_img_feats'], hist_ang_feats=ep['hist_ang_feats'], ob_step=ep['ob_step'],
                     hist_pano_img_feats=ep['hist_pano_img_feats'], hist_pano_ang_feats=ep['hist_pano_ang_feats'])
        cls_hist = model('history')
    assert torch.equal(logits, logits2)
    return dict(txt_embeds=txt, aux_loss=loss, aligned_imagine_embeds=img2, act_logits=logits, txt_out=txt_o,
                hist_out=hist_o, ob_out=ob_o, hist_embed=hist, cls_hist=cls_hist, states=states)


@pytest.mark.parametrize('tag,shape,seed', [('tiny', 'TINY', 7), ('cfg1', 'CFG1', 1234)])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_hamt_vs_reference_golden(env, tag, shape, seed, precision):
    synth, model, _, _ = env
    model.vln_bert.precision = precision
    ep = to_dev(synth.to_torch(synth.hamt_episode(getattr(synth, shape), seed)))
    out = run_product(model, ep)
    gold = golden('hamt_' + tag)
    tol = TOL[precision]
    f = (lambda t: t) if tag == 'tiny' else sub16
    for k in ('txt_embeds', 'aligned_imagine_embeds', 'txt_out', 'hist_out', 'ob_out'):
        assert max_rel(f(out[k]), gold[k]) < tol, k
    for k in ('act_logits', 'hist_embed', 'cls_hist'):
        assert max_rel(out[k], gold[k]) < tol, k
    assert abs(float(out['aux_loss']) - float(gold['aux_loss'])) < tol * abs(float(gold['aux_loss']))
    assert max_rel(out['states'], (out['txt_out'][:, 0] * out['hist_out'][:, 0])) < 1e-6
    if precision == 'fp32':
        assert torch.equal(out['act_logits'].cpu().argmax(-1), gold['act_logits'].argmax(-1))


def test_hamt_bf16_argmax_agreement_over_many_decisions(env):
    """bf16 product vs fp32 oracle on 8 x 48 = 384 decisions: logits within 2e-2, every decisive decision
    agrees, raw agreement >= 99 % (see the DUET twin of this test for the rationale)."""
    synth, model, O, sd = env
    model.vln_bert.precision = 'bf16'
    torch.set_num_threads(os.cpu_count())
    shape = dataclasses.replace(synth.CFG1, batch=48)
    agree = total = bad = 0
    worst = 0.0
    for seed in range(300, 308):
        ep_cpu = synth.to_torch(synth.hamt_episode(shape, seed))
        with torch.no_grad():
            o_txt, o_img, o_loss, o_img2 = O.episode_prelude(sd, ep_cpu)
            o_logits = O.nav_step(sd, ep_cpu, o_txt, o_img2)[0]
        out = run_product(model, to_dev(ep_cpu))
        worst = max(worst, max_rel(out['act_logits'], o_logits))
        a, n, b = argmax_report(out['act_logits'], o_logits, TOL['bf16'])
        agree, total, bad = agree + a, total + n, bad + b
    assert worst < TOL['bf16']
    assert bad == 0, 'a decisive decision flipped'
    assert agree / total >= 0.99, (agree, total)


def test_hamt_api_graph_replay_equals_eager_launches(env):
    synth, model, _, _ = env
    model.vln_bert.precision = 'bf16'
    eps = [to_dev(synth.to_torch(synth.hamt_episode(synth.CFG1, s))) for s in (41, 42)]
    model.use_cuda_graphs = False
    eager = [run_product(model, ep) for ep in eps]
    model.use_cuda_graphs = True
    for rep in range(2):
        for ep, ref in zip(eps, eager):
            out = run_product(model, ep)
            for k in ('act_logits', 'hist_embed', 'states'):
                assert torch.equal(out[k], ref[k]), (rep, k)
    assert all(e['graph'] is not None for e in model._g_vis.entries.values())


@pytest.mark.parametrize('tag,shape,seed', [('tiny', 'TINY', 7), ('cfg1', 'CFG1', 1234)])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_hamt_encoder_visual_variant_vs_reference_golden(lib_built, tag, shape, seed, precision):
    """HAMT-Imagine with the parser defaults of the imagination flags (r2r/parser.py:109,122): the ImagineEmbeddings encoder
    (bypass_imag_encoder=False) and the imagination tokens on the vision stream (concat_imagine_with='visual'), against the
    real reference's outputs (oracle/gen_golden.py --model hamt_encvis)."""
    synth = importlib.import_module('vln_imagine_b200.synth')
    hamt = importlib.import_module('vln_imagine_b200.hamt')
    config = importlib.import_module('vln_imagine_b200.config')
    model = hamt.VLNBertCMT(config.default_hamt_args(bypass_imag_encoder=False, concat_imagine_with='visual')).cuda().eval()
    model.vln_bert.load_state_dict(synth.synth_state_dict(manifest('hamt_encvis'), seed=0))
    model.vln_bert.precision = precision
    ep = to_dev(synth.to_torch(synth.hamt_episode(getattr(synth, shape), seed)))
    inner = model.vln_bert
    with torch.no_grad():
        txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
        img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=ep['imagine_masks'])
        loss, img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=ep['txt_masks'],
                           align_imagine_embeds=img.clone(), imagine_masks=ep['imagine_masks'],
                           sub_instr_segs=ep['sub_instr_segs'], sub_instr_imag_flag=ep['sub_instr_imag_flag'],
                           noun_phrase_segs=ep['noun_phrase_segs'], obs_instr_ids=ep['obs_instr_ids'])
        hist_lens = [int(x) for x in ep['hist_lens']]
        hist_list = [ep['hist_embeds'][:, t] for t in range(ep['hist_embeds'].shape[1])]
        kw = dict(txt_embeds=txt, txt_masks=ep['txt_masks'], ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'],
                  ob_nav_types=ep['ob_nav_types'], ob_masks=ep['ob_masks'], imagine_embeds=img2, imagine_masks=ep['imagine_masks'])
        (logits_a,) = model('visual', hist_embeds=hist_list, hist_lens=hist_lens, **kw)        # eager, then the graphed replay
        (logits_b,) = model('visual', hist_embeds=hist_list, hist_lens=hist_lens, **kw)
        (logits_c,) = model('visual', hist_embeds=hist_list, hist_lens=hist_lens, **kw)
        hm = torch.arange(ep['hist_embeds'].shape[1], device='cuda')[None] < torch.as_tensor(hist_lens, device='cuda')[:, None]
        logits, txt_o, hist_o, ob_o = inner('visual', hist_embeds=ep['hist_embeds'], hist_masks=hm, **kw)
    assert torch.equal(logits_a, logits_b) and torch.equal(logits_b, logits_c) and torch.equal(logits_a, logits)
    gold = golden('hamt_encvis_' + tag)
    tol = TOL[precision]
    f = (lambda t: t) if tag == 'tiny' else sub16
    out = dict(imagine_embeds=img, aligned_imagine_embeds=img2, txt_out=txt_o, hist_out=hist_o, ob_out=ob_o)
    for k, v in out.items():
        assert max_rel(f(v), gold[k]) < tol, k
    assert max_rel(logits, gold['act_logits']) < tol
    assert abs(float(loss) - float(gold['aux_loss'])) < tol * abs(float(gold['aux_loss']))
    if precision == 'fp32':
        assert torch.equal(logits.cpu().argmax(-1), gold['act_logits'].argmax(-1))


@pytest.mark.parametrize('tag,shape,seed', [('tiny', 'TINY', 7), ('cfg1', 'CFG1', 1234)])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_hamt_margin_alignment_loss_vs_reference_golden(lib_built, tag, shape, seed, precision):
    """aux_loss_type 'constrastive-margin' (sic; H/r2r/parser.py:117, H/models/vilmodel_cmt.py:825-856) against the real reference"""
    synth = importlib.import_module('vln_imagine_b200.synth')
    hamt = importlib.import_module('vln_imagine_b200.hamt')
    config = importlib.import_module('vln_imagine_b200.config')
    model = hamt.VLNBertCMT(config.default_hamt_args(aux_loss_type='constrastive-margin', contrastive_margin_value=0.5)).cuda().eval()
    model.vln_bert.load_state_dict(synth.synth_state_dict(manifest('hamt'), seed=0))
    model.vln_bert.precision = precision
    ep = to_dev(synth.to_torch(synth.hamt_episode(getattr(synth, shape), seed)))
    with torch.no_grad():
        txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
        img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
        loss, img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=ep['txt_masks'],
                           align_imagine_embeds=img.clone(), imagine_masks=ep['imagine_masks'],
                           sub_instr_segs=ep['sub_instr_segs'], sub_instr_imag_flag=ep['sub_instr_imag_flag'],
                           noun_phrase_segs=ep['noun_phrase_segs'], obs_instr_ids=ep['obs_instr_ids'])
    gold = golden('hamt_margin_' + tag)
    tol = TOL[precision]
    assert abs(float(loss) - float(gold['margin_loss'])) < tol * abs(float(gold['margin_loss']))
    assert max_rel(sub16(img2), gold['margin_imagine_embeds']) < tol


@pytest.mark.parametrize('concat', ['language', 'visual'])
@pytest.mark.parametrize('tok', ['ob', 'ob_hist', 'ob_txt_hist', 'ob_imagine_text'])
def test_hamt_action_token_variants_vs_reference_golden(lib_built, concat, tok):
    """every act_pred_token of H/r2r/parser.py:67 (models/vilmodel_cmt.py:1189-1199) with the imagination tokens on either
    stream, logits against the real reference (oracle/gen_golden.py --model hamt_actpred), both precisions, both sizes"""
    synth = importlib.import_module('vln_imagine_b200.synth')
    hamt = importlib.import_module('vln_imagine_b200.hamt')
    config = importlib.import_module('vln_imagine_b200.config')
    model = hamt.VLNBertCMT(config.default_hamt_args(act_pred_token=tok, concat_imagine_with=concat)).cuda().eval()
    model.vln_bert.load_state_dict(synth.synth_state_dict(manifest('hamt'), seed=0))
    gold = golden('hamt_actpred')
    for tag, shape, seed in (('tiny', synth.TINY, 7), ('cfg1', synth.CFG1, 1234)):
        ep = to_dev(synth.to_torch(synth.hamt_episode(shape, seed)))
        hist_lens = [int(x) for x in ep['hist_lens']]
        hist_list = [ep['hist_embeds'][:, t] for t in range(ep['hist_embeds'].shape[1])]
        for precision in ('fp32', 'bf16'):
            model.vln_bert.precision = precision
            with torch.no_grad():
                txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
                img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
                outs = [model('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=hist_list, hist_lens=hist_lens,
                              ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'],
                              ob_masks=ep['ob_masks'], imagine_embeds=img, imagine_masks=ep['imagine_masks'])[0] for _ in range(3)]
            assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])          # eager call == graph replays
            ref = gold['%s_%s_%s' % (tag, concat, tok)]
            assert max_rel(outs[0], ref) < TOL[precision], (tag, precision)
            if precision == 'fp32':
                assert torch.equal(outs[0].cpu().argmax(-1), ref.argmax(-1))
            # the same call with autograd recording (eval(): no dropout) matches the reference too, and every parameter of the
            # cross-modal layers, the observation embedding and the action head gets a finite gradient
            model.zero_grad(set_to_none=True)
            logits = model('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=hist_list, hist_lens=hist_lens,
                           ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'],
                           ob_masks=ep['ob_masks'], imagine_embeds=img, imagine_masks=ep['imagine_masks'])[0]
            assert logits.requires_grad
            assert max_rel(logits, ref) < TOL[precision], (tag, precision, 'recording')
            logits.sum().backward()
            trained = [(n, p) for n, p in model.vln_bert.named_parameters()
                       if p.requires_grad and n.startswith(('encoder.x_layers.', 'img_embeddings.', 'next_action.'))]
            assert trained
            bad = [n for n, p in trained if p.grad is None or not bool(torch.isfinite(p.grad).all())]
            assert not bad, (tag, precision, bad)
