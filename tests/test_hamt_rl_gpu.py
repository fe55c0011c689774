"""HAMT fine-tuning by imitation + A2C on the GPU (vi_rl.cu, hamt.Critic, train.hamt_finetune_iteration).

* vi_policy_sample / vi_policy_bwd against fp64 torch (Categorical), masked tokens never drawn, reproducible draws, action
  frequencies against the softmax over a fixed set of seeds;
* vi_a2c_loss and its adjoint against an fp64 restatement of the agent's loop (r2r/agent_cmt.py:661-744);
* hamt.Critic: the reference's parameter names, forward, gradients and the dropout path;
* states = txt[:, 0] * hist[:, 0] of 'visual' with return_states=True carry gradient into the cross-modal layers;
* the whole iteration against autograd of the CPU oracle (tests/hamt_rl_oracle.il_a2c_iteration) fed with the kernels' actions,
  and its CUDA-graph replay.
Gradient fixtures are built in memory from the oracle, as in tests/test_pretrain_grads_gpu.py."""
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import hamt_rl_oracle as R
from parity_utils import LOSS_TOL, check_gradients, manifest, max_rel, to_dev

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def m(lib_built):
    names = ('ops', 'autograd_ops', 'hamt', 'train', 'synth', 'config')
    return type('M', (), {n: importlib.import_module('vln_imagine_b200.' + n) for n in names})


def _logits(B, O, seed, single=False):
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.randn((B, O), generator=g, device='cuda') * 2.0
    x[torch.rand((B, O), generator=g, device='cuda') < 0.4] = float('-inf')
    x[:, 0] = torch.randn((B,), generator=g, device='cuda')          # every row keeps an admissible token
    if single:
        x[1::2, :] = float('-inf')
        x[1::2, O - 1] = 0.5                                          # rows with one admissible token, the last one
    return x


def _seed(val):
    return torch.full((1,), val, dtype=torch.int32, device='cuda')


# ---- vi_policy_sample / vi_policy_bwd -----------------------------------------------------------------------------------------
@pytest.mark.parametrize('B,O', [(5, 7), (64, 37), (3, 70)])
def test_policy_sample_vs_torch(m, B, O):
    x = _logits(B, O, 1, single=True)
    stop = torch.randint(0, O, (B,), device='cuda')
    ended = torch.zeros((B,), dtype=torch.uint8, device='cuda')
    ended[0] = 1
    a, lp, ent, mask = m.ops.policy_sample(x, stop, _seed(11), 3, ended)
    c = torch.distributions.Categorical(logits=x.double())
    assert torch.isfinite(x.gather(1, a[:, None])).all()
    assert max_rel(lp.double(), c.log_prob(a)) < 1e-5
    assert max_rel(ent.double(), c.entropy()) < 1e-5
    assert torch.equal(mask, torch.tensor([0.0] + [1.0] * (B - 1), device='cuda'))
    want_ended = (a == stop).to(torch.uint8)
    want_ended[0] = 1
    assert torch.equal(ended, want_ended)
    assert bool((a[1::2] == O - 1).all())                             # single admissible token
    ended2 = torch.zeros_like(ended)
    ended2[0] = 1
    again = m.ops.policy_sample(x, stop, _seed(11), 3, ended2)
    for u, v in zip((a, lp, ent, mask), again):
        assert torch.equal(u, v)                                      # same (seed, site): same draw, same bits


def test_policy_never_samples_masked_tokens(m):
    B, O = 256, 40
    x = _logits(B, O, 2, single=True)
    stop = torch.zeros((B,), dtype=torch.int64, device='cuda')
    ok = torch.isfinite(x)
    for s in range(64):
        for site in (1, 2):
            a = m.ops.policy_sample(x, stop, _seed(1000 + s), site, torch.zeros((B,), dtype=torch.uint8, device='cuda'))[0]
            assert bool(ok.gather(1, a[:, None]).all()), (s, site)


def test_policy_action_frequencies_match_softmax(m):
    """4096 fixed (seed, site) draws per row against the softmax: every frequency within 5 binomial standard deviations
    (+ 1/n) - a deterministic test, the seeds are fixed"""
    B, O, n = 8, 12, 4096
    x = _logits(B, O, 3)
    stop = torch.full((B,), -1, dtype=torch.int64, device='cuda')
    counts = torch.zeros((B, O), dtype=torch.float64, device='cuda')
    for s in range(n // 4):
        for site in range(4):
            a = m.ops.policy_sample(x, stop, _seed(s), site, torch.zeros((B,), dtype=torch.uint8, device='cuda'))[0]
            counts[torch.arange(B, device='cuda'), a] += 1
    p = torch.softmax(x.double(), -1)
    sd = (p * (1 - p) / n).sqrt()
    assert bool(((counts / n - p).abs() <= 5 * sd + 1.0 / n).all())


def test_policy_bwd_vs_autograd(m):
    B, O = 33, 29
    x = _logits(B, O, 4, single=True)
    stop = torch.zeros((B,), dtype=torch.int64, device='cuda')
    a = m.ops.policy_sample(x, stop, _seed(5), 1, torch.zeros((B,), dtype=torch.uint8, device='cuda'))[0]
    g1, g2 = torch.randn(B, device='cuda'), torch.randn(B, device='cuda')
    x64 = x.double().requires_grad_()
    lp = F.log_softmax(x64, -1)
    H = -(lp.exp() * lp.masked_fill(~torch.isfinite(lp), 0.0)).sum(-1)
    (-(g1.double() * lp.gather(1, a[:, None]).squeeze(1) + g2.double() * H)).sum().backward()
    d = m.ops.policy_bwd(x, a, -g1, -g2)
    assert torch.isfinite(d).all() and bool((d[~torch.isfinite(x)] == 0).all())
    assert float((d.double() - x64.grad).abs().max()) < 1e-5 * max(1.0, float(x64.grad.abs().max()))


# ---- vi_a2c_loss ----------------------------------------------------------------------------------------------------------------
def _a2c_reference(v, lp, ent, msk, rew, boot, ended, gamma, w, norm):
    B = v.shape[1]
    R = torch.where(ended.bool(), torch.zeros_like(boot), boot) if boot is not None else torch.zeros_like(v[0])
    pol = crit = en = 0.0
    total = 0.0
    for t in range(v.shape[0] - 1, -1, -1):
        R = R * gamma + rew[t]
        adv = (R - v[t]).detach()
        pol = pol + (-lp[t] * adv * msk[t]).sum()
        crit = crit + ((R - v[t]) ** 2 * msk[t]).sum() * 0.5
        en = en + (-w * ent[t] * msk[t]).sum()
        total = total + msk[t].sum()
    n = {'total': total, 'batch': B, 'none': 1.0}[norm]
    return torch.stack([(pol + crit + en) / n, pol / n, crit / n, en / n])


@pytest.mark.parametrize('norm', ['total', 'batch', 'none'])
@pytest.mark.parametrize('gamma', [0.0, 0.9])
@pytest.mark.parametrize('bootstrap', [True, False])
def test_a2c_loss_vs_loop(m, norm, gamma, bootstrap):
    T, B = 6, 37
    g = torch.Generator(device='cuda').manual_seed(7)
    r = lambda *s: torch.randn(s, generator=g, device='cuda')      # noqa: E731
    v, lp, ent, rew = r(T, B), -r(T, B).abs(), r(T, B).abs(), r(T, B)
    end_at = torch.randint(0, T + 2, (B,), generator=g, device='cuda')       # episodes that end mid-rollout, and some never
    msk = (torch.arange(T, device='cuda')[:, None] <= end_at[None, :]).float()
    ended = (end_at < T).to(torch.uint8)
    boot = r(B) if bootstrap else None
    out = m.ops.a2c_loss(v, lp, ent, msk, rew, boot, ended, gamma, 0.01, norm)
    args = [t.double().requires_grad_() for t in (v, lp, ent)]
    ref = _a2c_reference(*args, msk.double(), rew.double(), boot.double() if boot is not None else None, ended, gamma, 0.01, norm)
    assert float((out.double() - ref.detach()).abs().max()) < 1e-5 * float(ref.detach().abs().max())
    gout = torch.tensor([1.0, 0.3, -0.7, 2.0], device='cuda')
    (ref * gout.double()).sum().backward()
    got = m.ops.a2c_loss_bwd(v, lp, ent, msk, rew, boot, ended, gamma, 0.01, norm, gout)
    for d, a in zip(got, args):
        assert float((d.double() - a.grad).abs().max()) < 1e-5 * max(1e-3, float(a.grad.abs().max()))
    again = m.ops.a2c_loss(v, lp, ent, msk, rew, boot, ended, gamma, 0.01, norm)
    assert torch.equal(out, again)
    assert all(torch.equal(a, b) for a, b in zip(got, m.ops.a2c_loss_bwd(v, lp, ent, msk, rew, boot, ended, gamma, 0.01, norm, gout)))


# ---- hamt.Critic ----------------------------------------------------------------------------------------------------------------
def _critic(m, p=0.0, seed=3):
    c = m.hamt.Critic(m.config.default_hamt_args(dropout=p)).cuda()
    c.load_state_dict(_critic_sd(seed))
    return c


def _critic_sd(seed):
    synth = importlib.import_module('vln_imagine_b200.synth')
    return synth.synth_state_dict({'state2value.0.weight': [512, 768], 'state2value.0.bias': [512], 'state2value.3.weight': [1, 512],
                                   'state2value.3.bias': [1]}, seed=seed)


def test_critic_names_and_shapes(m):
    c = _critic(m, 0.5)
    assert {n: tuple(p.shape) for n, p in c.named_parameters()} == {
        'state2value.0.weight': (512, 768), 'state2value.0.bias': (512,), 'state2value.3.weight': (1, 512), 'state2value.3.bias': (1,)}
    assert c.state2value[2].p == 0.5


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_critic_forward_and_gradients(m, precision):
    c = _critic(m)
    c.precision = precision
    x = torch.randn((90, 768), device='cuda')
    sd = {k: v.double().cuda().requires_grad_() for k, v in c.state_dict().items()}
    x64 = x.double().requires_grad_()
    ref = R.critic(sd, x64)
    gv = torch.randn(90, device='cuda')
    if precision == 'bf16':     # the gradients against the function the kernels evaluate: bf16-rounded states and first-layer weight
        r16 = lambda t: t.detach().to(torch.bfloat16).double().requires_grad_()     # noqa: E731
        x64, sd = r16(x), {k: (r16(v) if k == 'state2value.0.weight' else v.detach().clone().requires_grad_()) for k, v in sd.items()}
        (R.critic(sd, x64) * gv.double()).sum().backward()
    else:
        (ref * gv.double()).sum().backward()
    xr = x.clone().requires_grad_()
    v = c(xr)
    assert v.shape == (90,)
    assert max_rel(v, ref.detach()) < (1e-4 if precision == 'fp32' else 2e-2)
    (v * gv).sum().backward()
    if precision == 'fp32':
        close = lambda a, b: max_rel(a, b) < 1e-3                   # noqa: E731
    else:       # dh is rounded to bf16 as the operand of the gradient GEMMs: a norm-wise bound
        close = lambda a, b: float((a.double() - b).norm() / b.norm()) < 1e-2     # noqa: E731
    assert close(xr.grad, x64.grad)
    for n, p in c.named_parameters():
        assert close(p.grad, sd[n].grad), n
    with torch.no_grad():
        assert torch.equal(c(x), v.detach())


def test_critic_dropout_mask_and_backward(m):
    """train-mode dropout: the mask rebuilt from the hash by vi_dropout on the hidden layer, checked through torch autograd"""
    ag = m.autograd_ops
    c = _critic(m, 0.5).train()
    c.precision = 'fp32'
    x = torch.randn((40, 768), device='cuda', requires_grad=True)
    site0 = ag._DropState.site
    v = c(x)
    assert ag._DropState.site == site0 + 1
    w1, b1 = c.state2value[0].weight, c.state2value[0].bias
    w2, b2 = c.state2value[3].weight, c.state2value[3].bias
    h = torch.relu(x.detach() @ w1.detach().t() + b1.detach())
    keep = m.ops.dropout(torch.ones_like(h), 0.5, ag.dropout_seed(x.device), site0 + 1)     # 0 or 1 / (1 - p)
    assert 0.4 < float((keep > 0).float().mean()) < 0.6
    xs, w1s, b1s, w2s, b2s = (t.detach().double().requires_grad_() for t in (x, w1, b1, w2, b2))
    ref = ((torch.relu(xs @ w1s.t() + b1s) * keep.double()) @ w2s.t() + b2s).squeeze(-1)
    assert max_rel(v, ref.detach()) < 1e-4
    gv = torch.randn(40, device='cuda')
    (v * gv).sum().backward()
    (ref * gv.double()).sum().backward()
    for got, want in ((x.grad, xs.grad), (w1.grad, w1s.grad), (b1.grad, b1s.grad), (w2.grad, w2s.grad), (b2.grad, b2s.grad)):
        assert max_rel(got, want) < 1e-3


# ---- states, the iteration against the oracle ------------------------------------------------------------------------------------
_MODELS = {}


def _model(m):
    if 'm' not in _MODELS:
        model = m.hamt.VLNBertCMT(m.config.default_hamt_args(dropout=0.0, feat_dropout=0.0)).cuda().eval()
        c = model.vln_bert.config                                     # train() mode with every dropout probability at 0
        c.hidden_dropout_prob = c.attention_probs_dropout_prob = c.pred_head_dropout_prob = 0.0
        sd = m.synth.synth_state_dict(manifest('hamt'), seed=0)
        model.vln_bert.load_state_dict(sd)
        _MODELS['m'] = (model, sd, _critic(m).eval())
    return _MODELS['m']


class _Both(torch.nn.Module):
    def __init__(self, net, critic):
        super().__init__()
        self.net, self.critic = net, critic


class _OracleParams(torch.nn.Module):
    """oracle state dicts as leaf tensors under the product's parameter names (net.* = NavCMT, critic.* = Critic)"""

    def __init__(self, sd, csd, names):
        super().__init__()
        self.sd = {k: (v.clone().requires_grad_() if v.is_floating_point() else v) for k, v in sd.items()}
        self.csd = {k: v.clone().requires_grad_() for k, v in csd.items()}
        self.names = list(names)

    def named_parameters(self, *a, **k):
        for n in self.names:
            yield n, (self.sd[n[4:]] if n.startswith('net.') else self.csd[n[7:]])


def _cpu(module):
    return {k: v.detach().cpu() for k, v in module.state_dict().items()}


def _episode(m, shape):
    return m.synth.to_torch(m.synth.hamt_episode(*((m.synth.TINY, 7) if shape == 'tiny' else (m.synth.CFG1, 1234))))


def _states_oracle(sd, csd, ep):
    from oracle import hamt_oracle as H
    from oracle import duet_oracle as D
    B = ep['txt_ids'].shape[0]
    txt = H.forward_text(sd, ep['txt_ids'], ep['txt_masks']).detach()         # fix_lang_embedding
    _, img2 = D.forward_align_cosine(sd, txt, D.forward_imagination(sd, ep['imagine_feats']), ep['sub_instr_imag_flag'],
                                     ep['noun_phrase_segs'])
    hm = H.hist_masks_from_lens(ep['hist_lens'], ep['hist_embeds'].shape[1])
    _, txt_o, hist_o, _ = H.forward_visual(sd, txt, ep['txt_masks'], ep['hist_embeds'], hm, ep['ob_img_feats'],
                                           ep['ob_ang_feats'], ep['ob_nav_types'], ep['ob_masks'], img2, ep['imagine_masks'])
    assert B == txt_o.shape[0]
    return R.critic(csd, txt_o[:, 0] * hist_o[:, 0])


def _states_product(model, critic, ep):
    txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
    img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
    _, img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=ep['txt_masks'], align_imagine_embeds=img,
                    imagine_masks=ep['imagine_masks'], sub_instr_imag_flag=ep['sub_instr_imag_flag'],
                    noun_phrase_segs=ep['noun_phrase_segs'])
    hist = list(ep['hist_embeds'].unbind(1))
    _, states = model('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=hist, hist_lens=ep['hist_lens'],
                      ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'],
                      ob_masks=ep['ob_masks'], imagine_embeds=img2, imagine_masks=ep['imagine_masks'], return_states=True)
    return states, critic(states)


_FIX = {}


def _fixture(key, both, sd, csd, run):
    if key not in _FIX:
        from oracle.gen_golden import _grad_fixture, autocast_noise
        ref = _OracleParams(sd, csd, [n for n, p in both.named_parameters() if p.requires_grad])
        loss = run(ref)
        loss.backward()
        out = {'loss': loss.detach()}
        autocast_noise(ref, lambda: run(ref), out)
        names = _grad_fixture(ref, out)
        _FIX[key] = ({k: torch.as_tensor(np.asarray(v.detach().numpy() if torch.is_tensor(v) else v)) for k, v in out.items()}, names)
    return _FIX[key]


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_states_carry_gradient(m, precision):
    model, sd, critic = _model(m)
    both = _Both(model.vln_bert, critic)
    ep = _episode(m, 'cfg1')                                         # 8 episodes: TINY's 3 critic rows are too few for bf16 statistics
    gold, names = _fixture(('states',), both, sd, _cpu(critic), lambda r: _states_oracle(r.sd, r.csd, ep).sum())
    with torch.no_grad():
        want = _states_oracle(sd, _cpu(critic), ep)
    assert any(n.startswith('net.encoder.x_layers.') for n in names)
    model.vln_bert.precision = critic.precision = precision
    # eval(): autograd records the same nodes as in train(); train() would add the alignment head's fixed 0.15 dropout
    # (MLPProjectionHead), which the oracle does not restate
    try:
        both.zero_grad(set_to_none=True)
        states, values = _states_product(model, critic, to_dev(ep))
        assert states.grad_fn is not None
        assert max_rel(values, want) < LOSS_TOL[precision]          # per episode: their sum cancels
        values.sum().backward()
        check_gradients(both, gold, names, precision, 'states ' + precision)
    finally:
        model.vln_bert.precision = critic.precision = 'bf16'
        both.zero_grad(set_to_none=True)


def test_inference_states_unchanged(m):
    """no autograd: the same single vi_mul_bcast as before, eager and graph-replayed, bit for bit"""
    model, _, _ = _model(m)
    ep = to_dev(_episode(m, 'cfg1'))
    with torch.no_grad():
        txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
        img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
        img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=ep['txt_masks'], align_imagine_embeds=img,
                     imagine_masks=ep['imagine_masks'], sub_instr_imag_flag=ep['sub_instr_imag_flag'],
                     noun_phrase_segs=ep['noun_phrase_segs'])[1]
        kw = dict(txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=list(ep['hist_embeds'].unbind(1)), hist_lens=ep['hist_lens'].cpu(),
                  ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'],
                  ob_masks=ep['ob_masks'], imagine_embeds=img2, imagine_masks=ep['imagine_masks'], return_states=True)
        model.use_cuda_graphs = False
        lo, st = model('visual', **kw)
        model.use_cuda_graphs = True
        lg, sg = model('visual', **kw)
        lg2, sg2 = model('visual', **kw)
        _, txt_o, hist_o, _ = model.vln_bert('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=ep['hist_embeds'],
                                             hist_masks=m.hamt.length2mask(ep['hist_lens'], ep['hist_embeds'].shape[1], 'cuda').logical_not(),
                                             ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'],
                                             ob_nav_types=ep['ob_nav_types'], ob_masks=ep['ob_masks'], imagine_embeds=img2,
                                             imagine_masks=ep['imagine_masks'])
    ref, _ = m.ops.mul_bcast(hist_o, hist_o.stride(0), txt_o, txt_o.stride(0), txt_o.shape[0], 1, want16=False)
    assert st.grad_fn is None and torch.equal(st, ref)
    assert torch.equal(sg, sg2)
    assert max_rel(sg, st) < 2e-2


def _rewards(B, T):
    g = torch.Generator().manual_seed(5)
    return torch.randn((T, B), generator=g)


def _iteration(m, model, critic, ep, T, **kw):
    return m.train.hamt_finetune_iteration(model, critic, ep, T, _rewards(ep['txt_ids'].shape[0], T).cuda(), **kw)


# bf16 at TINY is left out: the critic's first-layer gradients there are sums over 9 rows, so one pre-activation that bf16 rounding
# moves across the ReLU shifts a sampled element by a whole term (critic bias: 0.62 against the oracle's own autocast 0.17 x 1.5).
# CFG1 (24 rows) holds the bf16 iteration to the rule.
@pytest.mark.parametrize('shape,precision', [('tiny', 'fp32'), ('cfg1', 'fp32'), ('cfg1', 'bf16')])
def test_iteration_vs_oracle(m, shape, precision):
    model, sd, critic = _model(m)
    both = _Both(model.vln_bert, critic)
    ep = _episode(m, shape)
    T = 3
    model.vln_bert.precision = critic.precision = precision
    ag = m.autograd_ops
    ag.dropout_seed(torch.device('cuda', torch.cuda.current_device())).fill_(1234)   # the same draws whatever ran before
    ag._DropState.site = 0
    try:
        both.zero_grad(set_to_none=True)
        loss, parts, actions = _iteration(m, model, critic, to_dev(ep), T)
        torch.cuda.synchronize()
        acts = actions.cpu()
        rew = _rewards(ep['txt_ids'].shape[0], T)
        gold, names = _fixture(('it', shape, tuple(acts.reshape(-1).tolist())), both, sd, _cpu(critic),
                               lambda r: R.il_a2c_iteration(r.sd, r.csd, ep, T, rew, acts)[0])
        _, ref_parts = R.il_a2c_iteration(sd, _cpu(critic), ep, T, rew, acts)
        lt = LOSS_TOL[precision]
        assert abs(float(loss) - float(gold['loss'])) < lt * abs(float(gold['loss']))
        for k in ('ce', 'aux', 'policy', 'critic', 'entropy'):
            assert abs(float(parts[k]) - float(ref_parts[k])) < lt * max(abs(float(ref_parts[k])), 1e-3), k
        check_gradients(both, gold, names, precision, 'il+a2c %s %s' % (shape, precision))
    finally:
        model.vln_bert.precision = critic.precision = 'bf16'
        both.zero_grad(set_to_none=True)


def test_iteration_fused_and_graph_replay(m):
    """fused accumulation and a GraphedIteration replay equal the eager iteration at the same seed; two replays with the seed
    advanced in between sample different actions"""
    ag = m.autograd_ops
    model, _, critic = _model(m)
    both = _Both(model.vln_bert, critic)
    ep = to_dev(_episode(m, 'cfg1'))
    T = 3
    seed = ag.dropout_seed(torch.device('cuda', torch.cuda.current_device()))      # the key the kernels' tensors use
    seed0 = seed.clone()
    site0 = ag._DropState.site             # the same (seed, site) ids in every run below: the same draws

    def run(**kw):
        ag._DropState.site = site0
        return _iteration(m, model, critic, ep, T, **kw)

    def grads():
        torch.cuda.synchronize()
        return {n: p.grad.detach().clone() for n, p in both.named_parameters() if p.grad is not None}

    def close(g, ref, what):
        assert set(g) == set(ref), what
        for n in ref:
            assert float((g[n] - ref[n]).abs().max()) <= 1e-4 * float(ref[n].abs().max()) + 1e-12, (what, n)

    both.zero_grad(set_to_none=True)
    l0, _, a0 = run()
    l0, a0, ref = float(l0), a0.clone(), grads()
    assert float(ref['critic.state2value.0.weight'].abs().max()) > 0
    assert float(ref['net.encoder.x_layers.0.visual_attention.att.query.weight'].abs().max()) > 0
    both.zero_grad(set_to_none=True)
    l1, _, a1 = run(fused_accumulation=True)
    assert float(l1) == l0 and torch.equal(a1, a0)
    close(grads(), ref, 'fused')
    del l1, _                # the returned tensors keep the iteration's autograd graph alive (see the DUET graph test)

    both.zero_grad(set_to_none=True)
    flat = m.train.FlatGradients(both)
    names = {id(p): n for n, p in both.named_parameters()}
    rewards = _rewards(ep['txt_ids'].shape[0], T).cuda()
    holder = {}

    def grad_fn(d):
        flat.zero()
        ag._DropState.site = site0
        loss, _, acts = m.train.hamt_finetune_iteration(model, critic, d, T, rewards, fused_accumulation=True)
        holder['acts'] = acts
        return loss.detach()

    def update_fn():
        holder['grads'] = flat.buffer.clone()
        holder['acts_out'] = holder['acts'].clone()
        ag.advance_dropout_seeds()                                   # what an optimiser step does, without moving the weights

    it = m.train.GraphedIteration(both, grad_fn, update_fn, ep, warmup=1)
    try:
        seed.copy_(seed0)
        loss = float(it.replay())
        torch.cuda.synchronize()
        assert abs(loss - l0) < 1e-5 * abs(l0)
        assert torch.equal(holder['acts_out'], a0)
        g = {names[id(p)]: holder['grads'][off:off + p.numel()].view_as(p) for p, off in zip(flat.params, flat.offsets)}
        assert all(float(v.abs().max()) == 0.0 for n, v in g.items() if n not in ref)     # frozen history / text: no gradient
        close({n: v for n, v in g.items() if n in ref}, ref, 'graph replay')
        first = holder['acts_out'].clone()
        draws = []
        for _ in range(2):
            it.replay()
            torch.cuda.synchronize()
            draws.append(holder['acts_out'].clone())
        assert not torch.equal(draws[0], first) and not torch.equal(draws[1], draws[0])
    finally:
        it.finish()
        both.zero_grad(set_to_none=True)


def test_iteration_cfg3_finite(m):
    """cfg-3 shape (B = 64, 15 history steps, 6 decisions) in train() mode with the configuration's dropout everywhere"""
    model = m.hamt.VLNBertCMT(m.config.default_hamt_args()).cuda().train()
    model.vln_bert.load_state_dict(m.synth.synth_state_dict(manifest('hamt'), seed=0))
    critic = _critic(m, 0.5).train()
    ep = to_dev(m.synth.to_torch(m.synth.hamt_episode(m.synth.CFG3, 99)))
    loss, parts, actions = m.train.hamt_finetune_iteration(model, critic, ep, 6, torch.randn((6, 64), device='cuda'))
    torch.cuda.synchronize()
    assert torch.isfinite(loss) and all(torch.isfinite(v) for v in parts.values())
    assert actions.shape == (6, 64)
    assert all(p.grad is None or torch.isfinite(p.grad).all() for p in model.parameters())
    assert all(torch.isfinite(p.grad).all() for p in critic.parameters())
