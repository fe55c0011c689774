"""SURVEY.md 8(f) N4 - the backward pass of the DUET pre-training tasks (mlm, mrc, sap) on the GPU.

* the loss-gradient kernels vi_ce_rows_bwd / vi_kl_rows_bwd against torch autograd of F.cross_entropy / F.kl_div: the wide
  (CTA per row) and narrow (warp per row) layouts, -inf logits, padding columns, fp32 and 16-bit outputs, determinism;
* the parameter gradients of ``loss.mean().backward()`` against torch autograd of the CPU oracle (oracle/pretrain_oracle.py,
  pinned to the real reference's forward), fp32 check mode within 1e-3, bf16 within NOISE_MARGIN x the oracle's own
  autocast(bfloat16) noise on the same step (parity_utils.check_gradients);
* recording and non-recording forwards agree, train-mode dropout is reproducible, and a few AdamW steps lower the loss."""
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from parity_utils import LOSS_TOL, TOL, check_gradients, manifest, max_rel, to_dev

pytestmark = pytest.mark.gpu

TASKS = ('mlm', 'mrc', 'sap')


# ---- kernels ------------------------------------------------------------------------------------------------------------------
def _ulp_dist16(a, b):
    """distance in units in the last place of two bf16 tensors (sign-magnitude bit patterns mapped onto one integer line)"""
    def line(t):
        i = t.contiguous().view(torch.int16).to(torch.int32)
        return torch.where(i < 0, -(i & 0x7FFF), i)
    return (line(a) - line(b)).abs()


def _logits(rows, n, ld, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.randn((rows, ld), generator=g, device='cuda') * 3.0
    x[:, n:] = float('nan')                                    # the padded tail of a GEMM output is never read
    if rows:
        x[:, :n][torch.rand((rows, n), generator=g, device='cuda') < 0.15] = float('-inf')
    return x


def _case(mode, rows, n, ld, seed=0):
    """(logits, label / target operand, dloss, torch autograd's gradient in fp64 [rows, n])"""
    x = _logits(rows, n, ld, seed)
    g = torch.Generator(device='cuda').manual_seed(seed + 1)
    dloss = torch.rand((rows,), generator=g, device='cuda') * 2.0 - 0.5
    if mode == 'ce':
        lab = torch.randint(0, n, (rows,), generator=g, device='cuda')
        if rows:
            r = torch.arange(rows, device='cuda')
            x[r, lab] = torch.randn((rows,), generator=g, device='cuda')    # a finite label logit ...
            x[r, (lab + 1) % n] = float('-inf')                                # ... right next to masked columns
            x[r, (lab - 1) % n] = float('-inf')
        x64 = x[:, :n].double().requires_grad_()
        F.cross_entropy(x64, lab, reduction='none').backward(dloss.double())
        return x, lab, dloss, x64.grad
    t = torch.rand((rows, n), generator=g, device='cuda')
    t[torch.rand((rows, n), generator=g, device='cuda') < 0.3] = 0.0
    t[~torch.isfinite(x[:, :n])] = 0.0
    t = (t / t.sum(1, keepdim=True).clamp_min(1e-6) * 0.9).contiguous()     # soft targets that do not sum to 1
    x64 = x[:, :n].double().requires_grad_()
    F.kl_div(F.log_softmax(x64, -1), t.double(), reduction='none').sum(1).backward(dloss.double())
    return x, t, dloss, x64.grad


WIDTHS = [(30522, 30592), (1000, 1024), (7, 7), (21, 21), (37, 37)]


@pytest.mark.parametrize('rows', [0, 1, 1000])
@pytest.mark.parametrize('n,ld', WIDTHS)
@pytest.mark.parametrize('mode', ['ce', 'kl'])
def test_xent_rows_bwd_vs_torch(lib_built, mode, n, ld, rows):
    ops = importlib.import_module('vln_imagine_b200.ops')
    fn = ops.ce_rows_bwd if mode == 'ce' else ops.kl_rows_bwd
    if rows == 0:
        x = torch.empty((0, ld), device='cuda')
        y = torch.empty((0,), dtype=torch.int64, device='cuda') if mode == 'ce' else torch.empty((0, n), device='cuda')
        for dt in (torch.float32, torch.bfloat16):
            assert fn(x, y, n, torch.empty((0,), device='cuda'), dt).shape == (0, ld)
        return
    x, y, dloss, ref = _case(mode, rows, n, ld)
    d32 = fn(x, y, n, dloss, torch.float32)
    d16 = fn(x, y, n, dloss, torch.bfloat16)
    assert d32.shape == (rows, ld) and d16.shape == (rows, ld) and d16.dtype == torch.bfloat16
    assert torch.equal(d32[:, n:], torch.zeros_like(d32[:, n:])) and torch.equal(d16[:, n:], torch.zeros_like(d16[:, n:]))
    assert max_rel(d32[:, :n].double(), ref) < 1e-5
    assert torch.equal(d16, d32.to(torch.bfloat16))                           # the 16-bit operand is the fp32 gradient rounded
    # and within 1 ulp of torch's gradient rounded to bf16 wherever the fp32 tolerance above cannot move it across bf16 values
    # (p * T - t cancels to near zero in some entries: there the fp32 rounding dominates)
    big = ref.abs() > 1e-5 * ref.abs().max()
    assert int(_ulp_dist16(d16[:, :n][big], ref[big].to(torch.bfloat16)).max()) <= 1
    assert torch.all(d32[:, :n][torch.isinf(x[:, :n])] == 0)                  # masked logits: no gradient
    assert torch.equal(fn(x, y, n, dloss, torch.float32), d32) and torch.equal(fn(x, y, n, dloss, torch.bfloat16), d16)


# ---- the module against torch autograd of the oracle ---------------------------------------------------------------------------
def _batch(tag):
    synth = importlib.import_module('vln_imagine_b200.synth')
    if tag == 'golden':
        b = synth.duet_pretrain_batch()
    else:
        b = synth.duet_pretrain_batch(seed=11, batch=6, n_vp=30, max_steps=6, n_views=36, instr_len=60)
    return synth.to_torch(synth.duet_pretrain_sap_labels(b))


def _state_dict():
    synth = importlib.import_module('vln_imagine_b200.synth')
    sd = synth.synth_state_dict(manifest('duet_pretrain'), seed=0)
    sd['mlm_head.predictions.decoder.weight'] = sd['bert.embeddings.word_embeddings.weight']        # tied (pretrain_cmt.py:112-117)
    sd['bert.global_encoder.sprel_linear.weight'] = torch.full((1, 1), -0.3)                        # a real GASA bias
    return sd


@pytest.fixture(scope='module')
def env(lib_built):
    pretrain = importlib.import_module('vln_imagine_b200.pretrain')
    config = importlib.import_module('vln_imagine_b200.config')
    model = pretrain.GlocalTextPathCMTPreTraining(config.duet_config(config.default_duet_args())).cuda().eval()
    sd = _state_dict()
    model.load_state_dict(sd)
    return model, sd


def _oracle_losses(sd, ep, task):
    from oracle import pretrain_oracle as P
    if task == 'mlm':
        labels = ep['txt_labels']
        return F.cross_entropy(P.forward_mlm(sd, ep), labels[labels != -1], reduction='none')
    if task == 'mrc':
        logits, targets = P.forward_mrc(sd, ep)
        return F.kl_div(F.log_softmax(logits, -1), targets, reduction='none').sum(1)
    gl, ll, fl = P.forward_sap(sd, ep)
    ga, la = ep['global_act_labels'], ep['local_act_labels']
    return (F.cross_entropy(gl, ga, reduction='none') + F.cross_entropy(ll, la, reduction='none')
            + F.cross_entropy(fl, ga, reduction='none'))


class _OracleParams(torch.nn.Module):
    """the oracle's state dict as leaf tensors, listed in the product's parameter order (the tied decoder weight IS the
    word-embedding tensor, so its two uses sum in one .grad as in the product)"""

    def __init__(self, sd, product_names):
        super().__init__()
        self.sd = {k: (v.clone().requires_grad_() if v.is_floating_point() else v) for k, v in sd.items()}
        self.sd['mlm_head.predictions.decoder.weight'] = self.sd['bert.embeddings.word_embeddings.weight']
        self.names = list(product_names)

    def named_parameters(self, *a, **k):
        for n in self.names:
            yield n, self.sd[n]


_FIXTURES = {}


def _fixture(model, sd, task, tag):
    """gradient fixture of one oracle step built in memory (oracle/gen_golden: _grad_fixture + autocast_noise)"""
    key = (task, tag)
    if key not in _FIXTURES:
        from oracle.gen_golden import _grad_fixture, autocast_noise
        ep = _batch(tag)
        ref = _OracleParams(sd, [n for n, _ in model.named_parameters()])
        loss = _oracle_losses(ref.sd, ep, task)
        loss.mean().backward()
        out = {'loss': loss.detach()}
        autocast_noise(ref, lambda: _oracle_losses(ref.sd, ep, task).mean(), out)
        names = _grad_fixture(ref, out)
        out['word_embeddings_grad'] = ref.sd['bert.embeddings.word_embeddings.weight'].grad.detach().clone()
        gold = {k: torch.as_tensor(np.asarray(v.detach().numpy() if torch.is_tensor(v) else v)) for k, v in out.items()}
        _FIXTURES[key] = (gold, names)
    return _FIXTURES[key]


# bf16 on the golden batch's MRC step is left out: its loss has 6 rows, so which elements round where dominates the gradient
# error, and the oracle's own autocast noise on it (the bound) differs 1.7x between two CPUs' bf16 kernels (element error median
# 0.021 vs 0.036).  The larger batch (12 rows) holds the bf16 MRC gradients to the same rule.
CASES = [(p, t, g) for p in ('fp32', 'bf16') for t in TASKS for g in ('golden', 'larger') if (p, t, g) != ('bf16', 'mrc', 'golden')]


@pytest.mark.parametrize('precision,task,tag', CASES)
def test_pretraining_gradients_vs_oracle(env, precision, task, tag):
    model, sd = env
    gold, names = _fixture(model, sd, task, tag)
    model.bert.precision = precision
    model.zero_grad(set_to_none=True)
    loss = model(to_dev(_batch(tag)), task, compute_loss=True)
    assert loss.requires_grad and loss.shape == gold['loss'].shape
    assert max_rel(loss, gold['loss']) < LOSS_TOL[precision], task
    loss.mean().backward()
    check_gradients(model, gold, names, precision, '%s/%s' % (task, tag))
    params = dict(model.named_parameters())
    if task == 'mrc':                       # the reference's MRC never runs the global branch
        for n, p in params.items():
            if n.startswith('bert.global_encoder.'):
                assert p.grad is None or float(p.grad.abs().max()) == 0.0, n
    if task == 'mlm':                       # tied: embedding scatter-add + decoder dW in one gradient
        got = params['bert.embeddings.word_embeddings.weight'].grad.float().cpu()
        want = gold['word_embeddings_grad']
        assert max_rel(got, want) < (1e-3 if precision == 'fp32' else 5e-2)


@pytest.mark.parametrize('task', TASKS)
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_recording_matches_inference(env, precision, task):
    model, _ = env
    model.bert.precision = precision
    ep = to_dev(_batch('larger'))
    with torch.no_grad():
        ref = model(ep, task, compute_loss=True)
    got = model(ep, task, compute_loss=True)
    assert got.requires_grad and not ref.requires_grad
    assert max_rel(got, ref) < TOL[precision]


def test_train_mode_dropout(env):
    ag = importlib.import_module('vln_imagine_b200.autograd_ops')
    model, _ = env
    ep = to_dev(_batch('golden'))

    def run(seed):
        ag._DropState.seeds.clear()
        ag._DropState.site = 0
        torch.manual_seed(seed)
        model.zero_grad(set_to_none=True)
        total = sum(model(ep, task, compute_loss=True).mean() for task in TASKS)
        total.backward()
        return float(total), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}

    try:
        model.bert.precision = 'bf16'
        model.eval()
        base, _ = run(5)
        model.train()
        a, ga = run(5)
        b, gb = run(5)
        c, _ = run(6)
        assert a == b and a != base and a != c
        # same masks -> same loss; gradients agree up to the summation order of the fp32 atomics of the embedding scatter-add
        assert ga.keys() == gb.keys()
        g1, g2 = torch.cat([ga[n].reshape(-1) for n in ga]), torch.cat([gb[n].reshape(-1) for n in ga])
        assert float((g1 - g2).abs().max() / g1.abs().max()) < 1e-5
        assert all(torch.isfinite(g).all() for g in ga.values())
        model.bert.precision = 'fp32'
        with pytest.raises(NotImplementedError):
            model(ep, 'mlm', compute_loss=True)
    finally:
        model.eval()
        model.bert.precision = 'bf16'
        model.zero_grad(set_to_none=True)


def test_adamw_steps_lower_the_loss(lib_built):
    pretrain = importlib.import_module('vln_imagine_b200.pretrain')
    config = importlib.import_module('vln_imagine_b200.config')
    model = pretrain.GlocalTextPathCMTPreTraining(config.duet_config(config.default_duet_args())).cuda().eval()
    model.load_state_dict(_state_dict())
    model.bert.precision = 'bf16'
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, fused=True)
    ep = to_dev(_batch('golden'))
    losses = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        total = sum(model(ep, task, compute_loss=True).mean() for task in TASKS)
        losses.append(float(total))
        if len(losses) <= 5:
            total.backward()
            opt.step()
    assert np.isfinite(losses).all() and losses[-1] < losses[0], losses
