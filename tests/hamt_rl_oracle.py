"""TEST INFRASTRUCTURE - CPU restatement of HAMT's imitation + A2C fine-tuning losses and of its Critic, the reference against
which tests/test_hamt_rl_gpu.py pins train.hamt_finetune_iteration and hamt.Critic (fixtures built in memory with
oracle/gen_golden._grad_fixture + autocast_noise).

Builds on oracle/hamt_oracle.py and oracle/duet_oracle.py (the model's modes).  Unlike those, this restatement is NOT pinned to
outputs of the real reference: the agent code it restates (VLN-HAMT/finetune_src/r2r/agent_cmt.py:544-577 sampling, :661-744 the
A2C tail; models/model_HAMT.py:289-300 the Critic) was not available to run, so the loss, the critic's parameter names and the
parser defaults (gamma = 0.9, entropy weight 0.01, normalisation 'total') follow SURVEY.md section 3.3 and Recurrent-VLN-BERT,
which HAMT inherits.  Check them against the reference, and pin them with a generated fixture, wherever it is available.
"""
import torch
import torch.nn.functional as F

from oracle.duet_oracle import forward_align_cosine, forward_imagination, lin
from oracle.hamt_oracle import forward_history, forward_text, forward_visual


def critic(sd, state):
    """Critic.forward with dropout off: state2value = Linear(768, 512) -> ReLU -> Dropout -> Linear(512, 1), squeezed.
    models/model_HAMT.py:289-300 (names as in Recurrent-VLN-BERT, which HAMT inherits)."""
    return lin(sd, 'state2value.3', torch.relu(lin(sd, 'state2value.0', state))).squeeze(-1)


def _rollout(sd, ep, n_steps, step):
    """language (frozen) + imagine + cosine alignment, then n_steps of 'visual' with the history growing by one token per step
    (history embeddings frozen, the released configuration).  ``step(t, visual_outputs)``; returns (aux, bootstrap visual outputs)."""
    B = ep['txt_ids'].shape[0]
    txt = forward_text(sd, ep['txt_ids'], ep['txt_masks']).detach()
    img = forward_imagination(sd, ep['imagine_feats'])
    aux, img2 = forward_align_cosine(sd, txt, img, ep['sub_instr_imag_flag'], ep['noun_phrase_segs'])
    hist = [forward_history(sd, None, None, None, None, None, batch_size=B).detach()]

    def visual(n):
        h = torch.stack(hist, 1)
        hm = torch.arange(h.shape[1])[None, :] < torch.full((B,), n)[:, None]
        return forward_visual(sd, txt, ep['txt_masks'], h, hm, ep['ob_img_feats'], ep['ob_ang_feats'], ep['ob_nav_types'],
                              ep['ob_masks'], img2, ep['imagine_masks'])
    for t in range(n_steps):
        step(t, visual(t + 1))
        hist.append(forward_history(sd, ep['hist_img_feats'], ep['hist_ang_feats'], t, ep['hist_pano_img_feats'],
                                    ep['hist_pano_ang_feats']).detach())
    return aux, visual(n_steps + 1)


def il_a2c_iteration(sd, csd, ep, n_steps, rewards, actions, ml_weight=0.2, gamma=0.9, entropy_weight=0.01, normalize='total',
                     aux_weight=0.5):
    """The agent's IL + A2C losses (r2r/agent_cmt.py: teacher rollout weighted by ml_weight, sampled rollout trained by A2C,
    :544-577 and :661-744) for GIVEN sampled actions [n_steps, B]; teacher action and [stop] = the last admissible token.
    Returns (loss, dict(ce, aux, rl, policy, critic, entropy))."""
    B = ep['txt_ids'].shape[0]
    ok = ep['ob_nav_types'] != 0
    stop = torch.where(ok, torch.arange(ok.shape[1])[None, :], torch.zeros_like(ep['ob_nav_types'])).max(1).values
    out, loss = {}, 0.0
    if ml_weight != 0:
        ces = []
        aux, _ = _rollout(sd, ep, n_steps, lambda t, v: ces.append(F.cross_entropy(v[0], stop, reduction='sum')))
        ce = torch.stack(ces).sum()
        loss = ce * (ml_weight / B) + aux_weight * aux
        out.update(ce=ce / B, aux=aux)
    logps, ents, masks, states = [], [], [], []
    ended = torch.zeros(B, dtype=torch.bool)

    def sample(t, v):
        logits, txt_o, hist_o, _ = v
        lp = F.log_softmax(logits, -1)
        a = actions[t]
        logps.append(lp.gather(1, a[:, None]).squeeze(1))
        ents.append(-(lp.exp() * lp.masked_fill(~torch.isfinite(lp), 0.0)).sum(-1))           # Categorical.entropy
        masks.append((~ended).to(logits.dtype))
        ended.logical_or_(a == stop)
        states.append(txt_o[:, 0] * hist_o[:, 0])                                            # model_HAMT.py:86
    _, last = _rollout(sd, ep, n_steps, sample)
    boot = critic(csd, last[1][:, 0] * last[2][:, 0]).detach()
    R = torch.where(ended, torch.zeros_like(boot), boot)
    pol = crit = ent = 0.0
    total = 0.0
    for t in range(n_steps - 1, -1, -1):
        R = R * gamma + rewards[t]
        v = critic(csd, states[t])
        adv = (R - v).detach()
        pol = pol + (-logps[t] * adv * masks[t]).sum()
        crit = crit + ((R - v) ** 2 * masks[t]).sum() * 0.5
        ent = ent + (-entropy_weight * ents[t] * masks[t]).sum()
        total = total + masks[t].sum()
    n = {'total': total, 'batch': B, 'none': 1.0}[normalize]
    rl = (pol + crit + ent) / n
    out.update(rl=rl, policy=pol / n, critic=crit / n, entropy=ent / n)
    return loss + rl, out
