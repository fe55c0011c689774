"""HAMT IL + A2C fine-tuning iteration (train.hamt_finetune_iteration) at the cfg-3 shape: B = 64, 15 history steps, 6 decisions
per rollout, both rollouts (teacher-forced and sampled), forward + backward, no optimiser step (the update graph only advances the
device seed, as an optimiser step does).

    python tools/hamt_train_bench.py [--iters 10] [--rounds 5] [--out FILE]

Three arms alternate within every round, each timed over ``iters`` iterations ending in a device synchronise:
  graph     : the iteration replayed by train.GraphedIteration over the model and the critic (FlatGradients, fused accumulation);
  eager     : the same iteration launched eagerly;
  reference : the same rollouts with the policy, the critic and the A2C tail written as the reference agent writes them
              (torch Categorical per step, host copies of the actions, nn.Sequential critic per step, a Python loop with .item()).
Prints one JSON line: median ms per iteration and decisions/s (2 * B * n_steps decisions per iteration) of each arm, library
launches per eager iteration (vi_launch_count), and the card with its power limit and maximum SM clock read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vln_imagine_b200 import autograd_ops as ag, config, hamt, ops, synth, train  # noqa: E402

N_STEPS = 6


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = 'unavailable (%s)' % e
    return {'name': name, 'power_limit_and_max_sm_clock': q}


def reference_iteration(model, ref_critic, ep, rewards, ml_weight=0.2, gamma=0.9, entropy_weight=0.01, aux_weight=0.5):
    """hamt_finetune_iteration with the reference agent's policy / critic / A2C code (r2r/agent_cmt.py:544-577, 661-744)"""
    B = ep['txt_ids'].shape[0]
    tgt = train.hamt_stop_tokens(ep['ob_nav_types'])
    ces = []
    aux, _ = train._hamt_rollout(model, ep, N_STEPS, lambda *a: ces.append(torch.nn.functional.cross_entropy(
        train._hamt_visual(model, ep, *a)[0], tgt, reduction='sum')))
    loss = torch.stack(ces).sum() * (ml_weight / B) + aux_weight * aux
    stop = tgt.cpu().numpy()
    ended = np.zeros(B, bool)
    hidden, logps, ents, masks = [], [], [], []

    def step(*a):
        logit, h = train._hamt_visual(model, ep, *a, return_states=True)
        c = torch.distributions.Categorical(torch.softmax(logit, 1))
        ents.append(c.entropy())
        act = c.sample().detach()
        logps.append(c.log_prob(act))
        hidden.append(h)
        masks.append(np.array(~ended, np.float32))
        ended[:] = ended | (act.cpu().numpy() == stop)
    _, last = train._hamt_rollout(model, ep, N_STEPS, step)
    last_v = ref_critic(train._hamt_visual(model, ep, *last, return_states=True)[1]).squeeze().detach().cpu().numpy()
    R = np.where(ended, 0.0, last_v).astype(np.float32)
    rw = rewards.cpu().numpy()
    rl, total = 0.0, 0.0
    for t in range(N_STEPS - 1, -1, -1):
        R = R * gamma + rw[t]
        m_ = torch.from_numpy(masks[t]).cuda()
        r_ = torch.from_numpy(R.copy()).cuda()
        v_ = ref_critic(hidden[t]).squeeze()
        a_ = (r_ - v_).detach()
        t_pol = (-logps[t] * a_ * m_).sum()
        t_crit = (((r_ - v_) ** 2) * m_).sum() * 0.5
        rl = rl + t_pol + t_crit + (-entropy_weight * ents[t] * m_).sum()
        t_crit.item(), t_pol.item()                               # the agent's per-step loss logs
        total += float(np.sum(masks[t]))
    loss = loss + rl / total
    loss.backward()
    return loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('hamt_train_bench needs a GPU')
    dev = torch.device('cuda')
    model = hamt.VLNBertCMT(config.default_hamt_args()).to(dev).train()
    man = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'hamt_manifest.json')))
    model.vln_bert.load_state_dict(synth.synth_state_dict(man, seed=0))
    critic = hamt.Critic(config.default_hamt_args()).to(dev).train()
    ref_critic = torch.nn.Sequential(torch.nn.Linear(768, 512), torch.nn.ReLU(), torch.nn.Dropout(0.5), torch.nn.Linear(512, 1)).to(dev)
    ref_critic.load_state_dict(critic.state2value.state_dict())
    ep = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in synth.to_torch(synth.hamt_episode(synth.CFG3, 1234)).items()}
    B = ep['txt_ids'].shape[0]
    rewards = torch.randn((N_STEPS, B), generator=torch.Generator().manual_seed(3)).to(dev)
    both = torch.nn.ModuleList([model, critic])

    def eager():
        both.zero_grad(set_to_none=True)
        return train.hamt_finetune_iteration(model, critic, ep, N_STEPS, rewards)[0]

    def reference():
        both.zero_grad(set_to_none=True)
        ref_critic.zero_grad(set_to_none=True)
        return reference_iteration(model, ref_critic, ep, rewards)

    for _ in range(2):
        eager()
        reference()
    torch.cuda.synchronize()
    n0 = ops._Counters.launches
    loss_eager = float(eager().detach())
    launches = ops._Counters.launches - n0
    torch.cuda.synchronize()

    both.zero_grad(set_to_none=True)
    flat = train.FlatGradients(both)

    def grad_fn(d):
        flat.zero()
        return train.hamt_finetune_iteration(model, critic, d, N_STEPS, rewards, fused_accumulation=True)[0].detach()

    it = train.GraphedIteration(both, grad_fn, ag.advance_dropout_seeds, ep, warmup=2)
    arms = {'graph': it.replay, 'eager': eager, 'reference': reference}
    times = {k: [] for k in arms}
    try:
        for k, fn in arms.items():                                   # warm-up of every arm after the capture
            fn()
        for _ in range(a.rounds):
            for k, fn in arms.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(a.iters):
                    fn()
                torch.cuda.synchronize()
                times[k].append((time.perf_counter() - t0) * 1e3 / a.iters)
        loss_graph = float(it.loss)
    finally:
        it.finish()
    res = {'workload': 'hamt_il_a2c_iteration_cfg3', 'batch': B, 'n_hist': synth.CFG3.n_hist, 'n_steps': N_STEPS,
           'decisions_per_iteration': 2 * B * N_STEPS, 'launches_per_iteration': int(launches),
           'loss_eager': loss_eager, 'loss_graph': loss_graph}
    for k, v in times.items():
        med = statistics.median(v)
        res[k] = {'ms_per_iteration': round(med, 3), 'decisions_per_s': round(2 * B * N_STEPS / med * 1e3, 1),
                  'ms_rounds': [round(x, 3) for x in v]}
    res['card'] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
