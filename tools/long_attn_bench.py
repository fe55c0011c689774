"""Attention backward at the long-horizon training lengths (BASELINE.json configs[4]: 200-token instructions, 12 imaginations,
100-node graphs; 32 episodes per GPU), in three parts, printed as one JSON line:

  (a) per-launch time of vi_attn_bwd (CUDA events over many launches, dropout 0.1 as in training) at the cfg-5 problems:
      language self-attention 200 x 200, DUET cross-attention 100 x 212 and 37 x 212, HAMT vision-to-language 53 x 212;
      achieved TFLOP/s from algorithmic FLOPs, 5 x 2 * Lq * Lk * 64 per (episode, head): S = QK^T, dP = dO V^T, dV, dQ, dK,
      counting the recomputation of S (and dP) the key-blocked kernels do in both launches as free;
  (b) against the fp32-arithmetic kernel attn_bwd_kernel<float> on fp32 operands, on the cfg-5 problem it fits (p = 0,
      <= 201 keys: the 200 x 200 self-attention), alternating in one process - the nearest surviving form of the path those
      problems took before the key-blocked kernels;
  (c) one DUET fine-tuning iteration at the cfg-5 per-GPU shape (train.duet_finetune_iteration: B = 32, 6 steps, dropout on)
      replayed from CUDA graphs (train.GraphedIteration), in ms and decisions / s.

The card's name, power limit and maximum SM clock are read in the same run.

    python tools/long_attn_bench.py [--iters 200] [--iter-reps 10]
"""
import argparse
import dataclasses
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vln_imagine_b200 import autograd_ops as ag, config, duet, ops, synth, train  # noqa: E402

B, H = 32, 12
PROBLEMS = [('language self-attention', 200, 200, True), ('DUET cross-attention (global)', 100, 212, False),
            ('DUET cross-attention (local)', 37, 212, False), ('HAMT vision-to-language', 53, 212, False)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = 'unavailable (%s)' % e
    return {'name': name, 'power_limit_and_max_sm_clock': q}


def flops(Lq, Lk):
    return 5 * 2 * Lq * Lk * 64 * B * H


def operands(Lq, Lk, self_attn, dtype, seed=0):
    g = torch.Generator(device='cpu').manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g).cuda().to(dtype)          # noqa: E731
    if self_attn:
        qkv = r(B * Lq, 2304)
        q, k, v = qkv[:, :768], qkv[:, 768:1536], qkv[:, 1536:]
    else:
        q, kv = r(B * Lq, 768), r(B * Lk, 1536)
        k, v = kv[:, :768], kv[:, 768:]
    lens = torch.randint(Lk // 2, Lk + 1, (B,), generator=g)
    lens[0] = Lk
    km = (torch.arange(Lk)[None, :] < lens[:, None]).cuda().view(torch.uint8)
    do = r(B * Lq, 768)
    grads = [torch.empty_like(t) for t in (q, k, v)]
    return q, k, v, do, grads, km


def time_calls(fn, iters):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1000.0 / iters                            # us per launch


def per_launch(iters):
    seed_t = ag.dropout_seed(torch.device('cuda', 0))
    out = []
    for name, Lq, Lk, self_attn in PROBLEMS:
        q, k, v, do, (dq, dk, dv), km = operands(Lq, Lk, self_attn, torch.bfloat16)
        drop = (0.1, 1234, seed_t)
        us = time_calls(lambda: ops.attention_bwd(q, k, v, do, dq, dk, dv, B, Lq, Lk, ops.MASK_ADD_NEG10000, km, drop=drop), iters)
        out.append({'problem': name, 'B': B, 'Lq': Lq, 'Lk': Lk, 'dropout': 0.1, 'us': round(us, 2),
                    'tflops': round(flops(Lq, Lk) / us / 1e6, 1)})
    return out


def against_fp32_kernel(iters, rounds=5):
    out = []
    for name, Lq, Lk, self_attn in PROBLEMS:
        if Lk > 201:
            continue
        new = operands(Lq, Lk, self_attn, torch.bfloat16)
        old = operands(Lq, Lk, self_attn, torch.float32)
        runs = {'bf16 key-blocked tensor-core kernels': [], 'fp32-arithmetic attn_bwd_kernel<float> (fp32 operands)': []}
        for _ in range(rounds):                                            # alternate the two in one process
            for label, (q, k, v, do, (dq, dk, dv), km) in zip(runs, (new, old)):
                runs[label].append(time_calls(lambda: ops.attention_bwd(q, k, v, do, dq, dk, dv, B, Lq, Lk, ops.MASK_ADD_NEG10000, km),
                                              iters))
        med = {k: statistics.median(v) for k, v in runs.items()}
        a, b = list(med.values())
        out.append({'problem': name, 'Lq': Lq, 'Lk': Lk, 'dropout': 0.0, 'us_median': {k: round(v, 2) for k, v in med.items()},
                    'speedup': round(b / a, 2)})
    return out


def iteration(reps):
    ep = synth.to_torch(synth.duet_episode(dataclasses.replace(synth.CFG5, batch=B), 555))
    model = duet.VLNBert(config.default_duet_args()).cuda().train()
    net = model.vln_bert
    net.load_state_dict(synth.synth_state_dict({k: list(v.shape) for k, v in net.state_dict().items()}, seed=0))
    net.precision = 'bf16'
    d = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in ep.items()}
    G, P = ep['gmap_img_embeds'].shape[1], ep['vp_img_embeds'].shape[1]
    d['gmap_vpids'], d['vp_cand_vpids'] = net.intern_vpids(ep['gmap_vpids'], ep['vp_cand_vpids'], G, P, torch.device('cuda'))
    flat = train.FlatGradients(net)
    n_steps = 6

    def grad_fn(e):
        flat.zero()
        loss, _, _, _ = train.duet_finetune_iteration(model, e, n_steps=n_steps, fused_accumulation=True)
        return loss.detach()

    it = train.GraphedIteration(net, grad_fn, ag.advance_dropout_seeds, d, warmup=2)
    try:
        for _ in range(2):
            it.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            loss = it.replay()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        assert torch.isfinite(loss).all() and bool(torch.isfinite(flat.buffer).all())
    finally:
        it.finish()
    return {'B': B, 'steps': n_steps, 'dropout': 'configuration (attention 0.1)', 'graph_replay_ms': round(ms, 2),
            'decisions_per_s': round(B * n_steps / ms * 1000.0, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--iter-reps', type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('long_attn_bench needs a CUDA device: there is no CPU path')
    ops.ensure_init(torch.zeros(1, device='cuda'))
    res = {'card': card(), 'flop_count': '5 x 2 * Lq * Lk * 64 per (episode, head)', 'per_launch': per_launch(a.iters),
           'vs_fp32_arithmetic_kernel': against_fp32_kernel(a.iters), 'duet_cfg5_iteration': iteration(a.iter_reps)}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
