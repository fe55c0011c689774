"""Cost of training the text encoder through the contrastive alignment losses, on one GPU.

    python tools/align_text_grads.py [--rounds 5] [--iters 10] [--reps 200] [--json out.json]

Reported, in one run:
  * the card's name and power limit;
  * the alignment-loss backward (vi_infonce_loss_bwd / vi_margin_loss_bwd) at the alignment sizes of a cfg-4 batch of 64 episodes
    (R imagination rows and n_negs negatives as synth.duet_episode builds them), timed with CUDA events over ``--reps`` launches:
    proj only (the frozen-text call), with dtgt, and with dtgt + dnegs; plus the bytes the dnegs contraction must move at least
    (proj, negs and dnegs once, the g_rc scratch and the cosines) and the proj bytes it reads from L2 (once per 8 negatives);
  * the cfg-4 fine-tuning iteration (64 episodes x 6 navigation steps, forward + backward + clipping + AdamW, dropout on, bf16,
    CUDA-graph replay as in bench.py) in ms for four configurations timed alternately over ``--rounds`` rounds: cosine with the
    text frozen (the released recipe), cosine / InfoNCE / margin with the text trainable.  DUET's constructor rejects the margin
    form, as the reference's does: its model is built with InfoNCE and switched to the margin form afterwards, so the iteration
    runs DUET's path with the margin loss and its backward in place of InfoNCE's.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch                                                   # noqa: E402

# name: (constructor overrides, config attributes set after construction)
CONFIGS = {
    'cosine, text frozen': (dict(), {}),
    'cosine, text trainable': (dict(fix_lang_inside_cosine_model=False), {}),
    'InfoNCE, text trainable': (dict(aux_loss_type='contrastive-InfoNCE', fix_lang_inside_cosine_model=False), {}),
    'margin, text trainable': (dict(aux_loss_type='contrastive-InfoNCE', fix_lang_inside_cosine_model=False),
                               dict(aux_loss_type='constrastive-margin', contrastive_margin_value=0.5)),
}


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                      # pragma: no cover
        q = 'nvidia-smi unavailable (%s)' % e
    return {'device': torch.cuda.get_device_name(0), 'nvidia_smi': q}


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def loss_backward(ep, reps):
    """the alignment-loss backward at the sizes of this episode batch"""
    from vln_imagine_b200 import duet, ops
    from vln_imagine_b200._lib import check, lib
    B, L = ep['txt_ids'].shape
    I = ep['imagine_feats'].shape[1]
    rows = duet._align_rows(B, L, I, ep['sub_instr_imag_flag'], ep['noun_phrase_segs'], torch.device('cuda'))
    R, N = rows.R, rows.n_negs
    g = torch.Generator(device='cuda').manual_seed(0)
    p, t, negs = (torch.randn((n, 768), generator=g, device='cuda') for n in (R, R, N))
    dloss = torch.ones(1, device='cuda')
    dp, dt, dn = torch.empty_like(p), torch.empty_like(t), torch.empty_like(negs)
    work = torch.empty(R * (N + 1), device='cuda')
    out = {'R': R, 'n_negs': N,
           'contraction_min_bytes': 4 * (R * 768 + 2 * N * 768 + R * N + R * (N + 1) + R),
           'contraction_proj_l2_bytes': 4 * R * 768 * ((N + 7) // 8)}
    for form, param in (('infonce', 0.007), ('margin', 0.5)):
        fwd = ops.infonce_loss if form == 'infonce' else ops.margin_loss
        fn = lib.vi_infonce_loss_bwd if form == 'infonce' else lib.vi_margin_loss_bwd
        _, scratch = fwd(p, t, negs, rows.ep, rows.np_ep, param, R, N, p.device)
        stream = torch.cuda.current_stream().cuda_stream

        def call(with_t, with_n):
            check(fn(p.data_ptr(), t.data_ptr(), negs.data_ptr(), rows.ep.data_ptr(), rows.np_ep.data_ptr(), param,
                     scratch.data_ptr(), dloss.data_ptr(), dp.data_ptr(), dt.data_ptr() if with_t else None,
                     dn.data_ptr() if with_n else None, work.data_ptr() if with_n else None, R, N, stream), form)
        out[form] = {name: timed(lambda: call(*flags), reps, 10) * 1e3 for name, flags in
                     (('us_proj_only', (False, False)), ('us_with_dtgt', (True, False)), ('us_with_dtgt_dnegs', (True, True)))}
    return out


def iteration_for(over, post, ep_host, iters):
    """a graph-replayed cfg-4 iteration of one configuration -> (a function timing ``iters`` replays in ms, the first loss)"""
    from vln_imagine_b200 import config, duet, synth, train
    model = duet.VLNBert(config.default_duet_args(**over)).cuda()
    net = model.vln_bert
    for k, v in post.items():
        setattr(net.config, k, v)
    net.load_state_dict(synth.synth_state_dict({k: list(v.shape) for k, v in net.state_dict().items()}, seed=0))
    net.precision = 'bf16'
    model.train()
    flat = train.FlatGradients(net)
    opt = torch.optim.AdamW(net.parameters(), lr=1e-5, fused=True, capturable=True)
    dev = torch.device('cuda')
    d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in ep_host.items()}
    G, P = ep_host['gmap_img_embeds'].shape[1], ep_host['vp_img_embeds'].shape[1]
    d['gmap_vpids'], d['vp_cand_vpids'] = net.intern_vpids(ep_host['gmap_vpids'], ep_host['vp_cand_vpids'], G, P, dev)

    def grad_fn(ep):
        flat.zero()
        return train.duet_finetune_iteration(model, ep, n_steps=6, fused_accumulation=True)[0].detach()

    def update_fn():
        torch.nn.utils.clip_grad_norm_(net.parameters(), 40.)         # agent_base.py:225
        opt.step()
    graphed = train.GraphedIteration(net, grad_fn, update_fn, d, warmup=2)
    loss = float(graphed.replay())
    # the replayed graphs hold raw pointers into the optimiser state, the gradient buffer and the static inputs: the returned
    # function keeps every one of them alive for as long as it can replay
    keep = (graphed, model, flat, opt, d)
    return (lambda: timed(keep[0].replay, iters, 1)), loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--reps', type=int, default=200)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('align_text_grads.py needs a GPU')
    from vln_imagine_b200 import ops, synth
    ops.ensure_init(torch.zeros(1, device='cuda'))
    res = {'card': card()}
    ep_host = synth.to_torch(synth.duet_episode(synth.CFG2, 1234))
    res['loss_backward'] = loss_backward(ep_host, a.reps)
    runs, first_loss, errors = {}, {}, {}
    for name, (over, post) in CONFIGS.items():
        try:
            runs[name], first_loss[name] = iteration_for(over, post, ep_host, a.iters)
        except Exception as e:                                  # report, do not guess
            errors[name] = 'not measured: ' + repr(e)[:300]
    times = {name: [] for name in runs}
    for _ in range(a.rounds):                                   # alternate the configurations
        for name, fn in runs.items():
            times[name].append(fn())
    res['iteration_ms'] = {name: {'median': statistics.median(v), 'min': min(v), 'max': max(v), 'rounds': v,
                                  'first_loss': first_loss[name]} for name, v in times.items()}
    res['iteration_ms'].update(errors)
    res['iteration'] = 'cfg-4: 64 episodes x 6 navigation steps, bf16, dropout on, fused accumulation, CUDA-graph replay, %d replays per round' % a.iters
    print(json.dumps(res, indent=1))
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    t0 = time.time()
    main()
    print('wall %.1f s' % (time.time() - t0))
