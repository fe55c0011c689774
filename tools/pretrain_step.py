"""Time one DUET pre-training iteration per proxy task (mlm / mrc / sap) on one GPU.

    python tools/pretrain_step.py [--batch 64] [--iters 10] [--warmup 3] [--json out.json]

An iteration is forward(batch, task) + loss.mean().backward() + a fused AdamW step, in train() mode (dropout on), bf16, on a
synthetic batch at R2R-like sizes (synth.duet_pretrain_batch: 36 views, trajectories of up to 7 panoramas, 80-token
instructions).  Also reported:
  * the loss-gradient kernel (vi_ce_rows_bwd at the MLM vocabulary shape, vi_kl_rows_bwd at the MRC shape) timed with CUDA
    events over 50 launches, its byte count rows * ld * (4 + 4 + 2) (the fp32 logits read twice, the bf16 gradient written once)
    and that traffic as a fraction of 7.7 TB/s;
  * the same iteration as eager PyTorch: oracle/pretrain_oracle.py under torch.autocast(bfloat16) on the same GPU, forward +
    backward (no optimizer step);
  * the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch                                                   # noqa: E402
import torch.nn.functional as F                                # noqa: E402

HBM_BPS = 7.7e12
TASKS = ('mlm', 'mrc', 'sap')


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


def kernel_time(ops, mode, rows, n, ld, reps=50):
    g = torch.Generator(device='cuda').manual_seed(0)
    x = torch.randn((rows, ld), generator=g, device='cuda')
    dloss = torch.rand((rows,), generator=g, device='cuda')
    if mode == 'ce':
        y = torch.randint(0, n, (rows,), generator=g, device='cuda')
        fn = lambda: ops.ce_rows_bwd(x, y, n, dloss, torch.bfloat16)      # noqa: E731
    else:
        y = torch.softmax(torch.randn((rows, n), generator=g, device='cuda'), -1).contiguous()
        fn = lambda: ops.kl_rows_bwd(x, y, n, dloss, torch.bfloat16)      # noqa: E731
    ms = timed(fn, reps, 5)
    nbytes = rows * ld * (4 + 4 + 2)
    return {'rows': rows, 'n_cols': n, 'ld': ld, 'us': ms * 1e3, 'bytes': nbytes, 'frac_of_7.7TBps': nbytes / (ms * 1e-3) / HBM_BPS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('pretrain_step.py needs a GPU')
    import importlib
    synth = importlib.import_module('vln_imagine_b200.synth')
    config = importlib.import_module('vln_imagine_b200.config')
    pretrain = importlib.import_module('vln_imagine_b200.pretrain')
    ops = importlib.import_module('vln_imagine_b200.ops')
    res = {'card': card(), 'batch': a.batch}
    batch = synth.duet_pretrain_sap_labels(synth.duet_pretrain_batch(seed=3, batch=a.batch, n_vp=40, max_steps=7, n_views=36,
                                                                     instr_len=80))
    ep = synth.to_torch(batch)
    dev = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in ep.items()}
    man = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'duet_pretrain_manifest.json')))
    sd = synth.synth_state_dict(man, seed=0)
    sd['mlm_head.predictions.decoder.weight'] = sd['bert.embeddings.word_embeddings.weight']
    model = pretrain.GlocalTextPathCMTPreTraining(config.duet_config(config.default_duet_args())).cuda()
    model.load_state_dict(sd)
    model.train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-5, fused=True)
    n_masked = int((ep['txt_labels'] != -1).sum())
    n_mrc = int(ep['vp_view_mrc_masks'].sum())
    res['shapes'] = {'trajectory_panoramas': int(sum(batch['traj_step_lens'])), 'mlm_rows': n_masked, 'mrc_rows': n_mrc}

    def step(task):
        opt.zero_grad(set_to_none=True)
        model(dev, task, compute_loss=True).mean().backward()
        opt.step()

    res['ms_per_iteration'] = {t: timed(lambda: step(t), a.iters, a.warmup) for t in TASKS}
    res['loss_grad_kernel'] = {'vi_ce_rows_bwd (mlm)': kernel_time(ops, 'ce', n_masked, 30522, 30592),
                               'vi_kl_rows_bwd (mrc)': kernel_time(ops, 'kl', n_mrc, 1000, 1024)}

    # eager yardstick: the CPU oracle's code on the GPU under autocast(bfloat16), forward + backward
    from oracle import pretrain_oracle as P
    eager = {}
    try:
        with torch.device('cuda'):
            sdr = {k: (v.cuda().requires_grad_() if v.is_floating_point() else v.cuda()) for k, v in sd.items()}
            sdr['mlm_head.predictions.decoder.weight'] = sdr['bert.embeddings.word_embeddings.weight']

            def ref_step(task):
                for v in sdr.values():
                    v.grad = None
                with torch.autocast('cuda', dtype=torch.bfloat16):
                    if task == 'mlm':
                        lab = dev['txt_labels']
                        loss = F.cross_entropy(P.forward_mlm(sdr, dev).float(), lab[lab != -1], reduction='none')
                    elif task == 'mrc':
                        lg, tg = P.forward_mrc(sdr, dev)
                        loss = F.kl_div(F.log_softmax(lg.float(), -1), tg, reduction='none').sum(1)
                    else:
                        gl, ll, fl = P.forward_sap(sdr, dev)
                        loss = sum(F.cross_entropy(z.float(), lab, reduction='none')
                                   for z, lab in ((gl, dev['global_act_labels']), (ll, dev['local_act_labels']),
                                                  (fl, dev['global_act_labels'])))
                loss.mean().backward()
            for t in TASKS:
                eager[t] = timed(lambda: ref_step(t), max(2, a.iters // 2), 1)
    except Exception as e:                                  # report, do not guess
        eager = {'not measured': repr(e)[:300]}
    res['eager_autocast_ms_per_iteration_fwd_bwd'] = eager
    print(json.dumps(res, indent=1))
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    t0 = time.time()
    main()
    print('wall %.1f s' % (time.time() - t0))
