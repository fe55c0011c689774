"""Dense image features against a device-resident feature store (feature_store.FeatureRows) through the module API.

    python tools/feature_store_bench.py [--steps 60] [--rounds 7] [--out FILE]

DUET cfg-2: bench.py's e2e step (panorama + navigation from pinned host inputs, logits copied back, one synchronise per step as
the agent needs them).  HAMT cfg-3: visual + history the same way.  The dense arm uploads the fp32 image features every step
(view_img_fts / ob_img_feats, hist_img_feats, hist_pano_img_feats); the store arm uploads int32 row indices into an fp16 store
holding the same features.  The two arms alternate within each round; the JSON line reports the median ms per step and
decisions/s of each, plus vi_gather_rows against the vi_cast_h16 it replaces at the panorama shape (2368 x 768, CUDA events
around a CUDA graph of 200 back-to-back launches; 3.6 - 7 MB working sets, resident in the 126 MB L2 as in the step), and the
card it ran on."""
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
import bench  # noqa: E402
from vln_imagine_b200 import feature_store as fs, ops  # noqa: E402

EP_LEN = 6


def _store_rows(store, key, feats, valid):
    """put feats [B, N, F] (fp32 numpy) into ``store`` under ``key`` and return their FeatureRows (-1 where not ``valid``)"""
    B, N, F = feats.shape
    store.add({key: feats.reshape(B * N, F)})
    start, _ = store.span(key)
    idx = (start + np.arange(B * N, dtype=np.int32)).reshape(B, N)
    idx[~valid] = -1
    return fs.FeatureRows(store, torch.from_numpy(idx).pin_memory())


def duet_arms(model, ep, store, dev):
    d = bench.device_inputs('duet', model, ep, dev)
    txt, img2, _ = bench.episode_prelude('duet', model, d)
    keys = [k for k in bench.step_tensor_keys('duet') if k in ep and torch.is_tensor(ep[k]) and k not in ('gmap_img_embeds', 'vp_img_embeds')]
    host = {k: ep[k].pin_memory() for k in keys}
    lists = {'gmap_vpids': ep['gmap_vpids'], 'vp_cand_vpids': ep['vp_cand_vpids']}
    V = ep['view_img_fts'].shape[1]
    rows = _store_rows(store, 'duet', ep['view_img_fts'].numpy(), np.arange(V)[None] < ep['view_lens'].numpy()[:, None])
    out_host = torch.empty((ep['gmap_img_embeds'].shape[0], ep['gmap_img_embeds'].shape[1]), dtype=torch.float32).pin_memory()

    def step(feats):
        dd = dict(d)
        dd.update(host)
        dd.update(lists)
        dd['view_img_fts'] = feats
        pano, _ = model('panorama', {k: dd[k] for k in bench.DUET_PANO_KEYS})
        dd['vp_img_embeds'] = torch.cat([torch.zeros_like(pano[:, :1]), pano], 1)
        lg = model('navigation', {**{k: dd[k] for k in bench.DUET_NAV_KEYS}, 'txt_embeds': txt, 'imagine_embeds': img2,
                                  'gmap_vpids': dd['gmap_vpids'], 'vp_cand_vpids': dd['vp_cand_vpids']})['fused_logits']
        out_host.copy_(lg, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    return {'dense': lambda: step(host['view_img_fts']), 'store': lambda: step(rows)}, model.vln_bert.drop_context


def hamt_arms(model, ep, store, dev):
    d = bench.device_inputs('hamt', model, ep, dev)
    txt, img2, _ = bench.episode_prelude('hamt', model, d)
    keys = [k for k in bench.step_tensor_keys('hamt') if k in ep and torch.is_tensor(ep[k])]
    host = {k: ep[k].pin_memory() for k in keys}
    hist_lens = [int(x) for x in ep['hist_lens']]
    B, O, _ = ep['ob_img_feats'].shape
    V = ep['hist_pano_img_feats'].shape[1]
    rows = {'ob_img_feats': _store_rows(store, 'ob', ep['ob_img_feats'].numpy(), ep['ob_masks'].numpy()),
            'hist_img_feats': _store_rows(store, 'hist', ep['hist_img_feats'].numpy()[:, None], np.ones((B, 1), bool)),
            'hist_pano_img_feats': _store_rows(store, 'pano', ep['hist_pano_img_feats'].numpy(), np.ones((B, V), bool))}
    rows['hist_img_feats'] = fs.FeatureRows(store, rows['hist_img_feats'].idx.view(B))
    out_host = torch.empty((B, O), dtype=torch.float32).pin_memory()

    def step(feats):
        dd = dict(d)
        dd.update(host)
        dd.update(feats)
        hh = host['hist_embeds'].to(dev, non_blocking=True)
        dd['hist_list'] = [hh[:, t] for t in range(hh.shape[1])]
        dd['hist_lens'] = hist_lens
        lg = bench.hamt_step(model, dd, txt, img2)['act_logits']
        out_host.copy_(lg, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    return {'dense': lambda: step({}), 'store': lambda: step(rows)}, lambda: None


def time_arms(arms, new_episode, steps, rounds, warmup=12):
    for name, fn in arms.items():
        for i in range(warmup):
            if i % EP_LEN == 0:
                new_episode()
            fn()
    ms = {name: [] for name in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for name in order:
            torch.cuda.synchronize()
            e0.record()
            for i in range(steps):
                if i % EP_LEN == 0:
                    new_episode()
                arms[name]()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / steps)
    return ms


def kernel_times(dev, launches=200, rounds=7):
    """vi_gather_rows (fp16 store -> fp16 operand) against vi_cast_h16 (fp32 -> fp16) at 2368 x 768"""
    n, F = 2368, 768
    g = torch.Generator().manual_seed(0)
    store = torch.randn((10 * n, F), generator=g).to(dev, torch.float16)
    idx = torch.randperm(10 * n, generator=g)[:n].to(torch.int32).to(dev)
    src = torch.randn((n, F), generator=g).to(dev)
    dst = torch.empty((n, F), dtype=torch.float16, device=dev)
    calls = {'vi_gather_rows': lambda: ops.gather_rows(store, idx, torch.float16),
             'vi_cast_h16': lambda: ops.cast_h16(src, dst)}
    # each call's launches are captured into one CUDA graph, so that the timing is the kernels', not the host's enqueue rate
    graphs = {}
    for k, fn in calls.items():
        for _ in range(20):
            fn()
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            for _ in range(launches):
                fn()
        cg.replay()
        graphs[k] = cg
    out = {k: [] for k in calls}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for k, cg in graphs.items():
            torch.cuda.synchronize()
            e0.record()
            cg.replay()
            e1.record()
            torch.cuda.synchronize()
            out[k].append(e0.elapsed_time(e1) / launches * 1e3)
    return {k: {'us_median': statistics.median(v), 'us_rounds': [round(x, 3) for x in v]} for k, v in out.items()}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = 'unavailable (%s)' % e
    return {'name': name, 'power_limit_and_max_sm_clock': q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=60)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('feature_store_bench.py measures on a GPU; none is visible')
    dev = torch.device('cuda')
    res = {'card': card(), 'steps_per_round': a.steps, 'rounds': a.rounds, 'store_dtype': 'float16'}
    with torch.no_grad():
        for wl, arms_fn in (('duet_cfg2', duet_arms), ('hamt_cfg3', hamt_arms)):
            kind, shape, _ = bench.workload(wl)
            model, ep = bench.build(kind, shape, 0, 'bf16')
            store = fs.DeviceFeatureStore(dev, 768, torch.float16)
            arms, new_episode = arms_fn(model, ep, store, dev)
            t0 = time.time()
            ms = time_arms(arms, new_episode, a.steps, a.rounds)
            B = shape.batch
            res[wl] = {arm: {'ms_per_step_median': statistics.median(v), 'decisions_per_s': B / (statistics.median(v) * 1e-3),
                             'ms_rounds': [round(x, 4) for x in v]} for arm, v in ms.items()}
            res[wl]['store_over_dense'] = res[wl]['store']['ms_per_step_median'] / res[wl]['dense']['ms_per_step_median']
            res[wl]['wall_s'] = round(time.time() - t0, 1)
            del model, store, arms
            torch.cuda.empty_cache()
        res['kernels_2368x768'] = kernel_times(dev)
    res['card_after'] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
