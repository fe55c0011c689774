#!/usr/bin/env python
"""bench.py - nav-step decisions/sec of the VLN-Imagine hot path on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload duet_cfg2|hamt_cfg3|duet_cfg5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # the reference algorithm on the host CPU cores

--dump-outputs DIR writes what the timed path computed in its last timed step (rank 0) as DIR/<name>.npy in float32, so
that two builds can be compared output for output: the inputs, weights and dropout seeds depend on the arguments only.
The files hold finite numbers only; where an output has -inf (masked logits), see dump_outputs / load_dump.

One "step" = one navigation decision for every episode of the batch = the two per-step model calls the
reference agent makes (DUET: 'panorama' + 'navigation', VLN-DUET/map_nav_src/r2r/agent.py:467,500; HAMT:
'visual' + 'history', VLN-HAMT/finetune_src/r2r/agent_cmt.py:538,604) on synthetic R2R-shaped inputs with
random-init weights.  Episodes are independent, so N GPUs run N independent per-rank batches (weak
scaling, no data-path collective); the time is the max over ranks of a CUDA-event interval.

The JSON line carries: `value` (inputs resident in HBM, CUDA-graph replay of the step), `e2e` (the public
module API with pinned HOST inputs copied in and the logits copied out every step), `roofline` (the tcgen05
GEMM kernel: algorithmic FLOPs / CUDA-event time per launch vs MEASURED_PEAKS.json), `cpu_baseline` (the CPU
oracle timed on this box's host cores), `clocks`, `gpu_launches`.
"""
import argparse
import contextlib
import dataclasses
import json
import os
import statistics
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'nav-step decisions/sec'
UNIT = 'decisions/s'


# ----------------------------------------------------------------------------------------------
# workloads and algorithmic FLOPs (SURVEY.md section 8(d); GEMM + attention, forward)
# ----------------------------------------------------------------------------------------------
def _lin(m, k, n):
    return 2.0 * m * k * n


def _bert(n):
    return 4 * _lin(n, 768, 768) + 4.0 * n * n * 768 + 2 * _lin(n, 768, 3072)


def _x(n, c):
    return 2 * _lin(n, 768, 768) + 2 * _lin(c, 768, 768) + 4.0 * n * c * 768


def _cls(n, k=768):
    return _lin(n, k, 768) + _lin(n, 768, 1)


def flops_per_decision(model, s):
    C = s.instr_len + s.n_imagine
    if model == 'duet':
        G, P, V = s.n_nodes, s.n_views + 1, s.n_views
        pano = _lin(V, 768, 768) + _lin(V, 7, 768) + 2 * _bert(V)
        nav = (_lin(G, 7, 768) + _lin(P, 14, 768) + 4 * (_x(G, C) + _bert(G)) + 4 * (_x(P, C) + _bert(P))
               + _cls(G) + _cls(P) + _cls(1, 1536))
        return pano + nav
    V, O = s.n_views, s.n_views + 1
    nv = s.n_hist + 1 + O
    hist = _lin(1, 768, 768) + _lin(1, 4, 768) + _lin(V, 768, 768) + _lin(V, 4, 768) + 2 * _bert(V)
    visual = _lin(O, 768, 768) + _lin(O, 4, 768) + 4 * (_x(C, nv) + _x(nv, C) + _bert(C) + _bert(nv)) + _cls(O)
    return hist + visual


def workload(name):
    import vln_imagine_b200.synth as synth
    if name == 'duet_cfg2':
        return 'duet', synth.CFG2, ('DUET-Imagine panorama+navigation forward, 64 episodes/GPU, 80-token instruction, '
                                    '5 imaginations, 30-node graph (GASA bias), 36 views')
    if name == 'duet_cfg5':
        return 'duet', dataclasses.replace(synth.CFG5, batch=32), ('DUET-Imagine long horizon, 32 episodes/GPU, '
                                                                   '200-token instruction, 12 imaginations, 100 nodes')
    if name == 'hamt_cfg3':
        return 'hamt', synth.CFG3, ('HAMT-Imagine visual+history forward, 64 episodes/GPU, 80-token instruction, '
                                    '5 imaginations, 15-step history, 37 observations')
    if name == 'duet_cfg4_train':
        return 'duet', synth.CFG2, ('DUET-Imagine fine-tuning iteration (forward + backward with the imagination-text aux '
                                    'loss, gradient all-reduce, AdamW step), 64 episodes/GPU x 6 navigation steps')
    raise SystemExit('unknown workload %r' % name)


# ----------------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown'}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        return {'sm_mhz': statistics.median(self.samples) if self.samples else None, 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ----------------------------------------------------------------------------------------------
# the step (shared by all legs)
# ----------------------------------------------------------------------------------------------
DUET_PANO_KEYS = ('view_img_fts', 'loc_fts', 'nav_types', 'view_lens')
DUET_NAV_KEYS = ('txt_masks', 'gmap_img_embeds', 'gmap_step_ids', 'gmap_pos_fts', 'gmap_masks', 'gmap_pair_dists',
                 'gmap_visited_masks', 'vp_img_embeds', 'vp_pos_fts', 'vp_masks', 'vp_nav_masks', 'imagine_masks')
HAMT_VIS_KEYS = ('txt_masks', 'ob_img_feats', 'ob_ang_feats', 'ob_nav_types', 'ob_masks', 'imagine_masks')
HAMT_HIST_KEYS = ('hist_img_feats', 'hist_ang_feats', 'hist_pano_img_feats', 'hist_pano_ang_feats')
LOGITS = {'duet': 'fused_logits', 'hamt': 'act_logits'}


def duet_step(model, d, txt, img):
    """every tensor the two calls of a step hand back, by name"""
    pano, pano_masks = model('panorama', {k: d[k] for k in DUET_PANO_KEYS})
    nav = model('navigation', {**{k: d[k] for k in DUET_NAV_KEYS}, 'txt_embeds': txt, 'imagine_embeds': img,
                               'gmap_vpids': d['gmap_vpids'], 'vp_cand_vpids': d['vp_cand_vpids']})
    return {'pano_embeds': pano, 'pano_masks': pano_masks, **{k: v for k, v in nav.items() if v is not None}}


def hamt_step(model, d, txt, img):
    """every tensor the two calls of a step hand back, by name"""
    out = model('visual', txt_embeds=txt, hist_embeds=d['hist_list'], hist_lens=d['hist_lens'], imagine_embeds=img,
                **{k: d[k] for k in HAMT_VIS_KEYS})
    h = model('history', ob_step=d['ob_step'], **{k: d[k] for k in HAMT_HIST_KEYS})
    return {'act_logits': out[0], 'hist_embeds': h}


DUMP_BYTES = 64 << 20                                   # --dump-outputs writes at most this much in all
NONFINITE = '_nonfinite'                                # <name>_nonfinite.npy: 0 finite, -1 -inf, 1 +inf, 2 NaN


def dump_outputs(directory, outputs):
    """--dump-outputs: every tensor of ``outputs`` ({name: tensor}) as directory/<name>.npy in float32, every element finite.
    Masked logits are -inf, so a tensor with non-finite elements is written with 0 in their place, and beside it
    <name>_nonfinite.npy of the same shape tells which they were (load_dump puts them back).  When together the files would
    exceed DUMP_BYTES, the smaller tensors are written whole and what is left of the budget is shared evenly by the others,
    each written as a fixed sample of its elements (flat indices from a generator seeded with the name, in increasing order),
    so that every run with the same arguments writes the same elements."""
    os.makedirs(directory, exist_ok=True)
    left = DUMP_BYTES // 4
    items = sorted(outputs.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        t = t.detach().float()
        files = 1 if bool(torch.isfinite(t).all()) else 2
        share = left // (len(items) - i) // files
        if t.numel() > share:
            idx = np.unique(np.random.default_rng(zlib.crc32(name.encode())).integers(0, t.numel(), share))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        left -= a.size * files
        fin = np.isfinite(a)
        np.save(os.path.join(directory, name + '.npy'), np.where(fin, a, 0).astype(np.float32))
        if files == 2:
            code = np.select([fin, np.isnan(a), a > 0], [0, 2, 1], -1).astype(np.float32)
            np.save(os.path.join(directory, name + NONFINITE + '.npy'), code)


def load_dump(directory):
    """{name: float32 array} of what dump_outputs wrote to ``directory``, the non-finite elements put back"""
    out = {}
    for f in sorted(os.listdir(directory)):
        if not f.endswith('.npy') or f.endswith(NONFINITE + '.npy'):
            continue
        name = f[:-4]
        a = np.load(os.path.join(directory, f))
        code_file = os.path.join(directory, name + NONFINITE + '.npy')
        if os.path.exists(code_file):
            code = np.load(code_file)
            a = np.where(code == 0, a, np.select([code == -1, code == 1], [-np.inf, np.inf], np.nan)).astype(np.float32)
        out[name] = a
    return out


def build(model_kind, shape, rank, precision):
    import vln_imagine_b200.synth as synth
    from vln_imagine_b200 import config
    if model_kind == 'duet':
        from vln_imagine_b200 import duet
        model = duet.VLNBert(config.default_duet_args()).cuda().eval()
        ep = synth.duet_episode(shape, 1234 + rank)
    else:
        from vln_imagine_b200 import hamt
        model = hamt.VLNBertCMT(config.default_hamt_args()).cuda().eval()
        ep = synth.hamt_episode(shape, 1234 + rank)
    shapes = {k: list(v.shape) for k, v in model.vln_bert.state_dict().items()}
    model.vln_bert.load_state_dict(synth.synth_state_dict(shapes, seed=0))
    model.vln_bert.precision = precision
    return model, synth.to_torch(ep)


def episode_prelude(model_kind, model, d):
    """once per episode: language -> imagine -> align (not part of a step; timed separately)"""
    if model_kind == 'duet':
        txt = model('language', {'txt_ids': d['txt_ids'], 'txt_masks': d['txt_masks']})
        img = model('imagine', {'imagine_feats': d['imagine_feats'], 'imagine_masks': None})
        loss, img2 = model('align_with_contrastive_loss', {
            'align_txt_embeds': txt, 'txt_masks': d['txt_masks'], 'align_imagine_embeds': img,
            'imagine_masks': d['imagine_masks'], 'sub_instr_segs': d['sub_instr_segs'],
            'sub_instr_imag_flag': d['sub_instr_imag_flag'], 'noun_phrase_segs': d['noun_phrase_segs'],
            'obs_instr_ids': d['obs_instr_ids']})
    else:
        txt = model('language', txt_ids=d['txt_ids'], txt_masks=d['txt_masks'])
        img = model('imagine', imagine_pano_img_feats=d['imagine_feats'], imagine_masks=None)
        loss, img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=d['txt_masks'],
                           align_imagine_embeds=img, imagine_masks=d['imagine_masks'], sub_instr_segs=d['sub_instr_segs'],
                           sub_instr_imag_flag=d['sub_instr_imag_flag'], noun_phrase_segs=d['noun_phrase_segs'],
                           obs_instr_ids=d['obs_instr_ids'])
    return txt, img2, loss


def step_tensor_keys(model_kind):
    return (DUET_PANO_KEYS + DUET_NAV_KEYS) if model_kind == 'duet' else (HAMT_VIS_KEYS + HAMT_HIST_KEYS + ('hist_embeds',))


def device_inputs(model_kind, model, ep, dev):
    d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in ep.items()}
    if model_kind == 'duet':
        G, P = ep['gmap_img_embeds'].shape[1], ep['vp_img_embeds'].shape[1]
        d['gmap_vpids'], d['vp_cand_vpids'] = model.vln_bert.intern_vpids(ep['gmap_vpids'], ep['vp_cand_vpids'], G, P, dev)
    else:
        d['hist_list'] = [d['hist_embeds'][:, t] for t in range(d['hist_embeds'].shape[1])]
        d['hist_lens'] = ep['hist_lens'].to(dev)          # device tensor: the whole-step graph must not copy from host
    return d


# ----------------------------------------------------------------------------------------------
# CPU legs (the oracle is the checker / reported baseline, never the product)
# ----------------------------------------------------------------------------------------------
def ncu_gemm_traffic(workload_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the tcgen05 GEMM, averaged over the GEMM launches of one
    step, from the committed `ncu --set full` capture of this workload (profiles/*_<workload>_step_full.csv, written by
    tools/profile.sh + tools/ncu_summary.py).  None when no capture of the workload is committed."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, 'profiles', '*_%s_step_full.csv' % workload_name)))
    if not files:
        return None, None
    tot, n = 0.0, 0
    with open(files[-1]) as f:
        for row in csv.DictReader(f):
            if row['kernel'].startswith('gemm_bf16_tc_kernel'):
                tot += float(row['dram_read_B']) + float(row['dram_write_B'])
                n += 1
    if n == 0:
        return None, None
    return tot / n, 'bytes per launch, mean over %d GEMM launches of one step in profiles/%s' % (n, os.path.basename(files[-1]))


def glue_leg(dev, batch, with_cpu):
    """Per-step graph glue of a DUET rollout (SURVEY.md 8(f) N1 / N2): DeviceGraphMaps (csrc/vi_graph.cu) through its host
    API, host packing and the packed upload included, against the CPU oracle of the reference's GraphMap loops on the same
    synthetic rollout.  Reported next to the metric, not part of it (the reference runs this in Python on the host)."""
    import vln_imagine_b200.synth as synth
    from vln_imagine_b200 import graph_map
    world = synth.nav_world(seed=21, n_vp=80, batch=batch, steps=7, hidden=768, degree=4)

    def rollout():
        gm = graph_map.DeviceGraphMaps(world[0]['obs'], dev)
        for t, st in enumerate(world):
            obs, ended = st['obs'], st['ended']
            gm.set_step_ids(obs, t, ended)
            pin = {'cand_vpids': [[c['viewpointId'] for c in ob['candidate']] for ob in obs], 'view_lens': st['view_lens_d'],
                   'nav_types': st['nav_types_d']}
            out = gm.nav_inputs(obs, st['pano_d'], st['masks_d'], pin, ended)
            if t + 1 < len(world):
                gm.update_graph(world[t + 1]['obs'], ended)
        return out
    for st in world:
        st['pano_d'] = torch.from_numpy(st['pano_embeds']).to(dev)
        st['masks_d'] = torch.ones(st['pano_d'].shape[:2], dtype=torch.bool, device=dev)
        st['view_lens_d'] = torch.from_numpy(st['view_lens']).to(dev)
        st['nav_types_d'] = torch.from_numpy(st['nav_types']).to(dev)
    rollout()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        rollout()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / reps / len(world) * 1e3
    res = {'what': 'graph update + node embeddings + position features + pair distances for %d episodes, ~%d known nodes, '
                   'wall time per step incl. host id interning and the packed upload' % (batch, 30),
           'ms_per_step': ms, 'launches_per_step': 3}
    if with_cpu:
        from oracle import graph_oracle as GO
        t0 = time.perf_counter()
        obs0 = world[0]['obs']
        states = [GO.GraphState(ob['viewpoint'], 768) for ob in obs0]
        for b, ob in enumerate(obs0):
            states[b].update_graph(ob['viewpoint'], ob['position'], [(c['viewpointId'], c['position']) for c in ob['candidate']])
        for t, st in enumerate(world):
            obs, ended = st['obs'], st['ended']
            cur = [s_.index[ob['viewpoint']] for s_, ob in zip(states, obs)]
            cands = [[s_.index[c['viewpointId']] for c in ob['candidate']] for s_, ob in zip(states, obs)]
            GO.update_node_embeds(states, cur, cands, st['pano_embeds'], np.ones(st['pano_embeds'].shape[:2], bool), ended)
            heads, elevs = [ob['heading'] for ob in obs], [ob['elevation'] for ob in obs]
            GO.nav_gmap_variable(states, cur, heads, elevs)
            GO.nav_vp_variable(states, cur, heads, elevs, st['pano_embeds'], cands, st['view_lens'], st['nav_types'])
            if t + 1 < len(world):
                for b, ob in enumerate(world[t + 1]['obs']):
                    if not ended[b]:
                        states[b].update_graph(ob['viewpoint'], ob['position'], [(c['viewpointId'], c['position']) for c in ob['candidate']])
        res['cpu_oracle_ms_per_step'] = (time.perf_counter() - t0) / len(world) * 1e3
    return res


def load_reference(model_kind):
    """(module, root) - the UNMODIFIED reference model class (GlocalTextPathNavCMT / NavCMT) built from the reference checkout
    (/root/reference in the build container) or from its files staged under baseline/_ref by tools/make_baseline_ref.py (the GPU
    box), with the synthetic weights; (None, why) when neither is present.  Harness-side shims only (oracle/gen_golden.py)."""
    for root in (os.environ.get('VLN_REFERENCE'), '/root/reference', os.path.join(ROOT, 'baseline', '_ref')):
        sub = ('VLN-DUET', 'map_nav_src') if model_kind == 'duet' else ('VLN-HAMT', 'finetune_src')
        if root and os.path.isfile(os.path.join(root, *sub, 'models', 'vilmodel.py' if model_kind == 'duet' else 'vilmodel_cmt.py')):
            try:
                from oracle import gen_golden
                gen_golden.REF = root
                import vln_imagine_b200.synth as synth
                ref = gen_golden.build_reference(model_kind)
                shapes = {k: list(v.shape) for k, v in ref.state_dict().items()}
                ref.load_state_dict(synth.synth_state_dict(shapes, seed=0))
                return ref, root
            except Exception as e:                      # a missing dependency of the reference tree: fall back to the port
                return None, '%s: %s' % (type(e).__name__, str(e)[:200])
    return None, 'no reference files (neither /root/reference nor baseline/_ref)'


def reference_stepper(model_kind, shape, device='cpu', seed=1234):
    """(step() -> logits, kind, note): one navigation decision per episode of the workload shape through the reference's own
    modules (kind 'reference'), or through the oracle port of them when the reference files are absent (kind 'port')."""
    import vln_imagine_b200.synth as synth
    from oracle import duet_oracle, hamt_oracle
    ep = synth.to_torch((synth.duet_episode if model_kind == 'duet' else synth.hamt_episode)(shape, seed))
    ep = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in ep.items()}
    g = torch.Generator().manual_seed(1)                 # the step's cost does not depend on the context VALUES
    txt = torch.randn(shape.batch, shape.instr_len, 768, generator=g).to(device)
    img2 = torch.randn(shape.batch, shape.n_imagine, 768, generator=g).to(device)
    ref, root = load_reference(model_kind)
    if ref is None:
        man = json.load(open(os.path.join(ROOT, 'tests', 'golden', '%s_manifest.json' % model_kind)))
        sd = {k: v.to(device) for k, v in synth.synth_state_dict(man, seed=0).items()}
        O = duet_oracle if model_kind == 'duet' else hamt_oracle
        if model_kind == 'duet':
            return (lambda: O.nav_step(sd, ep, txt, img2)[2]['fused_logits']), 'port', 'oracle port (%s)' % root
        return (lambda: O.nav_step(sd, ep, txt, img2)[0]), 'port', 'oracle port (%s)' % root
    ref = ref.to(device)
    if model_kind == 'duet':
        pano_in = {'view_img_fts': ep['view_img_fts'], 'obj_img_fts': None, 'loc_fts': ep['loc_fts'], 'nav_types': ep['nav_types'],
                   'view_lens': ep['view_lens'], 'obj_lens': None}
        nav_in = {k: ep[k] for k in ('txt_masks', 'gmap_img_embeds', 'gmap_step_ids', 'gmap_pos_fts', 'gmap_masks', 'gmap_pair_dists',
                                     'gmap_visited_masks', 'gmap_vpids', 'vp_img_embeds', 'vp_pos_fts', 'vp_masks', 'vp_nav_masks',
                                     'vp_cand_vpids', 'imagine_masks')}
        nav_in.update(txt_embeds=txt, imagine_embeds=img2, vp_obj_masks=None)

        def step():
            ref('panorama', pano_in)
            return ref('navigation', nav_in)['fused_logits']
    else:
        hm = hamt_oracle.hist_masks_from_lens(ep['hist_lens'], ep['hist_embeds'].shape[1]).to(device)
        step_ids = torch.LongTensor([ep['ob_step']]).to(device)

        def step():
            out = ref('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=ep['hist_embeds'], hist_masks=hm,
                      ob_img_feats=ep['ob_img_feats'], ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'],
                      ob_masks=ep['ob_masks'], imagine_embeds=img2, imagine_masks=ep['imagine_masks'])
            ref('history', hist_img_feats=ep['hist_img_feats'], hist_ang_feats=ep['hist_ang_feats'], ob_step_ids=step_ids,
                hist_pano_img_feats=ep['hist_pano_img_feats'], hist_pano_ang_feats=ep['hist_pano_ang_feats'])
            return out[0]
    return step, 'reference', 'unmodified reference modules from %s' % root


def eager_gpu_reference(model_kind, shape, budget_s=2.0):
    """The reference's own modules (else the oracle port), eager PyTorch on THIS GPU at the workload's batch size, in fp32 and
    under torch.autocast(bfloat16) - what running the reference on the same box looks like (SURVEY.md 8(d): "the real bar").
    A reported figure of the cpu_baseline leg; never a product path."""
    step, kind, note = reference_stepper(model_kind, shape, 'cuda')
    out = {'kind': kind, 'what': '%s, eager PyTorch on this GPU, %d episodes per step' % (note, shape.batch)}
    for tag, ctx in (('fp32', contextlib.nullcontext()), ('bf16_autocast', torch.autocast('cuda', dtype=torch.bfloat16))):
        try:
            with torch.no_grad(), ctx:
                step()
                torch.cuda.synchronize()
                n, t0 = 0, time.perf_counter()
                while time.perf_counter() - t0 < budget_s or n < 3:
                    step()
                    torch.cuda.synchronize()
                    n += 1
                dt = (time.perf_counter() - t0) / n
            out[tag] = {'value': shape.batch / dt, 'unit': UNIT, 'ms_per_step': dt * 1e3}
        except Exception as e:
            out[tag] = {'error': '%s: %s' % (type(e).__name__, str(e)[:200])}
    return out


def cpu_reference(model_kind, shape, budget_s=15.0):
    """The reference on the host cores (its own modules when staged under baseline/_ref, else the oracle port), fp32, all host
    threads, on a bounded sample of the same workload: steps of the workload's own batch for about budget_s seconds."""
    torch.set_num_threads(os.cpu_count())
    step, kind, note = reference_stepper(model_kind, shape, 'cpu')
    with torch.no_grad():
        step()                                              # warm-up
        times = []
        t_end = time.perf_counter() + budget_s
        while time.perf_counter() < t_end or len(times) < 3:
            t0 = time.perf_counter()
            step()
            times.append(time.perf_counter() - t0)
    best = min(times)
    return {'value': shape.batch / best, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': kind,
            'sample': '%d-episode steps (the workload batch) x %d repeats, best step %.1f ms, fp32 on the host CPU: %s'
                      % (shape.batch, len(times), best * 1e3, note)}, times


def run_reference_arm(args, model_kind, shape, desc, rank):
    """`--impl reference`: the reference's own CPU implementation of the path (its unmodified modules when staged, else the port)
    on the host cores, same workload shape and batch, exactly --steps steps after --warmup warm-up steps (rank 0 only)."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count())
    step, kind, note = reference_stepper(model_kind, shape, 'cpu')
    steps, warm = args.steps, args.warmup
    with torch.no_grad():
        for _ in range(warm):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = step()
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {LOGITS[model_kind]: out})
    B = shape.batch
    val = B * steps / dt
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
            'warmup': warm, 'ms_per_step': dt / steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': '%s: %s' % (args.workload, desc), 'episodes_per_step': B,
                       'requested': {'steps': args.steps, 'warmup': args.warmup},
                       'sample': 'each step = %d episodes (the workload batch) on the host CPU: %s' % (B, note)},
            'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': kind,
                             'sample': '%d-episode steps x %d, fp32, %d host threads: %s' % (B, steps, os.cpu_count(), note)},
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)



# ----------------------------------------------------------------------------------------------
# fine-tuning workload (BASELINE.json cfg-4): forward + backward + gradient all-reduce + optimiser step
# ----------------------------------------------------------------------------------------------
def train_measure(args, shape, rank, local_rank, world, K, W, detail=True, dump_dir=None):
    """Fine-tuning iterations (forward + backward + gradient all-reduce + clipping + AdamW) on this rank's episodes; the
    process group is the caller's.  Returns the measurements of rank 0's report (every rank must call it).  With dump_dir,
    rank 0 writes the loss, gradients and updated parameters of the last timed iteration there (dump_outputs)."""
    import torch.distributed as dist
    from vln_imagine_b200 import config, duet, ops, synth, train
    dev = torch.device('cuda', local_rank)
    T = 6                                                   # navigation steps per episode (SURVEY.md 8(d))
    B = shape.batch
    a = config.default_duet_args()
    model = duet.VLNBert(a).cuda()
    net = model.vln_bert
    shapes = {k: list(v.shape) for k, v in net.state_dict().items()}
    net.load_state_dict(synth.synth_state_dict(shapes, seed=0))
    net.precision = args.precision
    # train() mode with the released recipe's dropout (hidden / attention 0.1, feature dropout 0.4, projection head 0.15;
    # D/scripts/run_r2r.sh:66): counter-based masks, regenerated in the backward pass
    model.train()
    ep_host = synth.to_torch(synth.duet_episode(shape, 1234 + rank + int(os.environ.get('VI_BENCH_SEED_OFFSET', '0'))))
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in ep_host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))
    flat = train.FlatGradients(net)
    # the caller's optimiser (r2r/agent_base.py:141-160); capturable: its step is part of the replayed graph
    opt = torch.optim.AdamW(net.parameters(), lr=1e-5, fused=True, capturable=not args.no_graph)

    # data-parallel runs: the backward pass stops at the instruction embeddings, the all-reduce of everything but the text side
    # starts there and runs under the language encoder's backward (train.GraphedIteration(tail_fn=...)); VI_TRAIN_OVERLAP_AR=0: one
    # all-reduce after the whole backward pass
    fused_acc = os.environ.get('VI_TRAIN_FUSED_ACC', '1') != '0'
    lang_end = flat.prefix_end(net) if world > 1 and os.environ.get('VI_TRAIN_OVERLAP_AR', '1') != '0' else 0
    overlap = lang_end > 0
    pending = {}

    def grad_fn(ep):
        flat.zero()
        out = train.duet_finetune_iteration(model, ep, n_steps=T, fused_accumulation=fused_acc, split_language_backward=overlap)
        if overlap:
            pending['finish'] = out[4]
        return out[0].detach()

    def tail_fn():
        pending.pop('finish')()

    def before_tail():
        pending['work'] = flat.all_reduce_range(lang_end, flat.numel, async_op=True)

    def reduce_rest():
        w2 = flat.all_reduce_range(0, lang_end, async_op=True)
        for w in (pending.pop('work', None), w2):
            if w is not None:
                w.wait()

    def update_fn():
        torch.nn.utils.clip_grad_norm_(net.parameters(), 40.)         # agent_base.py:225
        opt.step()

    def iteration(ep):
        loss = grad_fn(ep)
        if overlap:
            before_tail()
            tail_fn()
            reduce_rest()
        else:
            flat.all_reduce()
        update_fn()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in ep_host.items()}
    G, P = ep_host['gmap_img_embeds'].shape[1], ep_host['vp_img_embeds'].shape[1]
    d['gmap_vpids'], d['vp_cand_vpids'] = net.intern_vpids(ep_host['gmap_vpids'], ep_host['vp_cand_vpids'], G, P, dev)
    host['gmap_vpids'], host['vp_cand_vpids'] = d['gmap_vpids'], d['vp_cand_vpids']
    for _ in range(W):
        iteration(d)
    torch.cuda.synchronize()
    n0 = ops._Counters.launches
    iteration(d)
    launches = ops._Counters.launches - n0
    eager_iteration = iteration
    graphed = None
    if not args.no_graph:
        if overlap:
            graphed = train.GraphedIteration(net, grad_fn, update_fn, d, between=reduce_rest, warmup=0, tail_fn=tail_fn, before_tail=before_tail)
        else:
            graphed = train.GraphedIteration(net, grad_fn, update_fn, d, between=flat.all_reduce, warmup=0)

        def iteration(ep):
            graphed.load(ep)
            return graphed.replay()
        for _ in range(2):
            iteration(d)
        torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    with sampler:
        e0.record()
        for _ in range(K):
            loss = iteration(d)
        e1.record()
        torch.cuda.synchronize()
    barrier()
    ms = e0.elapsed_time(e1)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {'loss': loss, 'gradients': flat.buffer,
                                'parameters': torch.cat([p.detach().reshape(-1) for p in flat.params])})
    # e2e: the iteration's inputs come from pinned host memory, the loss is read back
    barrier()
    e0.record()
    for _ in range(K):
        if graphed is not None:
            loss_host = float(iteration(host))              # pinned host tensors copied into the graph's static inputs
        else:
            dd = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in host.items()}
            loss_host = float(iteration(dd))
    e1.record()
    torch.cuda.synchronize()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    # the one collective of the path, alone: NCCL all-reduce (AVG) of the flat fp32 gradient buffer
    ar_ms = None
    if world > 1:
        barrier()
        for _ in range(2):
            flat.all_reduce()
        torch.cuda.synchronize()
        barrier()
        e0.record()
        for _ in range(5):
            flat.all_reduce()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / 5], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar_ms = float(t[0])
    loss_host = float(loss_host)
    res = dict(ms=ms, ms_e2e=ms_e2e, K=K, W=W, T=T, B=B, h2d=h2d, launches=launches, loss=loss_host,
               loss_finite=bool(np.isfinite(loss_host)), allreduce_ms=ar_ms, allreduce_bytes=flat.bytes(),
               allreduce_busbw_gbs=(2.0 * (world - 1) / world * flat.bytes() / (ar_ms * 1e-3) / 1e9) if ar_ms else None,
               clocks=sampler.summary(), graphed=graphed is not None, overlap=overlap,
               dropout=(net.config.hidden_dropout_prob, net.config.attention_probs_dropout_prob, model.drop_env.p))
    if graphed is not None:
        graphed.finish()
    if not detail:
        del graphed, opt, flat, model
        torch.cuda.empty_cache()
        return res
    # roofline of the GEMM kernel over one EAGER iteration (forward + dgrad + wgrad launches)
    iteration = eager_iteration
    torch.cuda.synchronize()
    torch.cuda._sleep(400_000_000)                          # ~0.2 s head start: the host queues ~4000 launches
    ops._Counters.gemm_trace = []
    iteration(d)
    torch.cuda.synchronize()
    trace, ops._Counters.gemm_trace = ops._Counters.gemm_trace, None
    gemm_flops = sum(2.0 * m * n * k for m, n, k, _, _ in trace)
    gemm_ms = sum(x.elapsed_time(y) for _, _, _, x, y in trace)
    torch.cuda._sleep(400_000_000)
    ops._Counters.trace = []
    iteration(d)
    torch.cuda.synchronize()
    tr2, ops._Counters.trace = ops._Counters.trace, None
    breakdown = {}
    for name, x, y in tr2:
        n_, t_ = breakdown.get(name, (0, 0.0))
        breakdown[name] = (n_ + 1, t_ + x.elapsed_time(y))
    breakdown = {k: {'launches': v[0], 'ms': round(v[1], 3)} for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1][1])}
    res.update(gemm_flops=gemm_flops, gemm_ms=gemm_ms, n_gemm=len(trace), breakdown=breakdown)
    return res


def run_train(args, shape, desc, rank, local_rank, world):
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    r = train_measure(args, shape, rank, local_rank, world, args.steps, args.warmup, detail=True, dump_dir=args.dump_outputs)
    ms, ms_e2e, K, W, T, B, h2d, launches, loss_host = (r[k] for k in ('ms', 'ms_e2e', 'K', 'W', 'T', 'B', 'h2d', 'launches', 'loss'))
    gemm_flops, gemm_ms, breakdown = r['gemm_flops'], r['gemm_ms'], r['breakdown']
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    fl_dec = flops_per_decision('duet', shape)
    C = shape.instr_len + shape.n_imagine
    fl_episode = 3.0 * (9 * _bert(shape.instr_len) + T * fl_dec)          # fwd + bwd ~ 3 x fwd (SURVEY.md 8(d))
    line = {
        'metric': METRIC + ' (fine-tuning: forward + backward + all-reduce + optimiser)', 'value': world * B * T * K / (ms * 1e-3),
        'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': ms / K, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': args.precision, 'data': 'synthetic',
        'config': {'workload': '%s: %s' % (args.workload, desc), 'episodes_per_gpu': B, 'nav_steps_per_iteration': T,
                   'replay': 'eager launches (autograd)' if args.no_graph else 'two CUDA graphs per iteration (forward + backward | '
                             'clipping + AdamW) around the eager NCCL all-reduce',
                   'dropout': 'on: hidden %.2f, attention %.2f, features %.2f, projection head 0.15'
                              % r['dropout'],
                   'l2': 'no flush: an iteration touches > 3 GB of weights, gradients and saved activations',
                   'collective': ('NCCL all-reduce (AVG) of the flat fp32 gradient buffer, %.0f MB, in two parts: everything but the text side '
                                  'starts when the backward pass reaches the instruction embeddings and runs under the language encoder\'s '
                                  'backward, the text side follows' if r.get('overlap') else
                                  'one NCCL all-reduce (AVG) of the flat fp32 gradient buffer, %.0f MB') % (r['allreduce_bytes'] / 1e6),
                   'weights': 'random-init (deterministic synthetic)'},
        'clocks': r['clocks'],
        'e2e': {'value': world * B * T * K / (ms_e2e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                'ms_per_step': ms_e2e / K, 'api': 'train.duet_finetune_iteration through the module API; episode batch copied '
                                                  'from pinned host memory every iteration, loss read back'},
        'gpu_launches': launches * K,
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved / peak_tf,
                     'traffic': None, 'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained' if peaks else 'fallback',
                     'kernel': 'gemm_bf16_tc_kernel + wgrad_tc_kernel (tcgen05): %d launches/iteration (forward, dgrad | wgrad incl. its split reduction), %.1f GFLOP executed, '
                               '%.3f ms of GEMM time' % (r['n_gemm'], gemm_flops / 1e9, gemm_ms)},
        'allreduce': {'ms': r['allreduce_ms'], 'bytes': r['allreduce_bytes'], 'busbw_gbs': r['allreduce_busbw_gbs']},
        'loss_finite': r['loss_finite'],
        'step': {'algorithmic_gflop_per_iteration': fl_episode * B / 1e9,
                 'tflops': fl_episode * B / (ms / K * 1e-3) / 1e12, 'launches_per_iteration': launches, 'loss': loss_host,
                 'breakdown': breakdown},
    }
    if not r['loss_finite']:
        line['invalid'] = 'the loss is not finite (%r): this is not a training measurement' % loss_host
    print(json.dumps(line), flush=True)
    if not r['loss_finite']:
        sys.exit(3)

# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='duet_cfg2')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--no-graph', action='store_true', help='time eager launches instead of a CUDA-graph replay')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed as DIR/<name>.npy '
                    '(float32, at most 64 MB in all; rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.manual_seed(1234 + rank)                      # the fine-tuning dropout seeds (autograd_ops.dropout_seed) follow it
    model_kind, shape, desc = workload(args.workload)

    if args.impl == 'reference':
        run_reference_arm(args, model_kind, shape, desc, rank)
        return
    if args.workload.endswith('_train'):
        run_train(args, shape, desc, rank, local_rank, world)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    from vln_imagine_b200 import graphs as vgraphs
    from vln_imagine_b200 import ops

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t)
        return ms

    model, ep = build(model_kind, shape, rank, args.precision)
    step_fn = duet_step if model_kind == 'duet' else hamt_step
    B = shape.batch
    K, W = args.steps, args.warmup
    # DUET keeps the K / V projections of the [txt ; imagine] context for the length of an episode (the reference
    # recomputes them identically at every step).  The bench is honest about it: every EP_LEN-th step is the first
    # step of a new episode and projects the context again (R2R paths are 4-6 hops + stop, SURVEY.md 8(d): T = 6).
    EP_LEN = 6
    ctx_cache = model_kind == 'duet' and model.vln_bert.context_cache

    def new_episode():
        if ctx_cache:
            model.vln_bert.drop_context()

    with torch.no_grad():
        d = device_inputs(model_kind, model, ep, dev)
        # ---- once-per-episode prelude (reported, not part of the metric)
        txt, img2, loss = episode_prelude(model_kind, model, d)
        torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(3):
            txt, img2, loss = episode_prelude(model_kind, model, d)
        t1.record(); torch.cuda.synchronize()
        prelude_ms = t0.elapsed_time(t1) / 3

        # ---- leg 1: inputs resident in HBM; the step replayed as a CUDA graph
        model.use_cuda_graphs = False                   # this leg captures the whole step itself
        for _ in range(3):
            step_fn(model, d, txt, img2)
        torch.cuda.synchronize()
        new_episode()
        n0 = ops._Counters.launches
        step_fn(model, d, txt, img2)                        # first step of an episode
        launches_first = ops._Counters.launches - n0
        n0 = ops._Counters.launches
        logits = step_fn(model, d, txt, img2)[LOGITS[model_kind]]      # a later step
        launches_later = ops._Counters.launches - n0
        state = {'i': 0}
        if not args.no_graph:
            def capture(first):
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    step_fn(model, d, txt, img2)
                torch.cuda.current_stream().wait_stream(side)
                if first:
                    new_episode()                           # the capture then contains the context projections
                g = torch.cuda.CUDAGraph()
                with vgraphs.capture(g):
                    out = step_fn(model, d, txt, img2)      # every replay of g writes its results into these tensors
                return g, out
            g_later, out_later = capture(False)
            g_first, out_first = capture(True) if ctx_cache else (g_later, out_later)

            def run():
                (g_first if state['i'] % EP_LEN == 0 else g_later).replay()
                state['i'] += 1
        else:
            def run():
                if state['i'] % EP_LEN == 0:
                    new_episode()
                state['out'] = step_fn(model, d, txt, img2)
                state['i'] += 1
        for _ in range(W):
            run()
        sampler = ClockSampler(local_rank)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        state['i'] = 0
        with sampler:
            e0.record()
            for _ in range(K):
                run()
            e1.record()
            torch.cuda.synchronize()
        barrier()
        n_first = (K + EP_LEN - 1) // EP_LEN
        total_launches = n_first * launches_first + (K - n_first) * launches_later
        launches_per_step = launches_first
        ms = max_over_ranks(e0.elapsed_time(e1))
        value = world * B * K / (ms * 1e-3)
        if args.dump_outputs and rank == 0:
            last = state['out'] if args.no_graph else out_first if (K - 1) % EP_LEN == 0 else out_later
            dump_outputs(args.dump_outputs, last)

        # ---- leg 2 (e2e): public module API; every step's inputs that the reference agent builds on the host
        # (r2r/agent.py:57-207: panorama / location features, nav types, graph step ids, position features, pair
        # distances, masks, viewpoint-id strings) come from pinned HOST memory and the logits are copied out.  Tensors that
        # are products of earlier model calls stay on the device, exactly as in the reference: txt_embeds / imagine_embeds
        # (agent.py:409-449), the graph-node embeddings gmap_img_embeds (GraphMap, agent.py:468-479) and
        # vp_img_embeds = [0 ; pano_embeds of this step] (agent.py:173-186).
        DEVICE_RESIDENT = ('gmap_img_embeds', 'vp_img_embeds') if model_kind == 'duet' else ()
        keys = [k for k in step_tensor_keys(model_kind) if k in ep and torch.is_tensor(ep[k]) and k not in DEVICE_RESIDENT]
        host = {k: ep[k].pin_memory() for k in keys}
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        out_host = torch.empty(tuple(logits.shape), dtype=logits.dtype).pin_memory()
        d2h = out_host.numel() * out_host.element_size()

        model.use_cuda_graphs = not args.no_graph       # the module API replays its own per-mode graphs
        if model_kind == 'duet':                         # the agent hands viewpoint-id STRINGS to the API
            host_lists = {'gmap_vpids': ep['gmap_vpids'], 'vp_cand_vpids': ep['vp_cand_vpids']}
        else:
            host_lists = {}
            hist_lens_host = [int(x) for x in ep['hist_lens']]

        def e2e_step(i):
            if i % EP_LEN == 0:
                new_episode()
            dd = dict(d)
            dd.update(host)                              # pinned host tensors: the API copies them in
            dd.update(host_lists)
            if model_kind == 'hamt':
                hh = host['hist_embeds'].to(dev, non_blocking=True)
                dd['hist_list'] = [hh[:, t] for t in range(hh.shape[1])]
                dd['hist_lens'] = hist_lens_host             # python ints, as the agent passes them
                lg = step_fn(model, dd, txt, img2)['act_logits']
            else:
                pano, _ = model('panorama', {k: dd[k] for k in DUET_PANO_KEYS})
                dd['vp_img_embeds'] = torch.cat([torch.zeros_like(pano[:, :1]), pano], 1)     # agent.py:173-186
                lg = model('navigation', {**{k: dd[k] for k in DUET_NAV_KEYS}, 'txt_embeds': txt, 'imagine_embeds': img2,
                                          'gmap_vpids': dd['gmap_vpids'], 'vp_cand_vpids': dd['vp_cand_vpids']})['fused_logits']
            out_host.copy_(lg, non_blocking=True)
            torch.cuda.current_stream().synchronize()          # the agent needs the logits to act

        for i in range(W):
            e2e_step(i)
        barrier()
        e0.record()
        for i in range(K):
            e2e_step(i)
        e1.record()
        torch.cuda.synchronize()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        e2e_value = world * B * K / (ms_e2e * 1e-3)

        model.use_cuda_graphs = False
        # ---- roofline of the dominant kernel (tcgen05 GEMM): CUDA events around every launch of 3 eager steps
        torch.cuda.synchronize()
        TRACE_STEPS = EP_LEN if ctx_cache else 3
        gemm_ms, gemm_flops, trace = float('inf'), 0.0, []
        for _ in range(2):                              # two passes, the less disturbed one counts
            new_episode()
            torch.cuda.synchronize()
            torch.cuda._sleep(200_000_000)              # ~0.1 s head start for the host: launches then queue back to back
            ops._Counters.gemm_trace = []               # and an event pair brackets device time only
            for _ in range(TRACE_STEPS):
                step_fn(model, d, txt, img2)
            torch.cuda.synchronize()
            tr, ops._Counters.gemm_trace = ops._Counters.gemm_trace, None
            t_ms = sum(a.elapsed_time(b) for _, _, _, a, b in tr)
            if t_ms < gemm_ms:
                gemm_ms, trace = t_ms, tr
                gemm_flops = sum(2.0 * m * n * k for m, n, k, _, _ in tr)
        # per-entry-point breakdown of one step, same method (diagnostic: the event pairs add ~1 us gaps)
        new_episode()
        torch.cuda.synchronize()
        torch.cuda._sleep(200_000_000)
        ops._Counters.trace = []
        for _ in range(TRACE_STEPS):
            step_fn(model, d, txt, img2)
        torch.cuda.synchronize()
        tr2, ops._Counters.trace = ops._Counters.trace, None
        breakdown = {}
        for name, a, b in tr2:
            n_, t_ = breakdown.get(name, (0, 0.0))
            breakdown[name] = (n_ + 1, t_ + a.elapsed_time(b))
        breakdown = {k: {'launches_per_step': round(v[0] / TRACE_STEPS, 2), 'ms_per_step': round(v[1] / TRACE_STEPS, 4)} for k, v in
                     sorted(breakdown.items(), key=lambda kv: -kv[1][1])}

    # cfg-4 beside the headline: a few fine-tuning iterations (forward + backward + NCCL gradient all-reduce + AdamW) on the
    # same ranks, so that the 1/2/4/8-GPU scaling runs also record the only collective this path has (every rank takes part)
    train_rec = None
    if model_kind == 'duet' and args.workload == 'duet_cfg2' and os.environ.get('VI_BENCH_TRAIN', '1') != '0':
        try:
            del model
            torch.cuda.empty_cache()
            tr_ = train_measure(args, shape, rank, local_rank, world, 4, 3, detail=False)
            train_rec = {'what': 'DUET-Imagine fine-tuning (cfg-4): %d episodes/GPU x %d navigation steps, forward + backward + gradient '
                                 'all-reduce + clipping + AdamW, dropout on, CUDA-graph replay' % (tr_['B'], tr_['T']),
                         'value': world * tr_['B'] * tr_['T'] * tr_['K'] / (tr_['ms'] * 1e-3), 'unit': UNIT,
                         'ms_per_iteration': tr_['ms'] / tr_['K'], 'iterations': tr_['K'], 'warmup': tr_['W'],
                         'allreduce_ms': tr_['allreduce_ms'], 'allreduce_bytes': tr_['allreduce_bytes'],
                         'allreduce_busbw_gbs': tr_['allreduce_busbw_gbs'], 'allreduce_overlapped': tr_.get('overlap', False),
                         'loss': tr_['loss'], 'loss_finite': tr_['loss_finite']}
        except Exception as e:                          # noqa: BLE001 - an auxiliary record must never cost the bench line
            train_rec = {'error': '%s: %s' % (type(e).__name__, str(e)[:300])}
            if world > 1:
                raise                                   # ranks must not diverge inside a collective

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
    peak_src = 'MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)' if peaks else 'fallback 1.4 PFLOP/s sustained'
    traffic, traffic_src = ncu_gemm_traffic(args.workload)
    fl_dec = flops_per_decision(model_kind, shape)
    step_tf = fl_dec * B / (ms / K * 1e-3) / 1e12
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    # the same kernel inside the replayed graph: the event pairs of the eager trace add a gap to every launch (their sum over ALL
    # kernels exceeds the replayed step), so the GEMM's time inside the timed region is estimated as its SHARE of the traced step
    # times the replayed step - an explanation next to the contract figure above, not a replacement for it
    traced_total = sum(v['ms_per_step'] for v in breakdown.values()) if breakdown else 0.0
    gemm_share = (breakdown.get('vi_gemm16', {}).get('ms_per_step', 0.0) / traced_total) if traced_total > 0 else None
    in_graph = None
    if gemm_share:
        in_graph_ms = gemm_share * ms / K
        in_graph = {'share_of_traced_step': gemm_share, 'ms_per_step': in_graph_ms,
                    'achieved': gemm_flops / TRACE_STEPS / (in_graph_ms * 1e-3) / 1e12,
                    'frac': gemm_flops / TRACE_STEPS / (in_graph_ms * 1e-3) / 1e12 / peak_tf}
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': args.precision, 'data': 'synthetic',
        'config': {'workload': '%s: %s' % (args.workload, desc), 'episodes_per_gpu': B,
                   'replay': 'eager launches' if args.no_graph else 'CUDA graph of the step',
                   'l2': 'no flush: each step streams 150+ MB of bf16 weights plus activations, more than the 126 MB L2',
                   'episode_len': EP_LEN if ctx_cache else None,
                   'context_cache': ('K/V projections of [txt;imagine] computed at the first step of each %d-step episode and '
                                     'reused by the other %d (the reference recomputes them every step); value counts '
                                     'wall time over all steps' % (EP_LEN, EP_LEN - 1)) if ctx_cache else 'n/a',
                   'weights': 'random-init (deterministic synthetic), shared with the oracle'},
        'clocks': sampler.summary(),
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': ms_e2e / K, 'api': 'the module API (DUET panorama+navigation / HAMT visual+history) called with the per-step inputs the '
                       'reference agent builds on the host (pinned): features, position features, ids, distances, masks, '
                       'viewpoint-id strings; products of earlier model calls (txt / imagine embeds, graph-node embeds, '
                       'vp_img_embeds = [0; pano_embeds]) stay on the device as in the reference (r2r/agent.py:173-186,409-479). '
                       'The API copies host tensors into the static buffers of its per-mode CUDA graphs, replays, and the '
                       'logits are read back and synchronised every step'},
        'gpu_launches': total_launches,
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s',
                     'frac': achieved / peak_tf, 'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                     'kernel': 'gemm_bf16_tc_kernel (tcgen05): %.1f launches/step, %.1f GFLOP/step EXECUTED, %.3f ms/step of GEMM '
                               'time (CUDA events around each launch of %d queued eager steps = one episode)'
                               % (len(trace) / TRACE_STEPS, gemm_flops / TRACE_STEPS / 1e9, gemm_ms / TRACE_STEPS, TRACE_STEPS),
                     'in_replayed_graph_estimate': in_graph},
        'step': {'algorithmic_gflop_per_decision': fl_dec / 1e9, 'tflops': step_tf, 'frac_of_peak': step_tf / peak_tf,
                 'executed_gemm_gflop_per_decision': gemm_flops / TRACE_STEPS / B / 1e9,
                 'launches_first_step_of_episode': launches_first, 'launches_later_steps': launches_later,
                 'prelude_ms_per_episode_batch': prelude_ms,
                 'breakdown': breakdown},
    }
    if train_rec is not None:
        line['train'] = train_rec
    if world == 1 and not args.no_cpu_baseline:
        cb, _ = cpu_reference(model_kind, shape)
        line['cpu_baseline'] = cb
        if model_kind == 'duet':
            try:                                        # an auxiliary figure must never cost the bench line
                cb['reference_torch_eager_on_this_gpu'] = eager_gpu_reference(model_kind, shape)
            except Exception as e:                      # noqa: BLE001
                cb['reference_torch_eager_on_this_gpu'] = {'error': '%s: %s' % (type(e).__name__, str(e)[:200])}
    if world == 1 and model_kind == 'duet':
        try:                                            # an auxiliary figure must never cost the bench line
            line['step']['graph_glue'] = glue_leg(dev, B, with_cpu=not args.no_cpu_baseline)
        except Exception as e:                          # noqa: BLE001
            line['step']['graph_glue'] = {'error': '%s: %s' % (type(e).__name__, e)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
