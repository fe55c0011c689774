"""Data-parallel fine-tuning plumbing for the navigation hot path (BASELINE.json cfg-4, SURVEY.md section 8(e)).

One process per GPU; episodes are sharded by rank; weights are replicated.  The only collective on the path is ONE
all-reduce of a flat gradient buffer per iteration (NCCL over NVLink / NVSwitch; average = the reference's
DistributedDataParallel semantics, VLN-DUET/map_nav_src/r2r/agent_base.py:131-134 + utils/distributed.py).
Everything before it - forward and backward of every mode - runs in libvlnimagine kernels recorded through
autograd_ops; the optimiser and the gradient clipping stay the caller's (agent_base.py:223-228).

    flat = FlatGradients(model)                 # .grad of every trainable parameter becomes a view of one buffer
    loss = duet_finetune_iteration(model, ep)   # prelude + T navigation steps, teacher forcing, loss.backward()
    flat.all_reduce()                           # one collective
    torch.nn.utils.clip_grad_norm_(model.parameters(), 40.); optimizer.step(); flat.zero()
"""
from __future__ import annotations

from typing import Iterable, List, Optional

import torch
import torch.distributed as dist

from . import graphs


class FlatGradients:
    """All trainable parameters' gradients in ONE contiguous fp32 buffer (parameter order = ``named_parameters()``
    order, each segment padded to 16 bytes).  ``p.grad`` is a view of the buffer, so autograd accumulates in place
    and the all-reduce needs no packing copy."""

    ALIGN = 4      # elements (16 bytes)

    def __init__(self, module: torch.nn.Module, params: Optional[Iterable[torch.nn.Parameter]] = None):
        ps = [p for p in (params if params is not None else module.parameters()) if p.requires_grad]
        if not ps:
            raise ValueError('FlatGradients: no trainable parameters')
        dev, dt = ps[0].device, ps[0].dtype
        self.params: List[torch.nn.Parameter] = ps
        self.offsets = []
        off = 0
        for p in ps:
            if p.device != dev or p.dtype != dt:
                raise ValueError('FlatGradients: parameters must share a device and a dtype')
            self.offsets.append(off)
            off += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.numel = off
        self.buffer = torch.zeros(off, dtype=dt, device=dev)
        self.attach()

    def attach(self):
        """(re)point every .grad at its segment (needed again after ``zero_grad(set_to_none=True)``)"""
        for p, off in zip(self.params, self.offsets):
            p.grad = self.buffer[off:off + p.numel()].view_as(p)

    def zero(self):
        self.buffer.zero_()
        self.attach()

    def all_reduce(self, group=None, async_op: bool = False):
        """average over the ranks of ``group``; no-op without an initialised process group or with one rank"""
        if not dist.is_available() or not dist.is_initialized():
            return None
        world = dist.get_world_size(group)
        if world == 1:
            return None
        if dist.get_backend(group) == 'nccl':
            return dist.all_reduce(self.buffer, op=dist.ReduceOp.AVG, group=group, async_op=async_op)
        work = dist.all_reduce(self.buffer, op=dist.ReduceOp.SUM, group=group, async_op=False)   # gloo: host-logic tests
        self.buffer.div_(world)
        return work

    def bytes(self) -> int:
        return self.numel * self.buffer.element_size()

    def prefix_end(self, module: torch.nn.Module, prefixes=('embeddings.', 'lang_encoder.')) -> int:
        """Buffer offset behind the leading parameters whose names start with one of ``prefixes`` (the text side: the only
        parameters the LAST part of the backward pass - the language encoder - still writes).  0 when the order does not allow it."""
        names = {id(p): n for n, p in module.named_parameters()}
        end = 0
        for p, off in zip(self.params, self.offsets):
            n = names.get(id(p), '')
            if not any(n.startswith(x) for x in prefixes):
                break
            end = off + (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        # every text-side parameter must sit inside the prefix
        for p, off in zip(self.params, self.offsets):
            if off >= end and any(names.get(id(p), '').startswith(x) for x in prefixes):
                return 0
        return end

    def all_reduce_range(self, lo: int, hi: int, group=None, async_op: bool = False):
        """average buffer[lo:hi] over the ranks (the two halves of an overlapped gradient all-reduce)"""
        if hi <= lo or not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
            return None
        seg = self.buffer[lo:hi]
        if dist.get_backend(group) == 'nccl':
            return dist.all_reduce(seg, op=dist.ReduceOp.AVG, group=group, async_op=async_op)
        dist.all_reduce(seg, op=dist.ReduceOp.SUM, group=group, async_op=False)
        seg.div_(dist.get_world_size(group))
        return None


def teacher_targets(gmap_masks: torch.Tensor, gmap_visited_masks: torch.Tensor) -> torch.Tensor:
    """Synthetic teacher action: the last admissible graph node (valid and not visited); [stop] (0) if none.
    Stands in for _teacher_action_r4r (r2r/agent.py:209-262), which needs the simulator."""
    ok = gmap_masks.bool() & ~gmap_visited_masks.bool()
    idx = torch.arange(ok.shape[1], device=ok.device)[None, :].expand_as(ok)
    return torch.where(ok, idx, torch.zeros_like(idx)).max(1).values


def duet_finetune_iteration(model, ep: dict, n_steps: int = 1, cosine_weight: float = 0.5, ml_weight: float = 1.0,
                            backward: bool = True, fused_accumulation: bool = False, split_language_backward: bool = False):
    """One imitation-learning iteration of the reference agent on a batch of episodes (r2r/agent.py:384-623):
    language + imagine + align once, then ``n_steps`` navigation steps (panorama -> navigation -> summed
    cross-entropy on the fused logits), loss = ml_weight * CE / B + cosine_weight * aux.  ``model`` is the drop-in
    VLNBert; ``ep`` holds device tensors (vln-imagine_b200/synth.py layout).  Returns (loss, ce, aux, last nav dict).
    ``fused_accumulation``: the per-step parameter gradients are summed inside the backward kernels instead of by one autograd
    ``add`` per parameter per step (autograd_ops.fused_grad_accumulation); same .grad at the end, not for DDP-wrapped modules.
    ``split_language_backward``: the backward pass stops at the instruction embeddings - every gradient except the text side
    (embeddings.*, lang_encoder.*) is then final - and a fifth return value ``finish()`` runs the rest (the language encoder's
    backward): the caller can start the all-reduce of the finished part in between (GraphedIteration(tail_fn=...))."""
    B = ep['txt_ids'].shape[0]
    txt = model('language', {'txt_ids': ep['txt_ids'], 'txt_masks': ep['txt_masks']})
    txt_graph = None
    if split_language_backward and backward and txt.requires_grad:
        txt_graph, txt = txt, txt.detach().requires_grad_(True)             # the navigation part sees a leaf
    img = model('imagine', {'imagine_feats': ep['imagine_feats'], 'imagine_masks': None})
    aux, img2 = model('align_with_contrastive_loss', {
        'align_txt_embeds': txt, 'txt_masks': ep['txt_masks'], 'align_imagine_embeds': img,
        'imagine_masks': ep['imagine_masks'], 'sub_instr_segs': ep['sub_instr_segs'],
        'sub_instr_imag_flag': ep['sub_instr_imag_flag'], 'noun_phrase_segs': ep['noun_phrase_segs'],
        'obs_instr_ids': ep['obs_instr_ids']})
    tgt = teacher_targets(ep['gmap_masks'], ep['gmap_visited_masks'])
    ce = None
    nav = None
    for _ in range(n_steps):
        pano, _ = model('panorama', {'view_img_fts': ep['view_img_fts'], 'obj_img_fts': None, 'loc_fts': ep['loc_fts'],
                                     'nav_types': ep['nav_types'], 'view_lens': ep['view_lens'], 'obj_lens': None})
        vp_img = torch.cat([torch.zeros_like(pano[:, :1]), pano], 1)                  # r2r/agent.py:173-186
        nav = model('navigation', {k: ep[k] for k in (
            'txt_masks', 'gmap_img_embeds', 'gmap_step_ids', 'gmap_pos_fts', 'gmap_masks', 'gmap_pair_dists',
            'gmap_visited_masks', 'gmap_vpids', 'vp_pos_fts', 'vp_masks', 'vp_nav_masks', 'vp_cand_vpids',
            'imagine_masks')} | {'txt_embeds': txt, 'imagine_embeds': img2, 'vp_obj_masks': None, 'vp_img_embeds': vp_img})
        step_ce = torch.nn.functional.cross_entropy(nav['fused_logits'], tgt, reduction='sum')     # agent_base.py:162
        ce = step_ce if ce is None else ce + step_ce
    loss = ce * (ml_weight / B) + cosine_weight * aux
    if backward:
        from . import autograd_ops as ag
        with ag.fused_grad_accumulation(fused_accumulation):
            loss.backward()
        if split_language_backward:
            leaf = txt

            def finish():
                """second half of the backward pass: the language encoder"""
                if txt_graph is not None and leaf.grad is not None:
                    with ag.fused_grad_accumulation(fused_accumulation):
                        txt_graph.backward(leaf.grad)
            return loss, ce / B, aux, nav, finish
    return loss, ce / B, aux, nav


def hamt_stop_tokens(ob_nav_types: torch.Tensor) -> torch.Tensor:
    """Index of the [stop] observation token per episode: the last admissible one (nav_type != 0), which is where HAMT's agent
    places it after the candidates (ob_cand_lens - 1, r2r/agent_cmt.py).  Also the synthetic teacher action of the IL rollout,
    standing in for _teacher_action (which needs the simulator), as in the gradient fixtures."""
    ok = ob_nav_types != 0
    idx = torch.arange(ok.shape[1], device=ok.device)[None, :].expand_as(ok)
    return torch.where(ok, idx, torch.zeros_like(idx)).max(1).values


def _hamt_rollout(model, ep: dict, n_steps: int, step):
    """language + imagine + align once, then ``n_steps`` calls of 'visual' followed by 'history' with the history growing by one
    token per step (r2r/agent_cmt.py:371-605); ``step(t, txt, img2, hist_embeds, hist_lens)`` runs the 'visual' call and whatever
    the rollout does with it.  Returns (aux, the last step's inputs for a bootstrap call)."""
    B = ep['txt_ids'].shape[0]
    dev = ep['txt_ids'].device
    txt = model('language', txt_ids=ep['txt_ids'], txt_masks=ep['txt_masks'])
    img = model('imagine', imagine_pano_img_feats=ep['imagine_feats'], imagine_masks=None)
    aux, img2 = model('align_with_contrastive_loss', align_txt_embeds=txt, txt_masks=ep['txt_masks'], align_imagine_embeds=img,
                      imagine_masks=ep['imagine_masks'], sub_instr_segs=ep['sub_instr_segs'],
                      sub_instr_imag_flag=ep['sub_instr_imag_flag'], noun_phrase_segs=ep['noun_phrase_segs'],
                      obs_instr_ids=ep['obs_instr_ids'])
    hist = [model('history').expand(B, -1)]
    for t in range(n_steps):
        step(txt, img2, hist, torch.full((B,), t + 1, dtype=torch.int64, device=dev))
        hist.append(model('history', hist_img_feats=ep['hist_img_feats'], hist_ang_feats=ep['hist_ang_feats'], ob_step=t,
                          hist_pano_img_feats=ep['hist_pano_img_feats'], hist_pano_ang_feats=ep['hist_pano_ang_feats']))
    return aux, (txt, img2, hist, torch.full((B,), n_steps + 1, dtype=torch.int64, device=dev))


def _hamt_visual(model, ep, txt, img2, hist, lens, return_states=False):
    return model('visual', txt_embeds=txt, txt_masks=ep['txt_masks'], hist_embeds=hist, hist_lens=lens, ob_img_feats=ep['ob_img_feats'],
                 ob_ang_feats=ep['ob_ang_feats'], ob_nav_types=ep['ob_nav_types'], ob_masks=ep['ob_masks'], imagine_embeds=img2,
                 imagine_masks=ep['imagine_masks'], return_states=return_states)


def hamt_finetune_iteration(model, critic, ep: dict, n_steps: int, rewards: torch.Tensor, ml_weight: float = 0.2, gamma: float = 0.9,
                            entropy_weight: float = 0.01, normalize: str = 'total', aux_weight: float = 0.5, backward: bool = True,
                            fused_accumulation: bool = False):
    """One IL + A2C iteration of HAMT's agent (Seq2SeqCMTAgent.train with feedback 'sample', r2r/agent_cmt.py) on a batch of episodes:

    * teacher-forced rollout (skipped when ``ml_weight`` is 0): cross-entropy of every step's logits on the teacher action
      (hamt_stop_tokens), scaled by ml_weight / B, plus aux_weight x the alignment loss;
    * sampled rollout: 'visual' with return_states=True, one vi_policy_sample per step (actions stay on the device, the device seed
      keys the draw), then one extra 'visual' call for the bootstrap state; the critic runs ONCE over all T + 1 steps' states and the
      A2C node (vi_a2c_loss) takes the first T values, the last one detached (r2r/agent_cmt.py:661-744).

    ``model`` is hamt.VLNBertCMT, ``critic`` hamt.Critic, ``ep`` device tensors of synth.hamt_episode, ``rewards`` fp32 [n_steps, B]
    (the simulator's distance reward is agent code).  No host synchronisation: a GraphedIteration over a container of both modules
    (torch.nn.ModuleList([model, critic])) replays the whole iteration.  Returns (loss, parts, actions [n_steps, B]) with parts =
    dict(ce, aux, rl, policy, critic, entropy)."""
    B = ep['txt_ids'].shape[0]
    dev = ep['txt_ids'].device
    parts = {}
    loss = None
    if ml_weight != 0:
        tgt = hamt_stop_tokens(ep['ob_nav_types'])
        ces = []

        def teacher_step(txt, img2, hist, lens):
            logits = _hamt_visual(model, ep, txt, img2, hist, lens)[0]
            ces.append(torch.nn.functional.cross_entropy(logits, tgt, reduction='sum'))
        aux, _ = _hamt_rollout(model, ep, n_steps, teacher_step)
        ce = torch.stack(ces).sum()
        loss = ce * (ml_weight / B) + aux_weight * aux
        parts.update(ce=ce / B, aux=aux)

    from . import autograd_ops as ag
    stop = hamt_stop_tokens(ep['ob_nav_types'])
    ended = torch.zeros((B,), dtype=torch.uint8, device=dev)
    states, logps, ents, masks, actions = [], [], [], [], []

    def sample_step(txt, img2, hist, lens):
        logits, h = _hamt_visual(model, ep, txt, img2, hist, lens, return_states=True)
        a, lp, e, m = ag.policy_sample(logits, stop, ended)
        for lst, v in ((states, h), (logps, lp), (ents, e), (masks, m), (actions, a)):
            lst.append(v)
    _, last = _hamt_rollout(model, ep, n_steps, sample_step)
    states.append(_hamt_visual(model, ep, *last, return_states=True)[1])        # bootstrap state s_T
    values = critic(torch.cat(states, 0)).view(n_steps + 1, B)
    rl = ag.A2CLossFn.apply(values[:n_steps], torch.stack(logps), torch.stack(ents), torch.stack(masks), rewards.float(),
                            values[n_steps].detach(), ended, float(gamma), float(entropy_weight), normalize)
    parts.update(rl=rl[0], policy=rl[1], critic=rl[2], entropy=rl[3])
    loss = rl[0] if loss is None else loss + rl[0]
    if backward:
        with ag.fused_grad_accumulation(fused_accumulation):
            loss.backward()
    return loss, parts, torch.stack(actions)


class GraphedIteration:
    """A whole fine-tuning iteration replayed from CUDA graphs over static inputs: an iteration is ~4000 kernel launches
    whose host cost (ctypes, autograd bookkeeping) exceeds their device time at batch 64.  Two graphs bracket the one
    collective, which stays an ordinary (eager) NCCL call between them:

        graph 1: zero the flat gradient buffer, forward, backward          (grad_fn(static_inputs) -> loss)
        eager  : FlatGradients.all_reduce()                                 (between())
        graph 2: gradient clipping + optimiser step                         (update_fn())

        it = GraphedIteration(model, grad_fn, update_fn, static_inputs, between=flat.all_reduce)
        it.load(host_or_device_batch); loss = it.replay()

    Requirements: fixed shapes; viewpoint ids passed as interned tensors (duet.GlocalTextPathNavCMT.intern_vpids);
    gradients living in a FlatGradients buffer (static .grad storage); the optimiser created with ``capturable=True``.
    The derived weight copies (bf16 shadows, transposes) are rebuilt INSIDE graph 1 at the start of every iteration; call
    ``finish()`` before using the model outside the graphs again."""

    def __init__(self, model, grad_fn, update_fn, static_inputs: dict, between=None, warmup: int = 3, tail_fn=None,
                 before_tail=None):
        """``tail_fn``: the rest of the backward pass when ``grad_fn`` stops early (duet_finetune_iteration(split_language_backward=
        True): ``grad_fn`` keeps the ``finish`` closure, ``tail_fn`` calls it), captured into its own graph in the SAME memory pool;
        ``before_tail`` runs eagerly between the two (start the asynchronous all-reduce of the gradients that are already final),
        ``between`` after the tail as before (all-reduce the rest, wait for both)."""
        self.model, self.static, self.between = model, static_inputs, between
        self.before_tail = before_tail
        dev = next(model.parameters()).device

        def eager():
            loss = grad_fn(static_inputs)
            if tail_fn is not None:
                if before_tail is not None:
                    before_tail()
                tail_fn()
            if between is not None:
                between()
            update_fn()
            return loss
        for _ in range(warmup):                               # autotuning, allocator and lazy-initialisation warm-up
            eager()
        torch.cuda.synchronize(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self._invalidate_packs()                              # graph 1 must contain the weight re-cast
        self.g_grad = torch.cuda.CUDAGraph()
        with graphs.capture(self.g_grad):
            self.loss = grad_fn(static_inputs)
        self.g_tail = None
        if tail_fn is not None:
            if before_tail is not None:
                before_tail()
                torch.cuda.synchronize(dev)                # no collective in flight while the next capture runs
            self.g_tail = torch.cuda.CUDAGraph()
            with graphs.capture(self.g_tail, pool=self.g_grad.pool()):   # it reads tensors the first graph saved for backward
                tail_fn()
        if between is not None:
            between()
        from . import autograd_ops
        self._keepalive = list(autograd_ops._GradAcc.buffers.values())    # the graphs hold raw pointers to these accumulators
        self.g_update = torch.cuda.CUDAGraph()
        with graphs.capture(self.g_update):
            update_fn()

    def _invalidate_packs(self):
        for m in self.model.modules():
            if hasattr(m, '_packs'):
                m._packs = None

    def load(self, batch: dict):
        for k, v in self.static.items():
            if torch.is_tensor(v) and k in batch and batch[k] is not v:
                v.copy_(batch[k], non_blocking=True)

    def replay(self):
        self.g_grad.replay()
        if self.g_tail is not None:
            if self.before_tail is not None:
                self.before_tail()
            self.g_tail.replay()
        if self.between is not None:
            self.between()
        self.g_update.replay()
        # the optimiser ran inside a graph: no Python hook fired and fused optimisers do not bump tensor versions, so tell
        # every consumer of derived weights (blocks.Pack keys, graphs.weights_token) that the parameters have moved
        from . import blocks
        blocks.touch_weights()
        return self.loss

    def finish(self):
        """Call before using the model outside the replayed iteration (validation between training phases): drops the
        derived weight copies, the inference CUDA graphs that hold raw pointers to them and the cached context projections,
        so the next eager / graphed inference call rebuilds all of them from the CURRENT parameters."""
        from . import autograd_ops, blocks
        blocks.touch_weights()
        self._invalidate_packs()
        autograd_ops.release_accumulators()                   # they may live in this iteration's graph pool
        for m in self.model.modules():
            for name in ('_g_pano', '_g_nav', '_g_vis', '_g_hist'):
                g = getattr(m, name, None)
                if g is not None:
                    g.clear()
            if hasattr(m, '_wt_cache'):
                m._wt_cache = {}
            if hasattr(m, 'drop_context'):
                m.drop_context()
