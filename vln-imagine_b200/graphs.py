"""CUDA-graph replay behind the module API (inference calls only).

A per-step model call is ~40-80 kernel launches whose host-side cost (ctypes + tensor bookkeeping) is of the
same order as the device time at batch 64.  ``GraphedCall`` removes it for the calls the agents repeat every
navigation step: for each distinct input signature (shapes, dtypes, precision) the launch sequence is captured
once into a ``torch.cuda.CUDAGraph`` over static input buffers; later calls copy their inputs into those
buffers (host -> device directly when the caller passes pinned host tensors), replay, and return clones of the
outputs, so callers may keep the results across steps exactly as with the eager path.

Graphs hold raw pointers to the derived bf16 weight copies, so they are dropped whenever a parameter changes
(in-place update, ``load_state_dict``, ``.to()``): the owner passes a ``weights_token`` that changes with them.
Nothing here is used when autograd is recording.
"""
from __future__ import annotations

import collections
import contextlib
import gc
from typing import Callable, Dict

import torch


@contextlib.contextmanager
def capture(graph: 'torch.cuda.CUDAGraph', **kw):
    """``torch.cuda.graph`` with the cyclic garbage collector held off.  A GC pass in the middle of a capture may free dead
    modules that own CUDAGraphs (GraphedCall <-> module cycles are only reclaimed by the cyclic collector); destroying a graph
    or releasing its memory pool is "not permitted when stream is capturing" and invalidates the capture in progress.  PyTorch
    no longer collects before a capture (torch.compiler.config.force_cudagraph_gc), so it is done here."""
    gc.collect()
    enabled = gc.isenabled()
    gc.disable()
    try:
        with torch.cuda.graph(graph, **kw):
            yield
    finally:
        if enabled:
            gc.enable()


def round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def pad_to(x, sizes: Dict[int, int], device, fill=0):
    """x padded with ``fill`` (default zero / False) along the dimensions of ``sizes`` ({dim: new size}); host tensors are moved
    to ``device`` first"""
    if x is None or all(x.shape[d] == n for d, n in sizes.items()):
        return x
    x = x if x.is_cuda else x.to(device, non_blocking=True)
    shape = list(x.shape)
    for d, n in sizes.items():
        shape[d] = n
    out = x.new_full(shape, fill)
    out[tuple(slice(0, k) for k in x.shape)] = x
    return out


class ShapeBuckets:
    """Per-step shapes of a real rollout change almost every step (graph nodes G, local tokens P, history length T, observation
    count O), and a CUDA graph is tied to one signature: without care every new (G, P) costs an eager run, a warm-up and a capture,
    and an LRU of a few dozen graphs thrashes.  Once a mode has seen more than ``after`` distinct signatures its callers pad the
    varying dimensions up to multiples of ``step`` - padded positions are masked out exactly as the batch padding the reference
    itself applies, so results are unchanged - and a handful of graphs serves the whole rollout.  Fixed-shape callers (benchmarks)
    never trigger it.  VLN_IMAGINE_SHAPE_BUCKETS=1 forces it from the first call, =0 disables it."""

    def __init__(self, step: int = 8, after: int = 2):
        import os
        self.step, self.after = step, after
        self.mode = os.environ.get('VLN_IMAGINE_SHAPE_BUCKETS', 'auto')
        self.seen = set()

    def active(self, signature) -> bool:
        if self.mode == '0':
            return False
        if self.mode == '1':
            return True
        if len(self.seen) <= self.after:
            self.seen.add(signature)
        return len(self.seen) > self.after

    def up(self, n: int, step: int = None) -> int:
        return round_up(n, step or self.step)


class GraphedCall:
    def __init__(self, fn: Callable[[Dict[str, torch.Tensor]], Dict[str, torch.Tensor]], max_entries: int = 24,
                 capture_after: int = 1):
        """fn maps a dict of device tensors to a dict of device tensors and must be a pure launch sequence
        (no host synchronisation, no data-dependent host control flow)."""
        self.fn = fn
        self.max_entries = max_entries
        self.capture_after = capture_after
        self.entries = collections.OrderedDict()
        self.token = None
        self._copy_streams = {}

    def clear(self):
        self.entries.clear()

    def __call__(self, inputs: Dict[str, torch.Tensor], device: torch.device, extra_key=(), weights_token=None,
                 borrowed: Dict[str, torch.Tensor] = None, no_clone_prefix: str = None):
        """``borrowed``: device tensors the graph reads IN PLACE (no copy into static buffers): persistent buffers
        owned by the caller, e.g. the per-episode context projections.  Their addresses are part of the signature
        and the entry keeps them alive.  Outputs whose key starts with ``no_clone_prefix`` are handed out as the graph's
        own static buffers (valid until the next replay of the same signature): for intermediates the caller consumes at
        once on the same stream."""
        if weights_token != self.token:
            self.clear()
            self.token = weights_token
        borrowed = borrowed or {}
        key = (extra_key, tuple((k, tuple(v.shape), v.dtype) for k, v in inputs.items()),
               tuple((k, v.data_ptr(), tuple(v.shape), v.dtype) for k, v in borrowed.items()))
        ent = self.entries.get(key)
        if ent is None:
            ent = {'seen': 0, 'graph': None}
            self.entries[key] = ent
            while len(self.entries) > self.max_entries:
                self.entries.popitem(last=False)
        else:
            self.entries.move_to_end(key)
        if ent['graph'] is None:
            dev_in = {k: (v if v.device == device else v.to(device, non_blocking=True)) for k, v in inputs.items()}
            if ent['seen'] < self.capture_after:
                ent['seen'] += 1
                return self.fn({**dev_in, **borrowed})       # eager: also warms autotuning and weight packs
            static_in = {k: v.clone() for k, v in dev_in.items()}
            static_in.update(borrowed)
            ent['borrowed'] = dict(borrowed)
            torch.cuda.synchronize(device)
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                self.fn(static_in)                           # once more on the side stream (allocator warm-up)
            torch.cuda.current_stream(device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with capture(graph):
                static_out = self.fn(static_in)
            ent.update(graph=graph, static_in=static_in, static_out=static_out)
        static_in = ent['static_in']
        main = torch.cuda.current_stream(device)
        host_items = [(k, v) for k, v in inputs.items() if not v.is_cuda]
        if host_items:
            # Host inputs go through a copy stream: they depend only on this graph's PREVIOUS replay having consumed the
            # static buffers, so the navigation call's uploads overlap the panorama graph still running on the main stream.
            cs = self._copy_stream(device)
            if ent.get('done') is not None:
                cs.wait_event(ent['done'])
            else:
                cs.wait_stream(main)
            with torch.cuda.stream(cs):
                for k, v in host_items:
                    static_in[k].copy_(v, non_blocking=True)
            ev = ent.get('uploaded')
            if ev is None:
                ev = ent['uploaded'] = torch.cuda.Event()
            ev.record(cs)
            main.wait_event(ev)
        for k, v in inputs.items():
            if v.is_cuda:
                static_in[k].copy_(v, non_blocking=True)
        ent['graph'].replay()
        # recorded on EVERY replay (also device-only calls): the next host upload into the static buffers waits for it
        if ent.get('done') is None:
            ent['done'] = torch.cuda.Event()
        ent['done'].record(main)
        return {k: (v.clone() if torch.is_tensor(v) and not (no_clone_prefix and k.startswith(no_clone_prefix)) else v)
                for k, v in ent['static_out'].items()}

    def _copy_stream(self, device):
        cs = self._copy_streams.get(device)
        if cs is None:
            cs = self._copy_streams[device] = torch.cuda.Stream(device)
        return cs


def weights_token(module: torch.nn.Module, cache: dict):
    """Cheap fingerprint of a module's parameters: changes on any in-place update or re-allocation."""
    params = cache.get('params')
    if params is None:
        params = cache['params'] = list(module.parameters())
    from .blocks import weights_epoch
    v = 0
    for p in params:
        v += p._version
    return (v, weights_epoch(), params[0].data_ptr() if params else 0, len(params))
