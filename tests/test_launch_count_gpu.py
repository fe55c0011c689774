"""The library's launch counter (vi_launch_count: what bench.py reports as gpu_launches) against the kernels torch.profiler records
for the same calls, on entry points whose kernel count depends on the problem: one launch per problem of fp32 attention, the
reduction pass of a split vi_wgrad16, the cluster launch of a CTA-pair GEMM, the multi-pass reductions of the backward kernels,
the optional second pass of the contrastive-loss adjoint, and a loss over no rows."""
import importlib

import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops(lib_built):
    o = importlib.import_module('vln_imagine_b200.ops')
    o.ensure_init(torch.zeros(1, device='cuda'))
    return o


def _rand(*shape, seed=0, dtype=torch.float32):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return torch.randn(*shape, generator=g).to('cuda', dtype)


def _cases(ops):
    dev, bf16 = torch.device('cuda'), torch.bfloat16
    cases = {}
    qkv, kv = _rand(2 * 16, 3 * 768, seed=1), _rand(2 * 40, 2 * 768, seed=2)
    o1, o2 = torch.empty(32, 768, device=dev), torch.empty(32, 768, device=dev)
    cases['fp32 attention, two problems'] = lambda: ops.attention_multi([
        dict(q=qkv[:, :768], k=qkv[:, 768:1536], v=qkv[:, 1536:], out=o1, B=2, Lq=16, Lk=16),
        dict(q=qkv[:, :768], k=kv[:, :768], v=kv[:, 768:], out=o2, B=2, Lq=16, Lk=40)])
    for name, (M, N, K, ends, split) in {'wgrad16, split': (4416, 768, 768, [2048, 4416], True),
                                        'wgrad16, one pass': (4416, 3072, 768, [2048, 4416], False)}.items():
        bounds = ends or [M]
        rows = [b - (bounds[i - 1] if i else 0) for i, b in enumerate(bounds)]
        assert (ops.lib.vi_wgrad16_splits(N, K, len(bounds), ops._lib.int_array(rows)) > 1) == split, name
        dy, x = _rand(M, N, seed=3, dtype=bf16), _rand(M, K, seed=4, dtype=bf16)
        cases[name] = lambda dy=dy, x=x, ends=ends: ops.wgrad16(dy, x, ends, True)
    xg, wg = _rand(512, 768, seed=5, dtype=bf16), _rand(768, 768, seed=6, dtype=bf16)
    cases['CTA-pair GEMM'] = lambda: ops.gemm(xg, wg, tile=256 | ops.TILE_PAIR)
    a, gamma, dy = _rand(300, 768, seed=7), _rand(768, seed=8), _rand(300, 768, seed=9)
    dg, db = torch.empty(1, 768, device=dev), torch.empty(1, 768, device=dev)
    cases['LayerNorm backward'] = lambda: ops.add_ln_drop_bwd(a, None, gamma, 1e-12, dy, None, dg, db, 0)
    x, w, dout = _rand(500, 768, seed=10), _rand(768, seed=11), _rand(500, seed=12)
    cases['rowdot backward'] = lambda: ops.rowdot_bwd(dout, x, w)
    R, Nn = 41, 57
    p, t, negs = _rand(R, 768, seed=13), _rand(R, 768, seed=14), _rand(Nn, 768, seed=15)
    row_ep = (torch.arange(R, device=dev) * 8 // R).int()
    neg_ep = (torch.arange(Nn, device=dev) * 8 // Nn).int()
    _, scratch = ops.infonce_loss(p, t, negs, row_ep, neg_ep, 0.1, R, Nn, dev)
    dloss = torch.ones(1, device=dev)
    for want in (False, True):
        cases['InfoNCE backward, dnegs %s' % want] = lambda want=want: ops.contrastive_loss_bwd(
            'infonce', p, t, negs, row_ep, neg_ep, 0.1, scratch, dloss, R, Nn, want, want)
    cases['cosine loss over no rows'] = lambda: ops.cosine_loss(None, None, 0, dev)
    return cases


def test_launch_count_matches_the_kernels_the_profiler_records(ops):
    for name, call in _cases(ops).items():
        call()                                       # workspaces and kernel attributes are set up outside the profiled call
        torch.cuda.synchronize()
        n0, c0 = ops.lib.vi_launch_count(), ops._Counters.launches
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        counted = ops.lib.vi_launch_count() - n0
        kernels = [e.name for e in prof.events()
                   if e.device_type == DeviceType.CUDA and not e.name.startswith(('Memcpy', 'Memset'))]
        assert counted == len(kernels) > 0, (name, counted, kernels)
        assert ops._Counters.launches - c0 == counted, name
