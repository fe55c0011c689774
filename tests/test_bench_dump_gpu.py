"""bench.py --dump-outputs on the GPU: the flagship workload writes every tensor its timed step hands back, and what the
CUDA-graph replay leaves there - last step the first of an episode (context projections inside the graph) or a later one -
is what eager launches of the same step compute."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

import bench  # the repository root is on sys.path (conftest.py)

pytestmark = pytest.mark.gpu

DUET_OUTPUTS = {'pano_embeds', 'pano_masks', 'gmap_embeds', 'vp_embeds', 'global_logits', 'local_logits', 'fused_logits'}


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '3', '--no-cpu-baseline',
           '--dump-outputs', str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, VI_BENCH_TRAIN='0'))
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert line['steps'] == steps
    for f in os.listdir(out_dir):
        stored = np.load(os.path.join(out_dir, f))
        assert stored.dtype == np.float32 and np.isfinite(stored).all(), f
    return bench.load_dump(out_dir)


def _eager_step():
    kind, shape, _ = bench.workload('duet_cfg2')
    model, ep = bench.build(kind, shape, 0, 'bf16')
    model.use_cuda_graphs = False
    with torch.no_grad():
        d = bench.device_inputs(kind, model, ep, torch.device('cuda'))
        txt, img2, _ = bench.episode_prelude(kind, model, d)
        out = bench.duet_step(model, d, txt, img2)
    return {k: v.float().cpu().numpy() for k, v in out.items()}


def test_bench_dumps_what_its_timed_step_computed(lib_built, tmp_path):
    first, later = _bench(tmp_path / 'first', 7), _bench(tmp_path / 'later', 8)      # episodes of 6 steps: step 7 starts one
    want = _eager_step()
    assert set(first) == set(later) == set(want) == DUET_OUTPUTS
    assert sum(os.path.getsize(tmp_path / 'first' / f) for f in os.listdir(tmp_path / 'first')) <= 64 << 20
    for name, b in want.items():
        assert np.isfinite(b).any(), name
        fin = np.isfinite(b)
        for a in (first[name], later[name]):
            assert a.dtype == np.float32 and a.shape == b.shape, name
            assert (np.isfinite(a) == fin).all(), name
            assert np.abs(a[fin] - b[fin]).max() <= 1e-3 * max(np.abs(b[fin]).max(), 1e-30), name
