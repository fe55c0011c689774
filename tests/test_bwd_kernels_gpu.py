"""Backward-pass kernels (fine-tuning path, BASELINE.json cfg-4) against torch.autograd of the same op in fp32.

Every check goes through the autograd wrappers of vln-imagine_b200/autograd_ops.py, i.e. through the C ABI.
Tolerances: fp32 kernels 1e-4 (max-norm relative); bf16 operand kernels 2e-2 against the fp32 reference.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ag(lib_built):
    import importlib
    o = importlib.import_module('vln_imagine_b200.ops')
    o.ensure_init(torch.zeros(1, device='cuda'))
    return importlib.import_module('vln_imagine_b200.autograd_ops')


@pytest.fixture(scope='module')
def ops(ag):
    import importlib
    return importlib.import_module('vln_imagine_b200.ops')


@pytest.fixture(scope='module')
def blocks(ag):
    import importlib
    return importlib.import_module('vln_imagine_b200.blocks')


def relerr(a, b):
    a, b = a.float(), b.float()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-20))


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


class _Lin:
    """nn.Linear-like parameter holder"""

    def __init__(self, n, k, seed, bias=True):
        self.weight = _rand(n, k, scale=0.05, seed=seed).requires_grad_()
        self.bias = _rand(n, scale=0.1, seed=seed + 1).requires_grad_() if bias else None


class _LN:
    def __init__(self, seed):
        self.weight = (1 + _rand(768, scale=0.1, seed=seed)).requires_grad_()
        self.bias = _rand(768, scale=0.1, seed=seed + 1).requires_grad_()


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('rows,cols,pad', [(37, 768, 64), (300, 2304, 320), (64, 64, 64), (1000, 14, 1000)])
def test_transpose_and_colsum(ops, dtype, rows, cols, pad):
    x = _rand(rows, cols, seed=1).to(dtype)
    t = ops.transpose(x, pad)
    assert t.shape == (cols, pad)
    assert torch.equal(t[:, :rows], x.t())
    assert float(t[:, rows:].float().abs().sum()) == 0.0
    view = _rand(rows, cols + 24, seed=2).to(dtype)[:, 8:8 + cols]         # strided source
    assert torch.equal(ops.transpose(view, pad)[:, :rows], view.t())
    cs = ops.colsum(x)
    assert relerr(cs, x.float().sum(0)) < 1e-5


@pytest.mark.parametrize('act', [1, 2])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_activation_fwd_bwd(ag, act, dtype):
    x = _rand(333, 3072, seed=3).to(dtype).requires_grad_()
    dy = _rand(333, 3072, seed=4).to(dtype)
    y = ag.ActFn.apply(x, act)
    y.backward(dy)
    xr = x.detach().float().requires_grad_()
    yr = F.gelu(xr) if act == 1 else F.relu(xr)
    yr.backward(dy.float())
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert relerr(y, yr) < tol
    assert relerr(x.grad, xr.grad) < tol


@pytest.mark.parametrize('lowp', [False, True])
@pytest.mark.parametrize('grouped', [False, True])
@pytest.mark.parametrize('residual', [False, True])
def test_layer_norm_bwd(ag, blocks, lowp, grouped, residual):
    rows = 1024 + 777 if grouped else 1000
    ends = [1024, rows] if grouped else None
    lns = [_LN(10), _LN(20)] if grouped else [_LN(10)]
    pack = blocks.LNPack(lns)
    a = _rand(rows, 768, seed=5).requires_grad_()
    b = _rand(rows, 768, seed=6).requires_grad_() if residual else None
    d32 = _rand(rows, 768, seed=7)
    d16 = _rand(rows, 768, seed=8).bfloat16() if lowp else None
    y32, y16 = ag.layer_norm(a, b, pack, 1e-12, lowp, ends)
    if lowp:
        torch.autograd.backward([y32, y16], [d32, d16])
    else:
        y32.backward(d32)
    # torch reference
    ar = a.detach().clone().requires_grad_()
    br = b.detach().clone().requires_grad_() if residual else None
    pr = [(l.weight.detach().clone().requires_grad_(), l.bias.detach().clone().requires_grad_()) for l in lns]
    xs = ar + br if residual else ar
    bounds = [0] + (ends or [rows])
    yr = torch.cat([F.layer_norm(xs[bounds[i]:bounds[i + 1]], (768,), pr[i][0], pr[i][1], 1e-12) for i in range(len(lns))], 0)
    dy = d32 + (d16.float() if lowp else 0)
    yr.backward(dy)
    assert relerr(y32, yr) < 1e-5
    assert relerr(a.grad, ar.grad) < 1e-4
    if residual:
        assert relerr(b.grad, br.grad) < 1e-4
    for l, (gw, gb) in zip(lns, pr):
        assert relerr(l.weight.grad, gw.grad) < 1e-4
        assert relerr(l.bias.grad, gb.grad) < 1e-4


@pytest.mark.parametrize('lowp', [False, True])
@pytest.mark.parametrize('case', ['plain', 'residual', 'grouped', 'nobias', 'smallM'])
def test_linear_bwd(ag, blocks, lowp, case):
    """dX = dY W (dgrad), dW = dY^T X (wgrad on transposed operands), db = colsum(dY); grouped rows -> per-group
    weight gradients"""
    K, N = 768, 1536 if case != 'grouped' else 768
    M = {'plain': 1000, 'residual': 1920, 'grouped': 2048 + 333, 'nobias': 512, 'smallM': 5}[case]
    ends = [2048, M] if case == 'grouped' else None
    lins = [_Lin(N, K, 30, bias=case != 'nobias')] + ([_Lin(N, K, 40)] if case == 'grouped' else [])
    pack = blocks.LinearPack([l.weight for l in lins], [l.bias for l in lins])
    x32 = _rand(M, K, seed=9)
    x = (x32.bfloat16() if lowp else x32).requires_grad_()
    res = _rand(M, N, seed=10).requires_grad_() if case == 'residual' else None
    dy = _rand(M, N, seed=11)
    y = ag.linear(x, pack, lowp, residual=res, out_dtype=torch.float32, ends=ends)
    y.backward(dy)
    xr = x.detach().float().requires_grad_()
    rr = res.detach().clone().requires_grad_() if res is not None else None
    pr = [(l.weight.detach().clone().requires_grad_(), l.bias.detach().clone().requires_grad_() if l.bias is not None else None)
          for l in lins]
    if lowp:       # the kernel rounds W (and dY for the gradient GEMMs) to bf16: the reference uses the rounded weight
        wq = [w.detach().bfloat16().float().requires_grad_() for w, _ in pr]
    else:
        wq = [w for w, _ in pr]
    bounds = [0] + (ends or [M])
    yr = torch.cat([F.linear(xr[bounds[i]:bounds[i + 1]], wq[i], pr[i][1]) for i in range(len(lins))], 0)
    if rr is not None:
        yr = yr + rr
    yr.backward(dy)
    tol = 2e-2 if lowp else 1e-4
    assert relerr(y, yr) < (2e-3 if lowp else 1e-4)
    assert relerr(x.grad, xr.grad) < tol
    if rr is not None:
        assert relerr(res.grad, rr.grad) < 1e-6
    for l, w, (_, b) in zip(lins, wq, pr):
        assert relerr(l.weight.grad, w.grad) < tol
        if b is not None:
            assert relerr(l.bias.grad, b.grad) < tol


def _torch_attention(q, k, v, B, Lq, Lk, key_mask, dist, aw, ab, neg_inf):
    qh = q.view(B, Lq, 12, 64).transpose(1, 2)
    kh = k.view(B, Lk, 12, 64).transpose(1, 2)
    vh = v.view(B, Lk, 12, 64).transpose(1, 2)
    s = qh @ kh.transpose(-1, -2) / 8.0
    if key_mask is not None:
        if neg_inf:
            s = s.masked_fill(~key_mask[:, None, None, :], float('-inf'))
        else:
            s = s + (~key_mask)[:, None, None, :].float() * -10000.0
    if dist is not None:
        s = s + (dist * aw + ab)[:, None]
    p = torch.softmax(s, -1)
    return (p @ vh).transpose(1, 2).reshape(B * Lq, 768)


@pytest.mark.parametrize('lowp', [False, True])
@pytest.mark.parametrize('case', ['self_gasa', 'cross', 'pano_neg_inf'])
def test_attention_bwd(ag, case, lowp):
    from vln_imagine_b200.ops import MASK_ADD_NEG10000, MASK_NEG_INF
    B = 5
    dt = torch.bfloat16 if lowp else torch.float32
    if case == 'cross':
        Lq, Lk = 30, 85
    elif case == 'self_gasa':
        Lq = Lk = 30
    else:
        Lq = Lk = 36
    lens = torch.tensor([Lk, Lk // 2, 3, Lk - 1, 7])
    key_mask = (torch.arange(Lk)[None, :] < lens[:, None]).cuda()
    gasa = case == 'self_gasa'
    dist = (_rand(B, Lq, Lk, seed=12).abs() * 5) if gasa else None
    aw = torch.tensor([[-0.5]], device='cuda', requires_grad=True)
    ab = torch.tensor([0.1], device='cuda', requires_grad=True)
    affine = torch.stack([aw.detach().view(()), ab.detach().view(())]).contiguous()
    mode = MASK_NEG_INF if case == 'pano_neg_inf' else MASK_ADD_NEG10000
    dout = _rand(B * Lq, 768, seed=13).to(dt)
    km = key_mask.view(torch.uint8)
    if case == 'cross':
        q = _rand(B * Lq, 768, seed=14).to(dt).requires_grad_()
        kv = _rand(B * Lk, 1536, seed=15).to(dt).requires_grad_()
        spec = [dict(q=(0, 0, 0), k=(1, 0, 0), v=(1, 0, 768), B=B, Lq=Lq, Lk=Lk, key_mask=km, out_row0=0)]
        out = ag.AttentionFn.apply(spec, B * Lq, mode, 2, q, kv)
        out.backward(dout)
        qr, kvr = q.detach().float().requires_grad_(), kv.detach().float().requires_grad_()
        ref = _torch_attention(qr, kvr[:, :768], kvr[:, 768:], B, Lq, Lk, key_mask, None, None, None, False)
        ref.backward(dout.float())
        got, want = [q.grad, kv.grad], [qr.grad, kvr.grad]
    else:
        qkv = _rand(B * Lq, 2304, seed=16).to(dt).requires_grad_()
        spec = [dict(q=(0, 0, 0), k=(0, 0, 768), v=(0, 0, 1536), B=B, Lq=Lq, Lk=Lk, key_mask=km, pair_dist=dist,
                     bias_affine=affine if gasa else None, out_row0=0)]
        extras = (aw, ab) if gasa else ()
        out = ag.AttentionFn.apply(spec, B * Lq, mode, 1, qkv, *extras)
        out.backward(dout)
        r = qkv.detach().float().requires_grad_()
        awr, abr = aw.detach().clone().requires_grad_(), ab.detach().clone().requires_grad_()
        ref = _torch_attention(r[:, :768], r[:, 768:1536], r[:, 1536:], B, Lq, Lk, key_mask, dist,
                               awr.view(()) if gasa else None, abr.view(()) if gasa else None, case == 'pano_neg_inf')
        ref.backward(dout.float())
        got, want = [qkv.grad], [r.grad]
        if gasa:
            got += [aw.grad, ab.grad]
            want += [awr.grad, abr.grad]
    tol = 2e-2 if lowp else 2e-4
    assert relerr(out, ref) < (1e-2 if lowp else 1e-4)
    for g, w in zip(got, want):
        assert g.shape == w.shape
        if float(w.abs().max()) < 1e-6 * float(want[0].abs().max()):
            # the GASA offset shifts every score of a row equally: its gradient is analytically zero
            assert float(g.abs().max()) < 1e-3 * float(want[0].abs().max())
        else:
            assert relerr(g, w) < tol


def test_embedding_pieces_bwd(ag):
    """small-feature linear, row gather (table / position) and the row sum with broadcast constants"""
    rows = 700
    feat = _rand(rows, 7, seed=17)
    lin = _Lin(768, 7, 50)
    t = ag.SmallLinearFn.apply(feat, lin.weight, lin.bias)
    table = _rand(100, 768, seed=18).requires_grad_()
    idx = torch.randint(0, 100, (rows,), generator=torch.Generator().manual_seed(1)).cuda()
    pos = _rand(512, 768, seed=19).requires_grad_()
    g1 = ag.GatherRowsFn.apply(table, idx, 0, rows)
    g2 = ag.GatherRowsFn.apply(pos, None, 35, rows)
    c = _rand(768, seed=20).requires_grad_()
    s = ag.SumRowsFn.apply(3, t, g1, g2, c)
    dy = _rand(rows, 768, seed=21)
    s.backward(dy)
    w, b, tb, ps, cr = [x.detach().clone().requires_grad_() for x in (lin.weight, lin.bias, table, pos, c)]
    ref = F.linear(feat, w, b) + tb[idx] + ps[torch.arange(rows, device='cuda') % 35] + cr
    ref.backward(dy)
    assert relerr(s, ref) < 1e-5
    for got, want in [(lin.weight.grad, w.grad), (lin.bias.grad, b.grad), (table.grad, tb.grad), (pos.grad, ps.grad),
                      (c.grad, cr.grad)]:
        assert relerr(got, want) < 1e-4


@pytest.mark.parametrize('grouped', [False, True])
def test_rowdot_bwd(ag, grouped):
    rows = 1024 + 300 if grouped else 500
    ends = [1024, rows] if grouped else None
    n = 2 if grouped else 1
    ws = [_rand(1, 768, scale=0.1, seed=60 + i).requires_grad_() for i in range(n)]
    bs = [_rand(1, scale=0.1, seed=70 + i).requires_grad_() for i in range(n)]
    x = _rand(rows, 768, seed=22).requires_grad_()
    wst = torch.stack([w.detach().view(-1) for w in ws]).contiguous() if grouped else ws[0].detach().view(-1).contiguous()
    bst = torch.cat([b.detach() for b in bs]).contiguous()
    out = ag.RowDotFn.apply(x, wst, bst, ends, n, *ws, *bs)
    dout = _rand(rows, seed=23)
    out.backward(dout)
    xr = x.detach().clone().requires_grad_()
    wr = [w.detach().clone().requires_grad_() for w in ws]
    br = [b.detach().clone().requires_grad_() for b in bs]
    bounds = [0] + (ends or [rows])
    ref = torch.cat([F.linear(xr[bounds[i]:bounds[i + 1]], wr[i], br[i]).view(-1) for i in range(n)])
    ref.backward(dout)
    assert relerr(out, ref) < 1e-5
    assert relerr(x.grad, xr.grad) < 1e-5
    for i in range(n):
        assert relerr(ws[i].grad, wr[i].grad) < 1e-4
        assert relerr(bs[i].grad, br[i].grad) < 1e-4


def test_cosine_loss_bwd(ag):
    R = 237
    p = _rand(R, 768, seed=24).requires_grad_()
    t = _rand(R, 768, seed=25).requires_grad_()
    loss = ag.CosineLossFn.apply(p, t, R)
    (loss * 0.5).backward()
    pr, tr = p.detach().clone().requires_grad_(), t.detach().clone().requires_grad_()
    ref = (1 - F.cosine_similarity(pr, tr, dim=-1)).mean()
    (ref * 0.5).backward()
    assert abs(float(loss) - float(ref)) < 1e-5
    assert relerr(p.grad, pr.grad) < 1e-4
    assert relerr(t.grad, tr.grad) < 1e-4


@pytest.mark.parametrize('T', [0.07, 0.3])
def test_infonce_loss_bwd(ag, T):
    """InfoNCE alignment loss (models/vilmodel.py:657-687): negatives = noun-phrase means of OTHER episodes; the gradient
    w.r.t. the projected imagination rows against torch autograd of F.cosine_similarity + F.cross_entropy"""
    R, Nn = 41, 57
    p = _rand(R, 768, seed=31).requires_grad_()
    t, negs = _rand(R, 768, seed=32), _rand(Nn, 768, seed=33)
    g = torch.Generator().manual_seed(5)
    row_ep = torch.sort(torch.randint(0, 8, (R,), generator=g)).values.int().cuda()
    neg_ep = torch.sort(torch.randint(0, 8, (Nn,), generator=g)).values.int().cuda()
    loss = ag.InfoNCELossFn.apply(p, t, negs, row_ep, neg_ep, T, R, Nn)
    (loss * 0.7).backward()
    pr = p.detach().clone().requires_grad_()
    ref = []
    for r in range(R):
        allt = torch.cat([t[r:r + 1], negs[neg_ep != row_ep[r]]], 0)
        sim = F.cosine_similarity(pr[r:r + 1], allt) / T
        ref.append(F.cross_entropy(sim[None], torch.zeros(1, dtype=torch.long, device='cuda')))
    ref = torch.stack(ref).mean()
    (ref * 0.7).backward()
    assert abs(float(loss) - float(ref)) < 1e-4 * max(1.0, abs(float(ref)))
    assert relerr(p.grad, pr.grad) < 1e-4
    # no negatives at all: the loss is log(1) = 0 and so is the gradient
    p2 = _rand(3, 768, seed=34).requires_grad_()
    l2 = ag.InfoNCELossFn.apply(p2, _rand(3, 768, seed=35), None, torch.zeros(3, dtype=torch.int32, device='cuda'), None, T, 3, 0)
    l2.backward()
    assert abs(float(l2)) < 1e-6 and float(p2.grad.abs().max()) < 1e-6


@pytest.mark.parametrize('dtype', [torch.bfloat16, torch.float16])
@pytest.mark.parametrize('M,N,K,ends', [
    (300, 128, 64, None),                 # one unit, rows not a multiple of 64 (TMA zero fill), 64-wide tile
    (4416, 768, 768, [2048, 4416]),       # cfg-2 grouped projection: 36 tiles x 4 splits
    (2304, 2304, 768, None),              # panorama QKV
    (4416, 768, 3072, [2048, 4416]),      # FFN2 weight gradient (256-wide tiles, no split)
    (2304, 3072, 768, None),              # FFN1
    (520, 512, 768, None),                # projection head
    (1000, 256, 192, [256, 1000]),        # 64-wide tiles, uneven groups
])
def test_wgrad16_vs_torch(ops, M, N, K, ends, dtype):
    """vi_wgrad16 (MN-major tcgen05 operands, split rows, ones-tile bias gradient) against dY^T X / dY.sum(0) in fp32 of the
    same 16-bit values; two calls are bit-identical (fixed-order reduction of the split partials)"""
    dy = (_rand(M, N, seed=51) * 0.5).to(dtype)
    x = _rand(M, K, seed=52).to(dtype)
    assert ops.wgrad16_ok(dy, x)
    dW, db = ops.wgrad16(dy, x, ends, True)
    dW2, db2 = ops.wgrad16(dy, x, ends, True)
    torch.cuda.synchronize()
    assert torch.equal(dW, dW2) and torch.equal(db, db2)
    bounds = [0] + (ends or [M])
    for g in range(len(bounds) - 1):
        r0, r1 = bounds[g], bounds[g + 1]
        ref_w = dy[r0:r1].float().t() @ x[r0:r1].float()
        ref_b = dy[r0:r1].float().sum(0)
        assert relerr(dW[g * N:(g + 1) * N], ref_w) < 2e-3, (g, relerr(dW[g * N:(g + 1) * N], ref_w))
        assert relerr(db[g * N:(g + 1) * N], ref_b) < 2e-3, (g, relerr(db[g * N:(g + 1) * N], ref_b))
    dW3, db3 = ops.wgrad16(dy, x, ends, False)
    assert db3 is None and torch.equal(dW3, dW)


@pytest.mark.parametrize('margin', [0.1, 0.5])
def test_margin_loss_bwd(ag, margin):
    """margin form of the alignment loss (H/models/vilmodel_cmt.py:825-856): (1 - cos_pos) + mean relu(margin + cos_neg - cos_pos)
    over the noun-phrase means of OTHER episodes; gradient w.r.t. the projected rows against torch autograd"""
    R, Nn = 37, 45
    p = _rand(R, 768, seed=41).requires_grad_()
    t, negs = _rand(R, 768, seed=42), _rand(Nn, 768, seed=43)
    with torch.no_grad():                                # some negatives close to the row, so both hinge states occur
        negs[::3] = p.detach()[: negs[::3].shape[0]] + 0.3 * negs[::3]
    g = torch.Generator().manual_seed(6)
    row_ep = torch.sort(torch.randint(0, 8, (R,), generator=g)).values.int().cuda()
    neg_ep = torch.sort(torch.randint(0, 8, (Nn,), generator=g)).values.int().cuda()
    loss = ag.MarginLossFn.apply(p, t, negs, row_ep, neg_ep, margin, R, Nn)
    (loss * 0.7).backward()
    pr = p.detach().clone().requires_grad_()
    ref, active = [], 0
    for r in range(R):
        ng = negs[neg_ep != row_ep[r]]
        pos = F.cosine_similarity(pr[r:r + 1], t[r:r + 1]).squeeze()
        hinge = F.relu(margin + F.cosine_similarity(pr[r:r + 1], ng) - pos)
        active += int((hinge > 0).sum())
        ref.append((1 - pos) + hinge.mean())
    ref = torch.stack(ref).mean()
    (ref * 0.7).backward()
    assert 0 < active < R * Nn
    assert abs(float(loss) - float(ref)) < 1e-4 * max(1.0, abs(float(ref)))
    assert relerr(p.grad, pr.grad) < 1e-4


def test_slot_gather_scatter_bwd(ag):
    n, R = 40, 9
    src = _rand(n, 768, seed=26).requires_grad_()
    slot = torch.tensor([3, 5, 8, 13, 21, 22, 30, 31, 39], dtype=torch.int32, device='cuda')
    unit = torch.arange(R + 1, dtype=torch.int32, device='cuda')
    rows = ag.GatherSlotsFn.apply(src, unit, slot, R, False)
    proj = rows * 1.0                                    # stands for the projection head
    proj.retain_grad()
    out = ag.ScatterSlotsFn.apply(src, proj, slot, unit)
    w = _rand(n, 768, seed=27)
    (out * w).sum().backward()
    sr = src.detach().clone().requires_grad_()
    rr = sr[slot.long()] * 1.0
    outr = sr.clone()
    outr[slot.long()] = rr
    (outr * w).sum().backward()
    assert torch.equal(out.detach(), outr.detach())
    assert relerr(src.grad, sr.grad) < 1e-6


def test_fuse_logits_bwd(ag):
    """adjoint of the global/local fusion against autograd through the oracle's restatement
    (VLN-DUET/map_nav_src/models/vilmodel.py:1182-1217)"""
    import numpy as np
    from oracle import duet_oracle as O
    from vln_imagine_b200 import synth
    from vln_imagine_b200.duet import _IdTable
    ep = synth.to_torch(synth.duet_episode(synth.CFG1, 99), 'cuda')
    B, G = ep['gmap_masks'].shape
    P = ep['vp_nav_masks'].shape[1]
    g_raw = _rand(B * G, seed=28).requires_grad_()
    l_raw = _rand(B * P, seed=29).requires_grad_()
    f_raw = _rand(B, seed=30).requires_grad_()
    ids = _IdTable()
    gids = torch.from_numpy(ids.encode(ep['gmap_vpids'], G, -1)).cuda()
    cids = torch.from_numpy(ids.encode(ep['vp_cand_vpids'], P, -2)).cuda()
    u8 = lambda m: m.contiguous().view(torch.uint8)      # noqa: E731
    gl, ll, fl = ag.FuseLogitsFn.apply(g_raw, l_raw, f_raw, u8(ep['gmap_masks']), u8(ep['gmap_visited_masks']),
                                       u8(ep['vp_nav_masks']), gids, cids, B, G, P)
    wg, wl, wf = _rand(B, G, seed=31), _rand(B, P, seed=32), _rand(B, G, seed=33)

    def scalar(a, b, c):
        z = lambda t, w: (torch.where(torch.isfinite(t), t, torch.zeros_like(t)) * w).sum()      # noqa: E731
        return z(a, wg) + z(b, wl) + z(c, wf)
    scalar(gl, ll, fl).backward()
    gr, lr, fr = [t.detach().clone().requires_grad_() for t in (g_raw, l_raw, f_raw)]
    fw = torch.sigmoid(fr)[:, None]
    glr = (gr.view(B, G) * fw).masked_fill(ep['gmap_visited_masks'], float('-inf')).masked_fill(~ep['gmap_masks'], float('-inf'))
    llr = (lr.view(B, P) * (1 - fw)).masked_fill(~ep['vp_nav_masks'], float('-inf'))
    flr = O.fuse_logits(glr, llr, ep['gmap_vpids'], ep['gmap_visited_masks'], ep['vp_cand_vpids'])
    scalar(glr, llr, flr).backward()
    for got, want in [(gl, glr), (ll, llr), (fl, flr)]:
        assert torch.equal(torch.isfinite(got), torch.isfinite(want))
        fin = torch.isfinite(want)
        assert relerr(got[fin], want[fin]) < 1e-5
    assert relerr(g_raw.grad, gr.grad) < 1e-4
    assert relerr(l_raw.grad, lr.grad) < 1e-4
    assert relerr(f_raw.grad, fr.grad) < 1e-4


M32 = 0xFFFFFFFF


def _hash32(idx, key):
    """vi_hash32 of vi_common.cuh on int64 tensors"""
    h = (idx * 0x9E3779B1 + key) & M32
    h = h ^ (h >> 16)
    h = (h * 0x7FEB352D) & M32
    h = h ^ (h >> 15)
    h = (h * 0x846CA68B) & M32
    return h ^ (h >> 16)


def _keep_mask(idx, seed, site, p):
    key = _hash32(torch.tensor(site, dtype=torch.int64), (int(seed) ^ 0xA511E9B3) & M32)
    return _hash32(idx, int(key)) >= int(p * 4294967296.0)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_dropout_mask_and_backward(ag, dtype):
    p = 0.3
    x = (_rand(1000, 768, seed=50) + 3.0).to(dtype).requires_grad_()
    ag._DropState.site = 100
    y = ag.dropout(x, p)
    site = ag._DropState.site
    seed = int(ag.dropout_seed(x.device).item()) & M32
    keep = _keep_mask(torch.arange(x.numel(), device='cuda', dtype=torch.int64), seed, site, p).view_as(x)
    ref = torch.where(keep, x.detach().float() / (1 - p), torch.zeros_like(x, dtype=torch.float32))
    assert relerr(y.detach(), ref) < (1e-6 if dtype == torch.float32 else 1e-2)
    assert abs(float(keep.float().mean()) - (1 - p)) < 5e-3
    dy = _rand(1000, 768, seed=51).to(dtype)
    y.backward(dy)
    assert relerr(x.grad, torch.where(keep, dy.float() / (1 - p), torch.zeros_like(ref))) < (1e-6 if dtype == torch.float32 else 1e-2)
    y2 = ag.dropout(x.detach(), p)                      # next site: an independent mask
    assert 0.3 < float(((y2 != 0) == (y.detach() != 0)).float().mean()) < 0.75
    ag.advance_dropout_seeds()                          # what the optimizer-step hook does
    y3 = ag.dropout_raw(x.detach(), p, site)
    assert 0.3 < float(((y3 != 0) == (y.detach() != 0)).float().mean()) < 0.75


@pytest.mark.parametrize('p', [0.0, 0.2])
@pytest.mark.parametrize('grouped', [False, True])
@pytest.mark.parametrize('fused_acc', [False, True])
def test_dense_residual_layernorm_node(ag, blocks, p, grouped, fused_acc):
    """DenseResLNFn: LN(dropout(x W^T + b) + res) as one autograd node with the dropout mask applied inside the LayerNorm kernels
    (vi_add_ln_drop / vi_add_ln_drop_bwd emit dropout(dx) as the 16-bit operand of the gradient GEMMs) against torch autograd with
    the SAME mask rebuilt from the hash; K = 768 and 3072, one and two row groups, with and without in-kernel accumulation"""
    for K in (768, 3072):
        ends = [256, 600] if grouped else None
        rows, G = 600, (2 if grouped else 1)
        lins = [_Lin(768, K, 70 + 2 * i) for i in range(G)]
        lns = [_LN(80 + 2 * i) for i in range(G)]
        pk = blocks.LinearPack([l.weight for l in lins], [l.bias for l in lins], n_groups=G)
        lnp = blocks.LNPack(lns)
        x = _rand(rows, K, seed=90).bfloat16().requires_grad_()
        res = _rand(rows, 768, seed=91).requires_grad_()
        for t in [x, res] + [q for l in lins for q in (l.weight, l.bias)] + [q for l in lns for q in (l.weight, l.bias)]:
            t.grad = None
        ag._DropState.site = 500
        with ag.fused_grad_accumulation(fused_acc):
            y32, y16 = ag.dense_res_ln(x, res, pk, lnp, 1e-12, ends, p)
            site = ag._DropState.site
            w32, w16 = _rand(rows, 768, seed=92), _rand(rows, 768, seed=93).bfloat16()
            ((y32 * w32).sum() + (y16.float() * w16.float()).sum()).backward()
        seed = int(ag.dropout_seed(x.device).item()) & M32
        keep = _keep_mask(torch.arange(rows * 768, device='cuda', dtype=torch.int64), seed, site, p).view(rows, 768) if p > 0 else \
            torch.ones(rows, 768, dtype=torch.bool, device='cuda')
        xr, rr = x.detach().float().requires_grad_(), res.detach().clone().requires_grad_()
        refs, outs = [], []
        bounds = [0] + (ends or [rows])
        for g in range(G):
            r0, r1 = bounds[g], bounds[g + 1]
            wr = lins[g].weight.detach().bfloat16().float().requires_grad_()
            br, gr, ber = (t.detach().clone().requires_grad_() for t in (lins[g].bias, lns[g].weight, lns[g].bias))
            d = F.linear(xr[r0:r1], wr, br)
            d = torch.where(keep[r0:r1], d / (1 - p), torch.zeros_like(d))
            outs.append(F.layer_norm(d + rr[r0:r1], (768,), gr, ber, 1e-12))
            refs.append((wr, br, gr, ber))
        yr = torch.cat(outs, 0)
        ((yr * w32).sum() + (yr * w16.float()).sum()).backward()
        assert relerr(y32, yr) < 2e-2 and relerr(y16, yr) < 2e-2
        assert relerr(res.grad, rr.grad) < 2e-2 and relerr(x.grad, xr.grad) < 3e-2
        for g in range(G):
            wr, br, gr, ber = refs[g]
            assert relerr(lins[g].weight.grad, wr.grad) < 3e-2, (K, g)
            assert relerr(lins[g].bias.grad, br.grad) < 3e-2 and relerr(lns[g].weight.grad, gr.grad) < 3e-2 and relerr(lns[g].bias.grad, ber.grad) < 3e-2


@pytest.mark.parametrize('case', ['self_gasa', 'cross'])
def test_attention_dropout_fwd_bwd(ag, case):
    """attention-probability dropout inside the fused kernels against torch with the SAME mask (rebuilt from the hash)"""
    from vln_imagine_b200.ops import MASK_ADD_NEG10000
    B, p = 4, 0.25
    Lq, Lk = (30, 30) if case == 'self_gasa' else (37, 85)
    LkP = (Lk + 15) // 16 * 16
    lens = torch.tensor([Lk, Lk // 2, 5, Lk - 1])
    key_mask = (torch.arange(Lk)[None, :] < lens[:, None]).cuda()
    km = key_mask.view(torch.uint8)
    seed_t = ag.dropout_seed(torch.device('cuda', 0))
    site = 777
    dout = _rand(B * Lq, 768, seed=60).bfloat16()
    if case == 'cross':
        q = _rand(B * Lq, 768, seed=61).bfloat16().requires_grad_()
        kv = _rand(B * Lk, 1536, seed=62).bfloat16().requires_grad_()
        spec = [dict(q=(0, 0, 0), k=(1, 0, 0), v=(1, 0, 768), B=B, Lq=Lq, Lk=Lk, key_mask=km, out_row0=0, drop=(p, site, seed_t))]
        out = ag.AttentionFn.apply(spec, B * Lq, MASK_ADD_NEG10000, 2, q, kv)
        leaves = [q, kv]
        qr, kvr = q.detach().float().requires_grad_(), kv.detach().float().requires_grad_()
        Q, K, V = qr, kvr[:, :768], kvr[:, 768:]
        refs, dist, aw, ab = [qr, kvr], None, None, None
    else:
        qkv = _rand(B * Lq, 2304, seed=63).bfloat16().requires_grad_()
        dist = _rand(B, Lq, Lk, seed=64).abs() * 5
        aw = torch.tensor([[-0.5]], device='cuda', requires_grad=True)
        ab = torch.tensor([0.1], device='cuda', requires_grad=True)
        affine = torch.stack([aw.detach().view(()), ab.detach().view(())]).contiguous()
        spec = [dict(q=(0, 0, 0), k=(0, 0, 768), v=(0, 0, 1536), B=B, Lq=Lq, Lk=Lk, key_mask=km, pair_dist=dist, bias_affine=affine,
                     out_row0=0, drop=(p, site, seed_t))]
        out = ag.AttentionFn.apply(spec, B * Lq, MASK_ADD_NEG10000, 1, qkv, aw, ab)
        leaves = [qkv]
        r = qkv.detach().float().requires_grad_()
        Q, K, V = r[:, :768], r[:, 768:1536], r[:, 1536:]
        refs = [r]
    out.backward(dout)
    # torch reference with the identical mask
    seed = int(seed_t.item()) & M32
    b_i, h_i, q_i, k_i = torch.meshgrid(torch.arange(B), torch.arange(12), torch.arange(Lq), torch.arange(Lk), indexing='ij')
    eid = ((((b_i * 12 + h_i) * Lq + q_i) * LkP + k_i) & M32).cuda()
    keep = _keep_mask(eid, seed, site, p)
    qh = Q.reshape(B, Lq, 12, 64).transpose(1, 2)
    kh = K.reshape(B, Lk, 12, 64).transpose(1, 2)
    vh = V.reshape(B, Lk, 12, 64).transpose(1, 2)
    sc = qh @ kh.transpose(-1, -2) / 8.0 + (~key_mask)[:, None, None, :].float() * -10000.0
    if dist is not None:
        awr, abr = aw.detach().clone().requires_grad_(), ab.detach().clone().requires_grad_()
        sc = sc + (dist * awr.view(()) + abr.view(()))[:, None]
    pr = torch.softmax(sc, -1)
    pr = torch.where(keep, pr / (1 - p), torch.zeros_like(pr))
    ref = (pr @ vh).transpose(1, 2).reshape(B * Lq, 768)
    ref.backward(dout.float())
    assert abs(float(keep.float().mean()) - (1 - p)) < 1e-2
    assert relerr(out, ref) < 1e-2
    for got, want in zip(leaves, refs):
        assert relerr(got.grad, want.grad) < 2e-2
    if dist is not None:
        assert relerr(aw.grad, awr.grad) < 2e-2
