"""Kernel-level parity (through the C ABI) against plain PyTorch fp32 references of the same op.

Tolerances: the fp32 check-mode kernels must agree to 1e-4 (max-norm relative); the bf16
tensor-core kernels to 2e-2 against the fp32 reference and to 2e-3 against a reference that
rounds its operands to bf16 first (which isolates kernel bugs from format rounding).
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops(lib_built):
    import importlib
    o = importlib.import_module('vln_imagine_b200.ops')
    o.ensure_init(torch.zeros(1, device='cuda'))
    return o


def relerr(a, b):
    a, b = a.float(), b.float()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-20))


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


GEMM_SHAPES = [(1920, 768, 768), (2368, 2304, 768), (5440, 3072, 768), (300, 768, 3072), (128, 64, 64),
               (1, 768, 768), (129, 1536, 768), (4288, 768, 3072), (37, 512, 768), (2048, 256, 64)]


@pytest.mark.parametrize('M,N,K', GEMM_SHAPES)
@pytest.mark.parametrize('epi', [0, 1, 2])
def test_gemm_bf16(ops, M, N, K, epi):
    x = _rand(M, K, seed=1)
    w = _rand(N, K, scale=0.05, seed=2)
    b = _rand(N, scale=0.1, seed=3)
    res = _rand(M, N, seed=4)
    x16, w16 = x.bfloat16(), w.bfloat16()
    ref = F.linear(x16.float(), w16.float(), b)
    ref = [ref, F.gelu(ref), F.relu(ref)][epi]
    y = ops.gemm(x16, w16, b, epilogue=epi, out_dtype=torch.float32)
    assert relerr(y, ref) < 2e-3
    y2 = ops.gemm(x16, w16, b, residual=res, epilogue=epi, out_dtype=torch.float32)
    assert relerr(y2, ref + res) < 2e-3
    y3 = ops.gemm(x16, w16, None, epilogue=epi, out_dtype=torch.bfloat16)
    ref3 = F.linear(x16.float(), w16.float())
    ref3 = [ref3, F.gelu(ref3), F.relu(ref3)][epi]
    assert relerr(y3, ref3) < 1e-2


def _tile(ops, name: str) -> int:
    """'192' -> 192, '256p' -> 256 | TILE_PAIR (the two-CTA form)"""
    return int(name.rstrip('p')) | (ops.TILE_PAIR if name.endswith('p') else 0)


@pytest.mark.parametrize('tile', ['64', '96', '128', '192', '256', '128p', '192p', '256p'])
@pytest.mark.parametrize('M,N,K', [(1000, 768, 1536), (4416, 2304, 768), (300, 768, 64)])
def test_gemm_bf16_every_tile_shape(ops, tile, M, N, K):
    """every tile width of the tcgen05 kernel, single-CTA and CTA-pair ('p', cta_group::2) forms, with and
    without the TMA-fed residual, fp32 and bf16 outputs, GELU epilogue"""
    t = _tile(ops, tile)
    x16, w16 = _rand(M, K, seed=5).bfloat16(), _rand(N, K, scale=0.05, seed=6).bfloat16()
    b, res = _rand(N, scale=0.1, seed=7), _rand(M, N, seed=8)
    ref = F.linear(x16.float(), w16.float(), b)
    y = ops.gemm(x16, w16, b, out_dtype=torch.float32, tile=t)
    assert relerr(y, ref) < 2e-3
    y = ops.gemm(x16, w16, b, residual=res, out_dtype=torch.float32, tile=t)
    assert relerr(y, ref + res) < 2e-3
    y = ops.gemm(x16, w16, b, residual=res, epilogue=1, out_dtype=torch.float32, tile=t)
    assert relerr(y, F.gelu(ref) + res) < 2e-3
    y = ops.gemm(x16, w16, b, epilogue=1, out_dtype=torch.bfloat16, tile=t)
    assert relerr(y, F.gelu(ref)) < 1e-2


@pytest.mark.parametrize('tile', ['128', '256p'])
def test_gemm_grouped_pair_tiles(ops, tile):
    rows = [1920, 2368]
    K, N = 768, 768
    M0 = ops.pad_rows(rows[0])
    M = M0 + rows[1]
    x = torch.zeros(M, K, device='cuda')
    x[:rows[0]] = _rand(rows[0], K, seed=1)
    x[M0:] = _rand(rows[1], K, seed=2)
    w, b = _rand(2 * N, K, scale=0.05, seed=3).bfloat16(), _rand(2 * N, scale=0.1, seed=4)
    xx = x.bfloat16()
    y = ops.gemm(xx, w, b, out_dtype=torch.float32, group_row_end=[M0, M], tile=_tile(ops, tile))
    assert relerr(y[:rows[0]], F.linear(xx[:rows[0]].float(), w[:N].float(), b[:N])) < 2e-3
    assert relerr(y[M0:], F.linear(xx[M0:].float(), w[N:].float(), b[N:])) < 2e-3


def test_gemm_bf16_strided_operand_and_output(ops):
    M, K, N = 640, 768, 768
    big = _rand(M, 2304, seed=7).bfloat16()
    x16 = big[:, 768:1536]
    w16 = _rand(N, K, scale=0.05, seed=8).bfloat16()
    out = torch.zeros(M, 2 * N, dtype=torch.bfloat16, device='cuda')
    ops.gemm(x16, w16, None, out=out[:, N:])
    assert relerr(out[:, N:], x16.float() @ w16.float().t()) < 1e-2
    assert float(out[:, :N].abs().max()) == 0.0


@pytest.mark.parametrize('lowp', [True, False])
def test_gemm_grouped(ops, lowp):
    rows = [1920, 2368]
    K, N = 768, 768
    M0 = ops.pad128(rows[0])
    M = M0 + rows[1]
    x = torch.zeros(M, K, device='cuda')
    x[:rows[0]] = _rand(rows[0], K, seed=1)
    x[M0:] = _rand(rows[1], K, seed=2)
    w = _rand(2 * N, K, scale=0.05, seed=3)
    b = _rand(2 * N, scale=0.1, seed=4)
    if lowp:
        xx, ww = x.bfloat16(), w.bfloat16()
    else:
        xx, ww = x, w
    y = ops.gemm(xx, ww, b, out_dtype=torch.float32, group_row_end=[M0, M])
    ref0 = F.linear(xx[:rows[0]].float(), ww[:N].float(), b[:N])
    ref1 = F.linear(xx[M0:].float(), ww[N:].float(), b[N:])
    tol = 2e-3 if lowp else 1e-4
    assert relerr(y[:rows[0]], ref0) < tol
    assert relerr(y[M0:], ref1) < tol


@pytest.mark.parametrize('M,N,K', [(300, 768, 768), (77, 3072, 768), (1, 1, 7), (130, 768, 14), (65, 100, 33)])
@pytest.mark.parametrize('epi', [0, 1, 2])
def test_gemm_f32(ops, M, N, K, epi):
    x, w, b, res = _rand(M, K, seed=1), _rand(N, K, scale=0.05, seed=2), _rand(N, seed=3), _rand(M, N, seed=4)
    ref = F.linear(x.double(), w.double(), b.double())
    ref = [ref, F.gelu(ref), F.relu(ref)][epi] + res.double()
    y = ops.gemm(x, w, b, residual=res, epilogue=epi)
    assert relerr(y, ref.float()) < 1e-5


def _attn_ref(q, k, v, B, Lq, Lk, key_mask, pair_dist, affine, neg_inf):
    H = 12
    qh = q.float().view(B, Lq, H, 64).permute(0, 2, 1, 3)
    kh = k.float().view(B, Lk, H, 64).permute(0, 2, 1, 3)
    vh = v.float().view(B, Lk, H, 64).permute(0, 2, 1, 3)
    s = qh @ kh.transpose(-1, -2) / 8.0
    if key_mask is not None:
        if neg_inf:
            s = s.masked_fill(~key_mask.bool()[:, None, None, :], float('-inf'))
        else:
            s = s + (1.0 - key_mask.float())[:, None, None, :] * -10000.0
    if pair_dist is not None:
        s = s + (pair_dist * affine[0] + affine[1])[:, None]
    o = torch.softmax(s, -1) @ vh
    lse = torch.logsumexp(s, -1)
    return o.permute(0, 2, 1, 3).reshape(B * Lq, H * 64), lse


ATTN_CASES = [  # B, Lq, Lk, masked, gasa, neg_inf
    (3, 7, 7, True, True, False), (8, 30, 30, True, True, False), (8, 37, 85, True, False, False),
    (4, 36, 36, True, False, True), (2, 100, 212, True, False, False), (2, 100, 100, True, True, False),
    (2, 85, 53, True, False, False), (5, 1, 16, False, False, False), (2, 130, 300, True, False, False),
    (2, 16, 64, False, False, False), (2, 64, 128, True, False, True),
]


@pytest.mark.parametrize('B,Lq,Lk,masked,gasa,neg_inf', ATTN_CASES)
@pytest.mark.parametrize('lowp', [True, False])
def test_attention(ops, B, Lq, Lk, masked, gasa, neg_inf, lowp):
    dt = torch.bfloat16 if lowp else torch.float32
    qkv_q = _rand(B * Lq, 2304, seed=1).to(dt)            # strided views, like the fused QKV output
    qkv_k = _rand(B * Lk, 2304, seed=2).to(dt)
    q, k, v = qkv_q[:, :768], qkv_k[:, 768:1536], qkv_k[:, 1536:]
    key_mask = None
    if masked:
        g = torch.Generator().manual_seed(3)
        lens = torch.randint(1, Lk + 1, (B,), generator=g)
        lens[0] = Lk
        key_mask = (torch.arange(Lk)[None] < lens[:, None]).to(torch.uint8).cuda()
        if Lk > 4:
            key_mask[-1, 1] = 0                            # a hole in the middle (imagination flags)
    pair_dist = affine = None
    if gasa:
        pair_dist = (_rand(B, Lq, Lk, seed=4).abs() * 10).contiguous()
        affine = torch.tensor([-0.5, 0.1], device='cuda')
    lse = torch.empty(B, 12, Lq, device='cuda')
    o = ops.attention(q, k, v, B, Lq, Lk, key_mask=key_mask, pair_dist=pair_dist, bias_affine=affine,
                      mask_mode=ops.MASK_NEG_INF if neg_inf else ops.MASK_ADD_NEG10000, lse=lse)
    ref, ref_lse = _attn_ref(q, k, v, B, Lq, Lk, key_mask, pair_dist, affine, neg_inf)
    assert o.dtype == dt
    assert relerr(o, ref) < (1.5e-2 if lowp else 1e-5)
    assert relerr(lse, ref_lse) < (2e-3 if lowp else 1e-5)


@pytest.mark.parametrize('rows', [1, 5, 2368])
@pytest.mark.parametrize('eps', [1e-12, 1e-5])
def test_add_ln(ops, rows, eps):
    a, b = _rand(rows, 768, seed=1), _rand(rows, 768, seed=2)
    g, be = 1 + 0.1 * _rand(768, seed=3), _rand(768, seed=4)
    y32, y16 = ops.add_ln(a, b, g, be, eps, want16=True)
    ref = F.layer_norm(a + b, (768,), g, be, eps)
    assert relerr(y32, ref) < 1e-5
    assert relerr(y16, ref) < 1e-2
    y32, _ = ops.add_ln(a, None, g, be, eps, want16=False)
    assert relerr(y32, F.layer_norm(a, (768,), g, be, eps)) < 1e-5


def test_add_ln_grouped(ops):
    a = _rand(300, 768, seed=1)
    g, be = 1 + 0.1 * _rand(2, 768, seed=3), _rand(2, 768, seed=4)
    y32, _ = ops.add_ln(a, None, g, be, 1e-12, want16=False, group_row_end=[128, 300])
    assert relerr(y32[:128], F.layer_norm(a[:128], (768,), g[0], be[0], 1e-12)) < 1e-5
    assert relerr(y32[128:], F.layer_norm(a[128:], (768,), g[1], be[1], 1e-12)) < 1e-5


def test_embed_compose_bert_embeddings(ops):
    B, L = 4, 24
    ids = torch.randint(0, 1000, (B * L,), device='cuda')
    table, pos, tt = _rand(1000, 768, seed=1), _rand(512, 768, seed=2), _rand(768, seed=3)
    g, be = 1 + 0.1 * _rand(768, seed=4), _rand(768, seed=5)
    y32, y16 = ops.embed_compose(B * L, 'cuda', idx=ids, table=table, pos_table=pos, pos_period=L, const_row=tt,
                                 out_ln=(g, be), want16=True)
    ref = F.layer_norm(table[ids] + pos[:L].repeat(B, 1) + tt, (768,), g, be, 1e-12)
    assert relerr(y32, ref) < 1e-5
    assert relerr(y16, ref) < 1e-2


@pytest.mark.parametrize('fd', [4, 7, 14])
def test_embed_compose_feature_terms(ops, fd):
    rows = 333
    a, feat = _rand(rows, 768, seed=1), _rand(rows, fd, seed=2)
    fw, fb = _rand(768, fd, seed=3), _rand(768, seed=4)
    ga, ba = 1 + 0.1 * _rand(768, seed=5), _rand(768, seed=6)
    gf, bf = 1 + 0.1 * _rand(768, seed=7), _rand(768, seed=8)
    go, bo = 1 + 0.1 * _rand(768, seed=9), _rand(768, seed=10)
    idx = torch.randint(0, 3, (rows,), device='cuda')
    table, c1 = _rand(3, 768, seed=11), _rand(768, seed=12)
    y32, _ = ops.embed_compose(rows, 'cuda', a=a, a_ln=(ga, ba), feat=feat, feat_w=fw, feat_b=fb, feat_ln=(gf, bf),
                               idx=idx, table=table, const_row=c1, out_ln=(go, bo))
    ref = F.layer_norm(F.layer_norm(a, (768,), ga, ba, 1e-12) + F.layer_norm(F.linear(feat, fw, fb), (768,), gf, bf, 1e-12)
                       + table[idx] + c1, (768,), go, bo, 1e-12)
    assert relerr(y32, ref) < 1e-5
    y32, _ = ops.embed_compose(rows, 'cuda', a=a, feat=feat, feat_w=fw, feat_b=fb, feat_ln=(gf, bf))   # vp / gmap form
    assert relerr(y32, a + F.layer_norm(F.linear(feat, fw, fb), (768,), gf, bf, 1e-12)) < 1e-5
    # the padding rows behind a stream are zero-filled by the same launch (zero_rows), rows beyond them stay untouched; an updated
    # weight is picked up (the transposed copy the kernel reads follows the weight version)
    big32 = torch.full((rows + 60, 768), 7.0, device='cuda')
    big16 = torch.full((rows + 60, 768), 7.0, device='cuda', dtype=torch.bfloat16)
    fw.mul_(2.0)
    ops.embed_compose(rows, 'cuda', a=a, feat=feat, feat_w=fw, feat_b=fb, feat_ln=(gf, bf), y32=big32[:rows + 51], y16=big16[:rows + 51],
                      zero_rows=51)
    assert relerr(big32[:rows], a + F.layer_norm(F.linear(feat, fw, fb), (768,), gf, bf, 1e-12)) < 1e-5
    assert bool((big32[rows:rows + 51] == 0).all()) and bool((big16[rows:rows + 51].float() == 0).all())
    assert bool((big32[rows + 51:] == 7.0).all()) and bool((big16[rows + 51:].float() == 7.0).all())


def test_ln_dot_and_mul_bcast(ops):
    h = _rand(200, 768, seed=1)
    g, be, w, b = 1 + 0.1 * _rand(768, seed=2), _rand(768, seed=3), _rand(768, seed=4), _rand(1, seed=5)
    out = ops.ln_dot(h, g, be, 1e-12, w, b)
    ref = F.layer_norm(h, (768,), g, be, 1e-12) @ w + b
    assert relerr(out, ref) < 1e-5
    x, s = _rand(6 * 37, 768, seed=6), _rand(6 * 85, 768, seed=7)
    y32, y16 = ops.mul_bcast(x.view(6, 37, 768)[:, 5:], 37 * 768, s, 85 * 768, 6, 32, want16=True)
    ref = (x.view(6, 37, 768)[:, 5:] * s.view(6, 85, 768)[:, :1]).reshape(-1, 768)
    assert torch.equal(y32, ref)
    assert relerr(y16, ref) < 1e-2


def test_gather_mean_scatter_cosine(ops):
    src = _rand(50, 768, seed=1)
    offsets = torch.tensor([0, 3, 4, 9], dtype=torch.int32, device='cuda')
    row_idx = torch.tensor([1, 2, 2, 40, 5, 6, 7, 8, 8], dtype=torch.int32, device='cuda')
    y32, _ = ops.gather_mean(src, offsets, row_idx, 3, want16=False)
    ref = torch.stack([src[[1, 2, 2]].mean(0), src[[40]].mean(0), src[[5, 6, 7, 8, 8]].mean(0)])
    assert relerr(y32, ref) < 1e-6
    dst = torch.zeros(10, 768, device='cuda')
    ops.scatter_rows(y32, torch.tensor([7, 0, 3], dtype=torch.int32, device='cuda'), dst)
    assert torch.equal(dst[[7, 0, 3]], y32) and float(dst[[1, 2, 4, 5, 6, 8, 9]].abs().max()) == 0
    p, t = _rand(33, 768, seed=2), _rand(33, 768, seed=3)
    loss, rows = ops.cosine_loss(p, t, 33, 'cuda')
    ref_rows = 1 - F.cosine_similarity(p, t, dim=-1)
    assert relerr(rows, ref_rows) < 1e-5
    assert abs(float(loss) - float(ref_rows.mean())) < 1e-5
    loss0, _ = ops.cosine_loss(None, None, 0, 'cuda')
    assert float(loss0) == 0.0


def test_infonce(ops):
    R, Nn = 9, 14
    p, t, negs = _rand(R, 768, seed=1), _rand(R, 768, seed=2), _rand(Nn, 768, seed=3)
    row_ep = torch.tensor([0, 0, 1, 1, 1, 2, 3, 3, 3], dtype=torch.int32, device='cuda')
    neg_ep = torch.tensor([0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 3, 3, 3], dtype=torch.int32, device='cuda')
    T = 0.07
    loss, _ = ops.infonce_loss(p, t, negs, row_ep, neg_ep, T, R, Nn, 'cuda')
    ref = []
    for r in range(R):
        keep = negs[neg_ep != row_ep[r]]
        allt = torch.cat([t[r:r + 1], keep], 0)
        sim = F.cosine_similarity(p[r:r + 1], allt) / T
        ref.append(F.cross_entropy(sim[None], torch.zeros(1, dtype=torch.long, device='cuda')))
    assert abs(float(loss) - float(torch.stack(ref).mean())) < 1e-4


def test_margin_loss(ops):
    """margin alignment loss (H/models/vilmodel_cmt.py:825-856) against torch; a row without admissible negatives is NaN
    there (mean of an empty tensor) and here"""
    R, Nn = 9, 14
    p, t, negs = _rand(R, 768, seed=1), _rand(R, 768, seed=2), _rand(Nn, 768, seed=3)
    row_ep = torch.tensor([0, 0, 1, 1, 1, 2, 3, 3, 3], dtype=torch.int32, device='cuda')
    neg_ep = torch.tensor([0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 3, 3, 3], dtype=torch.int32, device='cuda')
    margin = 0.5
    loss, _ = ops.margin_loss(p, t, negs, row_ep, neg_ep, margin, R, Nn, 'cuda')
    ref = []
    for r in range(R):
        pos = F.cosine_similarity(p[r:r + 1], t[r:r + 1]).squeeze()
        neg = F.cosine_similarity(p[r:r + 1], negs[neg_ep != row_ep[r]])
        ref.append((1 - pos) + F.relu(margin + neg - pos).mean())
    assert abs(float(loss) - float(torch.stack(ref).mean())) < 1e-5
    same = torch.zeros(Nn, dtype=torch.int32, device='cuda')
    lone, _ = ops.margin_loss(p[:2], t[:2], negs, torch.zeros(2, dtype=torch.int32, device='cuda'), same, margin, 2, Nn, 'cuda')
    assert torch.isnan(lone)


def _fuse_reference(global_logits, local_logits, gmap_vpids, visited, vp_cand_vpids):
    """the per-episode python loop of the reference (VLN-DUET/map_nav_src/models/vilmodel.py:1198-1217)"""
    fused = global_logits.clone()
    fused[:, 0] += local_logits[:, 0]
    for i in range(global_logits.shape[0]):
        vis = set(vp for vp, m in zip(gmap_vpids[i], visited[i].tolist()) if m)
        tmp, bw = {}, 0
        for j, c in enumerate(vp_cand_vpids[i]):
            if j > 0:
                if c in vis:
                    bw = bw + local_logits[i, j]
                else:
                    tmp[c] = local_logits[i, j]
        for j, vp in enumerate(gmap_vpids[i]):
            if j > 0 and vp not in vis:
                fused[i, j] += tmp[vp] if vp in tmp else bw
    return fused


@pytest.mark.parametrize('use_fuse', [True, False])
def test_fuse_logits_and_navtype_mask(ops, use_fuse):
    import importlib
    duet = importlib.import_module('vln_imagine_b200.duet')
    B, G, P = 6, 40, 37
    g = torch.Generator().manual_seed(0)
    g_raw, l_raw, f_raw = _rand(B, G, seed=1), _rand(B, P, seed=2), _rand(B, seed=3)
    gm = torch.zeros(B, G, dtype=torch.bool); gv = torch.zeros(B, G, dtype=torch.bool)
    nav = torch.zeros(B, P, dtype=torch.bool)
    gmap_vpids, cand_vpids = [], []
    for b in range(B):
        n = int(torch.randint(6, G + 1, (1,), generator=g))
        nv = int(torch.randint(1, n - 3, (1,), generator=g))
        gm[b, :n] = True
        gv[b, 1:1 + nv] = True
        ids = [None] + ['n%d_%d' % (b, j) for j in range(1, n)]
        gmap_vpids.append(ids)
        nc = int(torch.randint(2, min(7, n - nv), (1,), generator=g))
        cands = [ids[1 + int(torch.randint(0, nv, (1,), generator=g))]]              # one visited candidate
        cands += [ids[j] for j in range(1 + nv, 1 + nv + nc - 1)]                    # unvisited ones in the graph
        if b == 0:
            cands.append('not_in_graph')
        if b == 1:
            cands.append(cands[-1])                                                  # duplicate id: the last one wins
            cands.append(ids[1])                                                     # a second visited candidate
        cand_vpids.append([None] + cands)
        nav[b, :len(cands) + 1] = True
    gids = torch.from_numpy(duet._IdTable().encode(gmap_vpids, G, -1))
    tab = duet._IdTable()
    gids = torch.from_numpy(tab.encode(gmap_vpids, G, -1)).cuda()
    cids = torch.from_numpy(tab.encode(cand_vpids, P, -2)).cuda()
    u8 = lambda t: t.to(torch.uint8).cuda()   # noqa: E731
    gl, ll, fl = ops.duet_fuse_logits(g_raw, l_raw, f_raw if use_fuse else None, u8(gm), u8(gv), u8(nav), gids, cids, B, G, P)
    fw = torch.sigmoid(f_raw)[:, None] if use_fuse else 0.5
    rg = (g_raw * fw).masked_fill(gv.cuda(), float('-inf')).masked_fill(~gm.cuda(), float('-inf'))
    rl = (l_raw * (1 - fw)).masked_fill(~nav.cuda(), float('-inf'))
    rf = _fuse_reference(rg.cpu(), rl.cpu(), gmap_vpids, gv, cand_vpids).cuda()
    for a, b in ((gl, rg), (ll, rl), (fl, rf)):
        assert torch.equal(torch.isinf(a), torch.isinf(b))
        fin = torch.isfinite(b)
        assert float((a[fin] - b[fin]).abs().max()) < 1e-6
    types = torch.randint(0, 3, (B, P), device='cuda')
    out = ops.mask_logits_navtype(l_raw, types)
    assert torch.equal(out, l_raw.masked_fill(types == 0, float('-inf')))


def test_copy_rows(ops):
    B, L, I = 3, 5, 2
    txt, img = _rand(B, L, 768, seed=1), _rand(B, I, 768, seed=2)
    C = L + I
    c32 = torch.zeros(B * C, 768, device='cuda')
    c16 = torch.zeros(B * C, 768, dtype=torch.bfloat16, device='cuda')
    ops.copy_rows(txt, L * 768, 768, B, L, c32, c16, C * 768, 768)
    ops.copy_rows(img, I * 768, 768, B, I, c32[L:], c16[L:], C * 768, 768)
    ref = torch.cat([txt, img], 1).view(B * C, 768)
    assert torch.equal(c32, ref) and torch.equal(c16, ref.bfloat16())
    first = torch.zeros(B, 1536, device='cuda')
    ops.copy_rows(txt, L * 768, 768, B, 1, first[:, 768:], None, 1536, 768)
    assert torch.equal(first[:, 768:], txt[:, 0]) and float(first[:, :768].abs().max()) == 0


def test_cast_bf16(ops):
    x = _rand(1003, seed=1)
    assert torch.equal(ops.cast_h16(x, dtype=torch.bfloat16), x.bfloat16())


def test_argument_errors_are_reported_not_fatal(ops):
    import importlib
    _lib = importlib.import_module('vln_imagine_b200._lib')
    x16 = _rand(128, 100, seed=1).bfloat16()              # K not a multiple of 64
    with pytest.raises(_lib.VlnImagineError, match='multiple of 64'):
        ops.gemm(x16, _rand(64, 100, seed=2).bfloat16())
    with pytest.raises(_lib.VlnImagineError, match='fp32 output'):
        ops.gemm(_rand(128, 64, seed=1).bfloat16(), _rand(64, 64, seed=2).bfloat16(), residual=_rand(128, 64, seed=3),
                 out_dtype=torch.bfloat16)
    with pytest.raises(_lib.VlnImagineError, match='CUDA tensor|no CPU path|must be'):
        ops.ensure_init(torch.zeros(1))




# ---------------------------------------------------------------------------------------------------------------------
# vi_gemm16: fp16 operands, the packed-polynomial GELU, LayerNorm folded into the neighbouring contractions
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('M,N,K', [(1920, 768, 768), (4416, 3072, 768), (300, 768, 3072), (37, 512, 768)])
@pytest.mark.parametrize('epi', [0, 1, 2])
def test_gemm_f16_operands(ops, M, N, K, epi):
    """fp16 operands through the same tcgen05 kernel (instruction-descriptor formats 0): exact up to fp32 accumulation
    against a reference that rounds its operands to fp16 first, and 8x closer to the unrounded product than bf16"""
    x, w, b = _rand(M, K, seed=1), _rand(N, K, scale=0.05, seed=2), _rand(N, scale=0.1, seed=3)
    res = _rand(M, N, seed=4)
    xh, wh = x.half(), w.half()
    ref = F.linear(xh.float(), wh.float(), b)
    ref = [ref, F.gelu(ref), F.relu(ref)][epi]
    y = ops.gemm(xh, wh, b, residual=res, epilogue=epi, out_dtype=torch.float32)
    assert relerr(y, ref + res) < 1e-4
    y16 = ops.gemm(xh, wh, b, epilogue=epi)
    assert y16.dtype == torch.float16 and relerr(y16, ref) < 2e-3
    exact = F.linear(x, w, b)
    exact = [exact, F.gelu(exact), F.relu(exact)][epi]
    e16 = relerr(ops.gemm(xh, wh, b, epilogue=epi, out_dtype=torch.float32), exact)
    eb = relerr(ops.gemm(x.bfloat16(), w.bfloat16(), b, epilogue=epi, out_dtype=torch.float32), exact)
    assert e16 < 0.3 * eb, (e16, eb)


def test_gemm_f16_saturates_instead_of_overflowing(ops):
    x = torch.full((128, 64), 60.0, device='cuda').half()
    w = torch.full((64, 64), 60.0, device='cuda').half()
    y = ops.gemm(x, w)                                   # 64 * 3600 = 230400 > 65504
    assert torch.isfinite(y.float()).all() and float(y.float().max()) == 65504.0


def test_gelu_polynomial_epilogue(ops):
    """the MUFU-free erf polynomial of the GEMM epilogue against F.gelu over the whole input range"""
    M, K = 512, 64
    x16 = torch.zeros((M, K), device='cuda').bfloat16()
    x16[:, 0] = 1.0
    w16 = torch.zeros((64, K), device='cuda').bfloat16()
    outs = []
    # y[m, n] = x[m, :] . w[n, :] + b[n] with w = 0: the bias sweeps the input range of the activation
    for i in range(8):
        b = torch.linspace(-12 + 3 * i, -9 + 3 * i, 64, device='cuda')
        y = ops.gemm(x16[:128], w16, b, epilogue=1, out_dtype=torch.float32)
        assert float((y[0] - F.gelu(b)).abs().max()) < 1e-4
        outs.append(y[0])
    assert torch.isfinite(torch.cat(outs)).all()


@pytest.mark.parametrize('fmt', [torch.bfloat16, torch.float16])
@pytest.mark.parametrize('M,grouped', [(4416, True), (2304, False), (300, False), (9024, True), (1, False)])
@pytest.mark.parametrize('eps', [1e-12, 1e-5])
def test_gemm_layernorm_folding(ops, fmt, M, grouped, eps):
    """producer (dense + residual, writes raw sums + per-chunk row statistics + a 16-bit copy), consumer with the LayerNorm
    folded into its weights (VI_LN_FOLD, also with GELU), consumer with the LayerNorm applied to its residual operand
    (VI_LN_RESIDUAL): against F.linear / F.layer_norm in fp32 on the same rounded operands"""
    from vln_imagine_b200 import _lib
    G = 2 if grouped else 1
    ends = [2048 if M == 4416 else 5632, M] if grouped else None
    bounds = [0] + (ends or [M])
    x16 = _rand(M, 768, seed=11).to(fmt)
    wo = _rand(G * 768, 768, scale=0.05, seed=12)
    bo = _rand(G * 768, scale=0.1, seed=13)
    res = _rand(M, 768, seed=14) * 2.0 + 0.3
    gamma = 1 + _rand(G, 768, scale=0.2, seed=15)
    beta = _rand(G, 768, scale=0.2, seed=16)
    w1 = _rand(G * 3072, 768, scale=0.05, seed=17)
    b1 = _rand(G * 3072, scale=0.1, seed=18)

    def per_group(fn):
        return torch.cat([fn(g, slice(bounds[g], bounds[g + 1])) for g in range(G)])

    # ---- producer
    z32 = torch.empty((M, 768), device='cuda')
    z16 = torch.empty((M, 768), device='cuda', dtype=fmt)
    stats = torch.full((24, M, 2), float('nan'), device='cuda')
    ops.gemm(x16, wo.to(fmt), bo, residual=res, out=z32, out16=z16, group_row_end=ends, stats_out=stats)
    z_ref = per_group(lambda g, r: F.linear(x16[r].float(), wo[g * 768:(g + 1) * 768].to(fmt).float(), bo[g * 768:(g + 1) * 768]) + res[r])
    assert relerr(z32, z_ref) < 1e-4
    assert torch.equal(z16, z32.to(fmt))
    ch = z32.view(M, 24, 32)
    assert relerr(stats[:, :, 0].t(), ch.mean(-1)) < 1e-5
    assert relerr(stats[:, :, 1].t(), ((ch - ch.mean(-1, keepdim=True)) ** 2).sum(-1)) < 1e-4
    ln_ref = per_group(lambda g, r: F.layer_norm(z32[r], (768,), gamma[g], beta[g], eps))

    # ---- VI_LN_FOLD consumer (with GELU): weights W * gamma, s = row sums of the ROUNDED product, c = W beta + b
    wg = (w1.view(G, 3072, 768) * gamma[:, None, :]).reshape(G * 3072, 768).to(fmt)
    s = wg.double().sum(1).float()
    c = (torch.einsum('gnk,gk->gn', w1.view(G, 3072, 768).double(), beta.double()).reshape(-1) + b1.double()).float()
    for epi in (0, 1):
        y = ops.gemm(z16, wg, c, epilogue=epi, out_dtype=torch.float32, group_row_end=ends, ln=(_lib.LN_FOLD, s, stats, eps))
        ref = per_group(lambda g, r: F.linear(ln_ref[r], w1[g * 3072:(g + 1) * 3072], b1[g * 3072:(g + 1) * 3072]))
        ref = F.gelu(ref) if epi else ref
        assert relerr(y, ref) < (3e-3 if fmt == torch.float16 else 2e-2), epi

    # ---- VI_LN_RESIDUAL consumer: out = x W^T + b + LayerNorm(z)
    h16 = _rand(M, 768, seed=19).to(fmt)
    w2 = _rand(G * 768, 768, scale=0.05, seed=20)
    b2 = _rand(G * 768, scale=0.1, seed=21)
    out = ops.gemm(h16, w2.to(fmt), (beta.reshape(-1) + b2).contiguous(), residual=z32, out_dtype=torch.float32, group_row_end=ends,
                   ln=(_lib.LN_RESIDUAL, gamma.reshape(-1).contiguous(), stats, eps))
    ref = per_group(lambda g, r: F.linear(h16[r].float(), w2[g * 768:(g + 1) * 768].to(fmt).float(), b2[g * 768:(g + 1) * 768])) + ln_ref
    assert relerr(out, ref) < 1e-4


def test_embed_compose_chained_layernorm(ops):
    """y32 = LN_out(sum), y16 = LN2(y32) from one launch (first pre-norm layer of the panorama encoder)"""
    rows = 777
    a = _rand(rows, 768, seed=31)
    g1, b1 = 1 + _rand(768, scale=0.1, seed=32), _rand(768, scale=0.1, seed=33)
    g2, b2 = 1 + _rand(768, scale=0.1, seed=34), _rand(768, scale=0.1, seed=35)
    with ops.half_format(torch.float16):
        y32, y16 = ops.embed_compose(rows, a.device, a=a, out_ln=(g1, b1), eps=1e-12, want16=True, want32=True, ln2=(g2, b2), ln2_eps=1e-5)
    r32 = F.layer_norm(a, (768,), g1, b1, 1e-12)
    assert relerr(y32, r32) < 1e-5
    assert y16.dtype == torch.float16 and relerr(y16, F.layer_norm(r32, (768,), g2, b2, 1e-5)) < 2e-3


# longer, wider and edge-case problems on top of ATTN_CASES (> 96 keys: the generic kernel; 1 key; odd query counts)
ATTN_EDGE_CASES = ATTN_CASES + [(64, 30, 85, True, False, False), (3, 64, 256, True, False, False), (2, 65, 17, True, True, False),
                                (2, 200, 200, True, False, False), (1, 37, 240, False, False, True)]


SP_ATTN_CASES = [c for c in ATTN_EDGE_CASES if c[2] <= 96] + [(64, 37, 85, True, False, False), (3, 50, 96, True, True, False),
                                                              (2, 40, 81, True, True, True), (2, 17, 1, False, False, False)]


@pytest.mark.parametrize('B,Lq,Lk,masked,gasa,neg_inf', SP_ATTN_CASES)
@pytest.mark.parametrize('fmt', [torch.bfloat16, torch.float16])
def test_attention_single_pass(ops, B, Lq, Lk, masked, gasa, neg_inf, fmt):
    """attn_fwd_sp_kernel (the default for <= 96 keys without dropout / lse: exactly unrolled key blocks, one softmax pass in the
    log2 domain) against the fp32 reference and against the generic kernel (which a log-sum-exp output selects) on the same
    inputs"""
    qkv_q = _rand(B * Lq, 2304, seed=1).to(fmt)
    qkv_k = _rand(B * Lk, 2304, seed=2).to(fmt)
    q, k, v = qkv_q[:, :768], qkv_k[:, 768:1536], qkv_k[:, 1536:]
    key_mask = None
    if masked:
        g = torch.Generator().manual_seed(3)
        lens = torch.randint(1, Lk + 1, (B,), generator=g)
        lens[0] = Lk
        key_mask = (torch.arange(Lk)[None] < lens[:, None]).to(torch.uint8).cuda()
        if Lk > 4:
            key_mask[-1, 1] = 0
    pair_dist = affine = None
    if gasa:
        pair_dist = (_rand(B, Lq, Lk, seed=4).abs() * 10).contiguous()
        affine = torch.tensor([-0.5, 0.1], device='cuda')
    mode = ops.MASK_NEG_INF if neg_inf else ops.MASK_ADD_NEG10000
    prob = dict(q=q, k=k, v=v, B=B, Lq=Lq, Lk=Lk, key_mask=key_mask, pair_dist=pair_dist, bias_affine=affine)
    o = torch.full((B * Lq + 3, 768), 7.0, dtype=fmt, device='cuda')
    ops.attention_multi([dict(prob, out=o[:B * Lq])], mask_mode=mode)
    o_gen = torch.empty((B * Lq, 768), dtype=fmt, device='cuda')
    lse = torch.empty((B, 12, Lq), dtype=torch.float32, device='cuda')
    ops.attention_multi([dict(prob, out=o_gen, lse=lse)], mask_mode=mode)
    ref, _ = _attn_ref(q, k, v, B, Lq, Lk, key_mask, pair_dist, affine, neg_inf)
    tol = 1.5e-2 if fmt == torch.bfloat16 else 2.5e-3
    assert relerr(o[:B * Lq], ref) < tol
    assert relerr(o[:B * Lq], o_gen) < tol / 3            # the two kernels differ in fp32 association only
    assert bool((o[B * Lq:].float() == 7.0).all())


@pytest.mark.parametrize('fmt', [torch.bfloat16, torch.float16])
def test_attention_single_pass_multi_problem(ops, fmt):
    """both token streams of a row-stacked activation in one launch through the default dispatcher (single-pass kernel): key-block
    counts differ per problem (30 -> 2 blocks, 37 -> 3, 85 -> 6); padding rows stay untouched"""
    B = 16
    for (La, Lb, Lka, Lkb, gasa) in ((30, 37, 85, 85, False), (30, 37, 30, 37, True), (85, 53, 53, 85, False)):
        ra = (B * La + 255) // 256 * 256
        R = ra + B * Lb
        x = _rand(R, 2304, seed=5).to(fmt)
        ctx = _rand(B * 85, 3072, seed=6).to(fmt)
        out = torch.full((R, 768), 7.0, device='cuda', dtype=fmt)
        ga, gb = torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)
        ma = (torch.arange(Lka)[None] < torch.randint(1, Lka + 1, (B,), generator=ga)[:, None]).to(torch.uint8).cuda()
        mb = (torch.arange(Lkb)[None] < torch.randint(1, Lkb + 1, (B,), generator=gb)[:, None]).to(torch.uint8).cuda()
        dist = (_rand(B, La, Lka, seed=7).abs() * 10).contiguous() if gasa else None
        aff = torch.tensor([-0.3, 0.05], device='cuda') if gasa else None
        if Lka == 85 and Lkb == 85:
            ka, va, kb, vb = ctx[:, :768], ctx[:, 768:1536], ctx[:, 1536:2304], ctx[:, 2304:]
        elif gasa:
            ka, va, kb, vb = x[:B * La, 768:1536], x[:B * La, 1536:], x[ra:, 768:1536], x[ra:, 1536:]
        else:
            ka, va, kb, vb = x[ra:, 768:1536], x[ra:, 1536:], x[:B * La, 768:1536], x[:B * La, 1536:]
        pa = dict(q=x[:B * La, :768], k=ka, v=va, out=out[:B * La], B=B, Lq=La, Lk=Lka, key_mask=ma, pair_dist=dist, bias_affine=aff)
        pb = dict(q=x[ra:, :768], k=kb, v=vb, out=out[ra:], B=B, Lq=Lb, Lk=Lkb, key_mask=mb)
        ops.attention_multi([pa, pb])
        refa, _ = _attn_ref(pa['q'], ka, va, B, La, Lka, ma, dist, aff, False)
        refb, _ = _attn_ref(pb['q'], kb, vb, B, Lb, Lkb, mb, None, None, False)
        tol = 1.5e-2 if fmt == torch.bfloat16 else 2.5e-3
        assert relerr(out[:B * La], refa) < tol and relerr(out[ra:], refb) < tol
        assert bool((out[B * La:ra].float() == 7.0).all())


@pytest.mark.parametrize('B,Lq,Lk,masked,gasa,neg_inf', [(8, 30, 30, True, True, False), (8, 37, 85, True, False, False),
                                                          (4, 36, 36, True, False, True), (2, 130, 300, True, False, False)])
def test_attention_fp16_operands(ops, B, Lq, Lk, masked, gasa, neg_inf):
    """the default (mma.sync) attention kernel with fp16 operands / output, as the 16-bit inference mode runs it"""
    qkv_q = _rand(B * Lq, 2304, seed=1).half()
    qkv_k = _rand(B * Lk, 2304, seed=2).half()
    q, k, v = qkv_q[:, :768], qkv_k[:, 768:1536], qkv_k[:, 1536:]
    g = torch.Generator().manual_seed(3)
    lens = torch.randint(1, Lk + 1, (B,), generator=g)
    lens[0] = Lk
    key_mask = (torch.arange(Lk)[None] < lens[:, None]).to(torch.uint8).cuda()
    pair_dist = affine = None
    if gasa:
        pair_dist = (_rand(B, Lq, Lk, seed=4).abs() * 10).contiguous()
        affine = torch.tensor([-0.5, 0.1], device='cuda')
    o = ops.attention(q, k, v, B, Lq, Lk, key_mask=key_mask, pair_dist=pair_dist, bias_affine=affine,
                      mask_mode=ops.MASK_NEG_INF if neg_inf else ops.MASK_ADD_NEG10000)
    ref, _ = _attn_ref(q, k, v, B, Lq, Lk, key_mask, pair_dist, affine, neg_inf)
    assert o.dtype == torch.float16 and relerr(o, ref) < 2.5e-3
