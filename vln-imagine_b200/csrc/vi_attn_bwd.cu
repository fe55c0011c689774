// vi_attn_bwd.cu - attention backward on bf16 operands with warp-level tensor-core tiles (fine-tuning path).
//
// One CTA (4 warps) per (episode, head).  Q, K, V, dO of the head are staged in shared memory with cp.async.
//   phase 1 (a warp per 16-query tile):  S = Q K^T / 8 + mask (+ GASA bias), P = softmax(S), dP = dO V^T,
//            D = rowsum(P o dP), dS = P o (dP - D), dQ = dS K / 8;  P and dS are parked in shared memory (bf16);
//   phase 2 (a warp per 16-key tile):    dV = P^T dO,  dK = dS^T Q / 8  (ldmatrix.trans gives the transposed operands).
// All contractions are mma.sync m16n8k16 (bf16 in, fp32 accumulate); softmax and the dS algebra are fp32.
// The single-CTA kernel takes the short sequences (<= 256 queries, <= 128 keys): nothing is tiled over keys, the whole score
// row of a query tile lives in registers.  GASA: d(w), d(b) of the affine bias w * dist + b are accumulated with two fp32
// atomics per CTA.  Longer sequences, up to the forward's 512 keys, take the two key-blocked kernels further down
// (attn_bwd_dq_kernel, attn_bwd_dkv_kernel), which are deterministic.
//
// Reference semantics: torch.autograd of BertSelfAttention / BertOutAttention (VLN-DUET/map_nav_src/models/vilmodel.py:
// 118-134, 336-349) and of nn.MultiheadAttention (models/transformer.py:176-177).
#include "vi_common.cuh"

namespace {

constexpr int DH = 64;
constexpr int ROW = 72;            // bf16 elements per staged row (64 + 8): conflict-free ldmatrix

struct AttnBwdTcParams {
  const bf16* q; long long ldq;
  const bf16* k; long long ldk;
  const bf16* v; long long ldv;
  const bf16* dout; long long ldo;
  bf16* dq; long long lddq;
  bf16* dk; long long lddk;
  bf16* dv; long long lddv;
  const uint8_t* key_mask;
  const float* pair_dist;
  const float* bias_affine;
  float* d_affine;
  int B, H, Lq, Lk, LqP, LkP, mask_mode;
  uint32_t drop_thresh;        // 0 = no attention dropout
  float drop_scale;
  uint32_t drop_site;
  const uint32_t* drop_seed;
  // key-blocked kernels only: per-row softmax statistics [3][B * H][LqP] (max, 1 / sum, D) and the GASA partials of the dQ
  // kernel's CTAs (n_aff pairs)
  float* stats;
  float* aff_part;
  int n_aff;
};

__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;       // src-size 0 zero-fills the 16 bytes
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}

// NT = 8-key score tiles per query row held in registers (LkP <= 8 * NT)
// CTAs per SM asked of the register allocator: the grid is episodes x heads (768 CTAs at the fine-tuning shapes), and at the
// 195 registers NT = 12 takes unconstrained only two CTAs fit an SM (2.6 waves); 167 registers (no spills) fit three.
template <int NT>
__global__ void __launch_bounds__(128, NT == 12 ? 3 : NT == 6 ? 4 : 1) attn_bwd_bf16_kernel(const AttnBwdTcParams p) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  const int LqP = p.LqP, LkP = p.LkP;
  const int PP = LkP + 8;                                    // pitch of the P / dS planes (bf16 elements)
  bf16* Ks = reinterpret_cast<bf16*>(smem);                  // [LkP][72]
  bf16* Vs = Ks + (size_t)LkP * ROW;                         // [LkP][72]
  bf16* Qs = Vs + (size_t)LkP * ROW;                         // [LqP][72]
  bf16* Os = Qs + (size_t)LqP * ROW;                         // [LqP][72]   dO
  bf16* Ps = Os + (size_t)LqP * ROW;                         // [LqP][PP]
  bf16* Ss = Ps + (size_t)LqP * PP;                          // [LqP][PP]   dS
  float* madd = reinterpret_cast<float*>(Ss + (size_t)LqP * PP);   // [LkP]
  const int b = blockIdx.y, h = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const bf16* qg = p.q + (long long)b * p.Lq * p.ldq + h * DH;
  const bf16* kg = p.k + (long long)b * p.Lk * p.ldk + h * DH;
  const bf16* vg = p.v + (long long)b * p.Lk * p.ldv + h * DH;
  const bf16* og = p.dout + (long long)b * p.Lq * p.ldo + h * DH;
  const uint32_t ks_u = smem_u32(Ks), vs_u = smem_u32(Vs), qs_u = smem_u32(Qs), os_u = smem_u32(Os);
  const uint32_t ps_u = smem_u32(Ps), ss_u = smem_u32(Ss);
  for (int e = tid; e < LkP * 8; e += 128) {
    const int key = e >> 3, ch = e & 7;
    const bool ok = key < p.Lk;
    const int kk = ok ? key : 0;
    cp_async16(ks_u + (uint32_t)(key * ROW + ch * 8) * 2, kg + (long long)kk * p.ldk + ch * 8, ok);
    cp_async16(vs_u + (uint32_t)(key * ROW + ch * 8) * 2, vg + (long long)kk * p.ldv + ch * 8, ok);
  }
  for (int e = tid; e < LqP * 8; e += 128) {
    const int r = e >> 3, ch = e & 7;
    const bool ok = r < p.Lq;
    const int rr = ok ? r : 0;
    cp_async16(qs_u + (uint32_t)(r * ROW + ch * 8) * 2, qg + (long long)rr * p.ldq + ch * 8, ok);
    cp_async16(os_u + (uint32_t)(r * ROW + ch * 8) * 2, og + (long long)rr * p.ldo + ch * 8, ok);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (int key = tid; key < LkP; key += 128) {
    float m = 0.f;
    if (key >= p.Lk) m = -INFINITY;
    else if (p.key_mask && !p.key_mask[(long long)b * p.Lk + key]) m = (p.mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f;
    madd[key] = m;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const int g = lane >> 2, tg = lane & 3;
  const int lm = lane >> 3, lr = lane & 7;                   // ldmatrix: this lane addresses row lr of matrix lm
  const int nt_run = LkP >> 3;                               // 8-key tiles actually present (even)
  float bw = 0.f, bb = 0.f;
  if (p.pair_dist) { bw = p.bias_affine[0]; bb = p.bias_affine[1]; }
  float aw = 0.f, ab = 0.f;                                  // GASA affine gradients of this thread
  const bool drop = p.drop_thresh != 0;
  const uint32_t dkey = drop ? vi_drop_key(p.drop_seed, p.drop_site) : 0u;
  // dropout element id = ((b * H + h) * Lq + q) * LkP + key, the same as in the forward kernel
  const uint32_t dbase = (uint32_t)((b * p.H + h) * p.Lq) * (uint32_t)LkP;

  // ------------------------------------------------ phase 1: a warp per 16-query tile
  for (int qt = warp; qt < (LqP >> 4); qt += 4) {
    const int q0 = qt * 16;
    const int r0 = q0 + g, r1 = q0 + g + 8;
    uint32_t qa[4][4], da[4][4];                             // Q and dO fragments of the tile, 4 k-steps over d
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t off = (uint32_t)((q0 + (lm & 1) * 8 + lr) * ROW + (lm >> 1) * 8 + ks * 16) * 2;
      ldsm_x4(qa[ks], qs_u + off);
      ldsm_x4(da[ks], os_u + off);
    }
    float s[NT][4], dp[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
      dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
    }
#pragma unroll
    for (int np = 0; np < NT / 2; ++np) {
      if (2 * np < nt_run) {
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          uint32_t kb[4], vb[4];   // (keys 0-7, d 0-7) (keys 0-7, d 8-15) (keys 8-15, d 0-7) (keys 8-15, d 8-15)
          const uint32_t off = (uint32_t)((np * 16 + (lm >> 1) * 8 + lr) * ROW + ks * 16 + (lm & 1) * 8) * 2;
          ldsm_x4(kb, ks_u + off);
          ldsm_x4(vb, vs_u + off);
          mma_16816(s[2 * np], qa[ks], kb[0], kb[1]);
          mma_16816(s[2 * np + 1], qa[ks], kb[2], kb[3]);
          mma_16816(dp[2 * np], da[ks], vb[0], vb[1]);
          mma_16816(dp[2 * np + 1], da[ks], vb[2], vb[3]);
        }
      }
    }
    const float* pd0 = nullptr;
    const float* pd1 = nullptr;
    if (p.pair_dist) {
      pd0 = p.pair_dist + ((long long)b * p.Lq + (r0 < p.Lq ? r0 : 0)) * p.Lk;
      pd1 = p.pair_dist + ((long long)b * p.Lq + (r1 < p.Lq ? r1 : 0)) * p.Lk;
    }
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      if (nt < nt_run) {
        const int key = nt * 8 + 2 * tg;
        const float2 ma = *reinterpret_cast<const float2*>(madd + key);
        float b00 = 0.f, b01 = 0.f, b10 = 0.f, b11 = 0.f;
        if (pd0) {
          if (key < p.Lk) { b00 = fmaf(bw, (*(pd0 + key)), bb); b10 = fmaf(bw, (*(pd1 + key)), bb); }
          if (key + 1 < p.Lk) { b01 = fmaf(bw, (*(pd0 + key + 1)), bb); b11 = fmaf(bw, (*(pd1 + key + 1)), bb); }
        }
        s[nt][0] = s[nt][0] * 0.125f + ma.x + b00;
        s[nt][1] = s[nt][1] * 0.125f + ma.y + b01;
        s[nt][2] = s[nt][2] * 0.125f + ma.x + b10;
        s[nt][3] = s[nt][3] * 0.125f + ma.y + b11;
        m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
        m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
      }
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    const float mu0 = (m0 == -INFINITY) ? 0.f : m0, mu1 = (m1 == -INFINITY) ? 0.f : m1;
    float l0 = 0.f, l1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      if (nt < nt_run) {
        s[nt][0] = __expf(s[nt][0] - mu0); s[nt][1] = __expf(s[nt][1] - mu0);
        s[nt][2] = __expf(s[nt][2] - mu1); s[nt][3] = __expf(s[nt][3] - mu1);
        l0 += s[nt][0] + s[nt][1];
        l1 += s[nt][2] + s[nt][3];
      }
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = l0 > 0.f ? 1.0f / l0 : 0.f, i1 = l1 > 0.f ? 1.0f / l1 : 0.f;
    float d0 = 0.f, d1 = 0.f;                                 // D = rowsum(P o dP)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      if (nt < nt_run) {
        s[nt][0] *= i0; s[nt][1] *= i0; s[nt][2] *= i1; s[nt][3] *= i1;
        if (drop) {      // O = (P o mask / (1 - p)) V: the mask scales dP here and P where it feeds dV below
          const uint32_t e0 = dbase + (uint32_t)r0 * (uint32_t)LkP + (uint32_t)(nt * 8 + 2 * tg);
          const uint32_t e1 = dbase + (uint32_t)r1 * (uint32_t)LkP + (uint32_t)(nt * 8 + 2 * tg);
          dp[nt][0] *= vi_hash32(e0, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
          dp[nt][1] *= vi_hash32(e0 + 1, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
          dp[nt][2] *= vi_hash32(e1, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
          dp[nt][3] *= vi_hash32(e1 + 1, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
        }
        d0 = fmaf(s[nt][0], dp[nt][0], fmaf(s[nt][1], dp[nt][1], d0));
        d1 = fmaf(s[nt][2], dp[nt][2], fmaf(s[nt][3], dp[nt][3], d1));
      }
    }
    d0 += __shfl_xor_sync(0xffffffffu, d0, 1);
    d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 1);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    // dS = P o (dP - D); park P and dS (bf16) for phase 2; GASA affine gradients
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      if (nt < nt_run) {
        const int key = nt * 8 + 2 * tg;
        dp[nt][0] = s[nt][0] * (dp[nt][0] - d0);
        dp[nt][1] = s[nt][1] * (dp[nt][1] - d0);
        dp[nt][2] = s[nt][2] * (dp[nt][2] - d1);
        dp[nt][3] = s[nt][3] * (dp[nt][3] - d1);
        if (pd0) {
          if (r0 < p.Lq) {
            if (key < p.Lk) { aw = fmaf(dp[nt][0], (*(pd0 + key)), aw); ab += dp[nt][0]; }
            if (key + 1 < p.Lk) { aw = fmaf(dp[nt][1], (*(pd0 + key + 1)), aw); ab += dp[nt][1]; }
          }
          if (r1 < p.Lq) {
            if (key < p.Lk) { aw = fmaf(dp[nt][2], (*(pd1 + key)), aw); ab += dp[nt][2]; }
            if (key + 1 < p.Lk) { aw = fmaf(dp[nt][3], (*(pd1 + key + 1)), aw); ab += dp[nt][3]; }
          }
        }
        if (drop) {      // dV = (P o mask / (1 - p))^T dO
          const uint32_t e0 = dbase + (uint32_t)r0 * (uint32_t)LkP + (uint32_t)key;
          const uint32_t e1 = dbase + (uint32_t)r1 * (uint32_t)LkP + (uint32_t)key;
          s[nt][0] *= vi_hash32(e0, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
          s[nt][1] *= vi_hash32(e0 + 1, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
          s[nt][2] *= vi_hash32(e1, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
          s[nt][3] *= vi_hash32(e1 + 1, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
        }
        *reinterpret_cast<uint32_t*>(Ps + (size_t)r0 * PP + key) = pack_bf16x2(s[nt][0], s[nt][1]);
        *reinterpret_cast<uint32_t*>(Ps + (size_t)r1 * PP + key) = pack_bf16x2(s[nt][2], s[nt][3]);
        *reinterpret_cast<uint32_t*>(Ss + (size_t)r0 * PP + key) = pack_bf16x2(dp[nt][0], dp[nt][1]);
        *reinterpret_cast<uint32_t*>(Ss + (size_t)r1 * PP + key) = pack_bf16x2(dp[nt][2], dp[nt][3]);
      }
    }
    // dQ = dS K / 8 : dS (accumulator layout) re-packed as the A operand; K^T fragments through ldmatrix.trans
    float dq[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NT / 2; ++kk) {
      if (2 * kk < nt_run) {
        uint32_t sa[4];
        sa[0] = pack_bf16x2(dp[2 * kk][0], dp[2 * kk][1]);
        sa[1] = pack_bf16x2(dp[2 * kk][2], dp[2 * kk][3]);
        sa[2] = pack_bf16x2(dp[2 * kk + 1][0], dp[2 * kk + 1][1]);
        sa[3] = pack_bf16x2(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
#pragma unroll
        for (int d2 = 0; d2 < 4; ++d2) {
          uint32_t kb[4];     // (keys 0-7, d 0-7)^T (keys 8-15, d 0-7)^T (keys 0-7, d 8-15)^T (keys 8-15, d 8-15)^T
          ldsm_x4_trans(kb, ks_u + (uint32_t)((kk * 16 + (lm & 1) * 8 + lr) * ROW + d2 * 16 + (lm >> 1) * 8) * 2);
          mma_16816(dq[2 * d2], sa, kb[0], kb[1]);
          mma_16816(dq[2 * d2 + 1], sa, kb[2], kb[3]);
        }
      }
    }
    bf16* dqg = p.dq + (long long)b * p.Lq * p.lddq + h * DH;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      const int c = dt * 8 + 2 * tg;
      if (r0 < p.Lq) *reinterpret_cast<uint32_t*>(dqg + (long long)r0 * p.lddq + c) = pack_bf16x2(dq[dt][0] * 0.125f, dq[dt][1] * 0.125f);
      if (r1 < p.Lq) *reinterpret_cast<uint32_t*>(dqg + (long long)r1 * p.lddq + c) = pack_bf16x2(dq[dt][2] * 0.125f, dq[dt][3] * 0.125f);
    }
  }
  if (p.pair_dist && p.d_affine) {
    aw = warp_sum(aw);
    ab = warp_sum(ab);
    if (lane == 0) { atomicAdd(p.d_affine, aw); atomicAdd(p.d_affine + 1, ab); }
  }
  __syncthreads();

  // ------------------------------------------------ phase 2: a warp per 16-key tile
  bf16* dkg = p.dk + (long long)b * p.Lk * p.lddk + h * DH;
  bf16* dvg = p.dv + (long long)b * p.Lk * p.lddv + h * DH;
  for (int kt = warp; kt < (LkP >> 4); kt += 4) {
    const int k0 = kt * 16;
    float dv[8][4], dk[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
      dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
    }
    for (int qb = 0; qb < (LqP >> 4); ++qb) {
      // A = P^T / dS^T (m = key, k = query): stored [query][key] -> transposed 8x8 blocks
      uint32_t pa[4], sa[4];
      const uint32_t aoff = (uint32_t)((qb * 16 + (lm >> 1) * 8 + lr) * PP + k0 + (lm & 1) * 8) * 2;
      ldsm_x4_trans(pa, ps_u + aoff);
      ldsm_x4_trans(sa, ss_u + aoff);
#pragma unroll
      for (int d2 = 0; d2 < 4; ++d2) {
        uint32_t ob[4], qb4[4];   // B = dO / Q (k = query, n = d): stored [query][d] -> .trans
        const uint32_t boff = (uint32_t)((qb * 16 + (lm & 1) * 8 + lr) * ROW + d2 * 16 + (lm >> 1) * 8) * 2;
        ldsm_x4_trans(ob, os_u + boff);
        ldsm_x4_trans(qb4, qs_u + boff);
        mma_16816(dv[2 * d2], pa, ob[0], ob[1]);
        mma_16816(dv[2 * d2 + 1], pa, ob[2], ob[3]);
        mma_16816(dk[2 * d2], sa, qb4[0], qb4[1]);
        mma_16816(dk[2 * d2 + 1], sa, qb4[2], qb4[3]);
      }
    }
    const int r0 = k0 + g, r1 = k0 + g + 8;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      const int c = dt * 8 + 2 * tg;
      if (r0 < p.Lk) {
        *reinterpret_cast<uint32_t*>(dvg + (long long)r0 * p.lddv + c) = pack_bf16x2(dv[dt][0], dv[dt][1]);
        *reinterpret_cast<uint32_t*>(dkg + (long long)r0 * p.lddk + c) = pack_bf16x2(dk[dt][0] * 0.125f, dk[dt][1] * 0.125f);
      }
      if (r1 < p.Lk) {
        *reinterpret_cast<uint32_t*>(dvg + (long long)r1 * p.lddv + c) = pack_bf16x2(dv[dt][2], dv[dt][3]);
        *reinterpret_cast<uint32_t*>(dkg + (long long)r1 * p.lddk + c) = pack_bf16x2(dk[dt][2] * 0.125f, dk[dt][3] * 0.125f);
      }
    }
  }
}

template <int NT>
int launch_tc(const AttnBwdTcParams& p, size_t smem, cudaStream_t st) {
  static bool set = false;
  if (!set) {
    VI_CUDA(cudaFuncSetAttribute(attn_bwd_bf16_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    set = true;
  }
  VI_CUDA(vi_launch(attn_bwd_bf16_kernel<NT>, dim3(p.H, p.B), dim3(128), smem, st, p));
  return VI_OK;
}

// ---------------------------------------------------------------------------------------------------------------------------
// Key-blocked form for up to 512 keys (FlashAttention-2 style: the softmax statistics are recomputed, not taken from the forward).
//
//   attn_bwd_dq_kernel   grid (query tiles, H, B), 1..4 warps of 16 queries.  K and V of the head are staged whole (as in the
//                        forward generic kernel); pass 1 walks the 64-key blocks with an online max / sum and D = rowsum(P o dP')
//                        (dP' = dP o mask / (1 - p)), stores (max, 1 / sum, D) per row; pass 2 recomputes S and dP, forms
//                        dS = P o (dP' - D) and accumulates dQ = dS K / 8 in registers.  GASA: d(w), d(b) of the CTA go to a
//                        per-CTA partial.
//   attn_bwd_dkv_kernel  grid (64-key blocks, H, B), 4 warps of 16 keys.  K and V of the block stay in shared memory; the kernel
//                        walks 64-query tiles (Q, dO and the row statistics double-buffered by cp.async) and accumulates
//                        dV = (P o mask / (1 - p))^T dO and dK = dS^T Q / 8 in registers.  Its first CTA adds the GASA partials to
//                        d_affine in a fixed order.
// Every output element has one writer and every sum a fixed order: two calls are bit-identical.  All contractions are mma.sync
// m16n8k16 (bf16 in, fp32 accumulate); P and dS are rounded to bf16 only as MMA operands.  Dropout element ids, threshold and
// scale are the forward generic kernel's, so the masks are rebuilt exactly.
// Resources (nvcc 12.9, -Xptxas -v): attn_bwd_dq_kernel 167 registers, shared memory 2 * LkP * 144 + 2 * qrows * 144 + 4 * LkP + 32
// bytes (164 KB at 512 keys: 1 CTA per SM; 82 KB at 212 keys: 2 per SM); attn_bwd_dkv_kernel 190 registers, 55.8 KB, 2 CTAs per
// SM (register-bound).  No spills, no local memory.
// ---------------------------------------------------------------------------------------------------------------------------
constexpr int KB = 64;             // keys per block of the dK / dV kernel, queries per tile of its walk

// S = Q K^T and dP = dO V^T of a warp's 16 queries against the 16-key pairs [kc, kc + 16 * npairs)
__device__ __forceinline__ void qtile_scores(float (&s)[8][4], float (&dp)[8][4], const uint32_t (&qa)[4][4], const uint32_t (&da)[4][4],
                                             uint32_t ks_u, uint32_t vs_u, int kc, int npairs, int lm, int lr) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
  }
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      if (np < npairs) {
        uint32_t kb[4], vb[4];
        const uint32_t off = (uint32_t)((kc + np * 16 + (lm >> 1) * 8 + lr) * ROW + ks * 16 + (lm & 1) * 8) * 2;
        ldsm_x4(kb, ks_u + off);
        ldsm_x4(vb, vs_u + off);
        mma_16816(s[2 * np], qa[ks], kb[0], kb[1]);
        mma_16816(s[2 * np + 1], qa[ks], kb[2], kb[3]);
        mma_16816(dp[2 * np], da[ks], vb[0], vb[1]);
        mma_16816(dp[2 * np + 1], da[ks], vb[2], vb[3]);
      }
    }
  }
}

// logits of a 64-key chunk: S / 8 + mask (+ w * dist + b), exactly as the forward generic kernel forms them
__device__ __forceinline__ void qtile_logits(float (&s)[8][4], const AttnBwdTcParams& p, const float* madd, const float* pd0,
                                             const float* pd1, float bw, float bb, int kc, int npairs, int tg) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if (nt < 2 * npairs) {
      const int key = kc + nt * 8 + 2 * tg;
      const float2 ma = *reinterpret_cast<const float2*>(madd + key);
      float b00 = 0.f, b01 = 0.f, b10 = 0.f, b11 = 0.f;
      if (pd0) {
        if (key < p.Lk) { b00 = fmaf(bw, pd0[key], bb); b10 = fmaf(bw, pd1[key], bb); }
        if (key + 1 < p.Lk) { b01 = fmaf(bw, pd0[key + 1], bb); b11 = fmaf(bw, pd1[key + 1], bb); }
      }
      s[nt][0] = s[nt][0] * 0.125f + ma.x + b00;
      s[nt][1] = s[nt][1] * 0.125f + ma.y + b01;
      s[nt][2] = s[nt][2] * 0.125f + ma.x + b10;
      s[nt][3] = s[nt][3] * 0.125f + ma.y + b11;
    }
  }
}

__device__ __forceinline__ float drop_factor(const AttnBwdTcParams& p, uint32_t e, uint32_t dkey) {
  return vi_hash32(e, dkey) >= p.drop_thresh ? p.drop_scale : 0.f;
}

__global__ void __launch_bounds__(128) attn_bwd_dq_kernel(const AttnBwdTcParams p) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  const int LkP = p.LkP, nthr = blockDim.x, qrows = (nthr >> 5) * 16;
  const int b = blockIdx.z, h = blockIdx.y, q_base = blockIdx.x * qrows;
  bf16* Ks = reinterpret_cast<bf16*>(smem);                  // [LkP][72]
  bf16* Vs = Ks + (size_t)LkP * ROW;                         // [LkP][72]
  bf16* Qs = Vs + (size_t)LkP * ROW;                         // [qrows][72]
  bf16* Os = Qs + (size_t)qrows * ROW;                       // [qrows][72]   dO
  float* madd = reinterpret_cast<float*>(Os + (size_t)qrows * ROW);   // [LkP]
  float* red = madd + LkP;                                   // [4][2] GASA partials of the warps
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const bf16* kg = p.k + (long long)b * p.Lk * p.ldk + h * DH;
  const bf16* vg = p.v + (long long)b * p.Lk * p.ldv + h * DH;
  const bf16* qg = p.q + ((long long)b * p.Lq + q_base) * p.ldq + h * DH;
  const bf16* og = p.dout + ((long long)b * p.Lq + q_base) * p.ldo + h * DH;
  const uint32_t ks_u = smem_u32(Ks), vs_u = smem_u32(Vs), qs_u = smem_u32(Qs), os_u = smem_u32(Os);
  for (int e = tid; e < LkP * 8; e += nthr) {
    const int key = e >> 3, ch = e & 7;
    const bool ok = key < p.Lk;
    const int kk = ok ? key : 0;
    cp_async16(ks_u + (uint32_t)(key * ROW + ch * 8) * 2, kg + (long long)kk * p.ldk + ch * 8, ok);
    cp_async16(vs_u + (uint32_t)(key * ROW + ch * 8) * 2, vg + (long long)kk * p.ldv + ch * 8, ok);
  }
  for (int e = tid; e < qrows * 8; e += nthr) {
    const int r = e >> 3, ch = e & 7;
    const bool ok = q_base + r < p.Lq;
    const int rr = ok ? r : 0;
    cp_async16(qs_u + (uint32_t)(r * ROW + ch * 8) * 2, qg + (long long)rr * p.ldq + ch * 8, ok);
    cp_async16(os_u + (uint32_t)(r * ROW + ch * 8) * 2, og + (long long)rr * p.ldo + ch * 8, ok);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (int key = tid; key < LkP; key += nthr) {
    float m = 0.f;
    if (key >= p.Lk) m = -INFINITY;
    else if (p.key_mask && !p.key_mask[(long long)b * p.Lk + key]) m = (p.mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f;
    madd[key] = m;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const int g = lane >> 2, tg = lane & 3;
  const int lm = lane >> 3, lr = lane & 7;
  const int q0 = q_base + warp * 16, r0 = q0 + g, r1 = q0 + g + 8;
  float aw = 0.f, ab = 0.f;                                  // GASA affine gradients of this thread
  if (q0 < p.Lq) {
    uint32_t qa[4][4], da[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t off = (uint32_t)((warp * 16 + (lm & 1) * 8 + lr) * ROW + (lm >> 1) * 8 + ks * 16) * 2;
      ldsm_x4(qa[ks], qs_u + off);
      ldsm_x4(da[ks], os_u + off);
    }
    float bw = 0.f, bb = 0.f;
    const float* pd0 = nullptr;
    const float* pd1 = nullptr;
    if (p.pair_dist) {
      bw = p.bias_affine[0];
      bb = p.bias_affine[1];
      pd0 = p.pair_dist + ((long long)b * p.Lq + (r0 < p.Lq ? r0 : 0)) * p.Lk;
      pd1 = p.pair_dist + ((long long)b * p.Lq + (r1 < p.Lq ? r1 : 0)) * p.Lk;
    }
    const bool drop = p.drop_thresh != 0;
    const uint32_t dkey = drop ? vi_drop_key(p.drop_seed, p.drop_site) : 0u;
    const uint32_t dbase = (uint32_t)((b * p.H + h) * p.Lq) * (uint32_t)LkP;
    const uint32_t e0r = dbase + (uint32_t)r0 * (uint32_t)LkP, e1r = dbase + (uint32_t)r1 * (uint32_t)LkP;

    // ---- pass 1: row max, sum and D = sum_k P dP' with online rescaling
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f, d0 = 0.f, d1 = 0.f;
    for (int kc = 0; kc < LkP; kc += 64) {
      const int npairs = min(4, (LkP - kc) >> 4);
      float s[8][4], dp[8][4];
      qtile_scores(s, dp, qa, da, ks_u, vs_u, kc, npairs, lm, lr);
      qtile_logits(s, p, madd, pd0, pd1, bw, bb, kc, npairs, tg);
      float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        if (nt < 2 * npairs) {
          cm0 = fmaxf(cm0, fmaxf(s[nt][0], s[nt][1]));
          cm1 = fmaxf(cm1, fmaxf(s[nt][2], s[nt][3]));
        }
      }
      cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1));
      cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
      cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1));
      cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
      const float mn0 = fmaxf(m0, cm0), mn1 = fmaxf(m1, cm1);
      const float mu0 = (mn0 == -INFINITY) ? 0.f : mn0, mu1 = (mn1 == -INFINITY) ? 0.f : mn1;
      const float sc0 = (m0 == -INFINITY) ? 0.f : __expf(m0 - mu0), sc1 = (m1 == -INFINITY) ? 0.f : __expf(m1 - mu1);
      l0 *= sc0; d0 *= sc0; l1 *= sc1; d1 *= sc1;
      m0 = mn0; m1 = mn1;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        if (nt < 2 * npairs) {
          const uint32_t key = (uint32_t)(kc + nt * 8 + 2 * tg);
          const float e00 = __expf(s[nt][0] - mu0), e01 = __expf(s[nt][1] - mu0);
          const float e10 = __expf(s[nt][2] - mu1), e11 = __expf(s[nt][3] - mu1);
          if (drop) {
            dp[nt][0] *= drop_factor(p, e0r + key, dkey);
            dp[nt][1] *= drop_factor(p, e0r + key + 1, dkey);
            dp[nt][2] *= drop_factor(p, e1r + key, dkey);
            dp[nt][3] *= drop_factor(p, e1r + key + 1, dkey);
          }
          l0 += e00 + e01;
          l1 += e10 + e11;
          d0 = fmaf(e00, dp[nt][0], fmaf(e01, dp[nt][1], d0));
          d1 = fmaf(e10, dp[nt][2], fmaf(e11, dp[nt][3], d1));
        }
      }
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    d0 += __shfl_xor_sync(0xffffffffu, d0, 1);
    d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 1);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    const float mu0 = (m0 == -INFINITY) ? 0.f : m0, mu1 = (m1 == -INFINITY) ? 0.f : m1;
    const float i0 = l0 > 0.f ? 1.0f / l0 : 0.f, i1 = l1 > 0.f ? 1.0f / l1 : 0.f;
    d0 *= i0;
    d1 *= i1;
    if (tg == 0) {
      const long long R = (long long)p.B * p.H * p.LqP, row = (long long)(b * p.H + h) * p.LqP;
      if (r0 < p.Lq) { p.stats[row + r0] = mu0; p.stats[R + row + r0] = i0; p.stats[2 * R + row + r0] = d0; }
      if (r1 < p.Lq) { p.stats[row + r1] = mu1; p.stats[R + row + r1] = i1; p.stats[2 * R + row + r1] = d1; }
    }

    // ---- pass 2: dS = P o (dP' - D), dQ = dS K / 8
    float dq[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
    for (int kc = 0; kc < LkP; kc += 64) {
      const int npairs = min(4, (LkP - kc) >> 4);
      float s[8][4], dp[8][4];
      qtile_scores(s, dp, qa, da, ks_u, vs_u, kc, npairs, lm, lr);
      qtile_logits(s, p, madd, pd0, pd1, bw, bb, kc, npairs, tg);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        if (nt < 2 * npairs) {
          const int key = kc + nt * 8 + 2 * tg;
          if (drop) {
            dp[nt][0] *= drop_factor(p, e0r + (uint32_t)key, dkey);
            dp[nt][1] *= drop_factor(p, e0r + (uint32_t)key + 1, dkey);
            dp[nt][2] *= drop_factor(p, e1r + (uint32_t)key, dkey);
            dp[nt][3] *= drop_factor(p, e1r + (uint32_t)key + 1, dkey);
          }
          dp[nt][0] = __expf(s[nt][0] - mu0) * i0 * (dp[nt][0] - d0);
          dp[nt][1] = __expf(s[nt][1] - mu0) * i0 * (dp[nt][1] - d0);
          dp[nt][2] = __expf(s[nt][2] - mu1) * i1 * (dp[nt][2] - d1);
          dp[nt][3] = __expf(s[nt][3] - mu1) * i1 * (dp[nt][3] - d1);
          if (pd0) {
            if (r0 < p.Lq) {
              if (key < p.Lk) { aw = fmaf(dp[nt][0], pd0[key], aw); ab += dp[nt][0]; }
              if (key + 1 < p.Lk) { aw = fmaf(dp[nt][1], pd0[key + 1], aw); ab += dp[nt][1]; }
            }
            if (r1 < p.Lq) {
              if (key < p.Lk) { aw = fmaf(dp[nt][2], pd1[key], aw); ab += dp[nt][2]; }
              if (key + 1 < p.Lk) { aw = fmaf(dp[nt][3], pd1[key + 1], aw); ab += dp[nt][3]; }
            }
          }
        }
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        if (kk < npairs) {
          uint32_t sa[4];
          sa[0] = pack_bf16x2(dp[2 * kk][0], dp[2 * kk][1]);
          sa[1] = pack_bf16x2(dp[2 * kk][2], dp[2 * kk][3]);
          sa[2] = pack_bf16x2(dp[2 * kk + 1][0], dp[2 * kk + 1][1]);
          sa[3] = pack_bf16x2(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
#pragma unroll
          for (int d2 = 0; d2 < 4; ++d2) {
            uint32_t kb[4];
            ldsm_x4_trans(kb, ks_u + (uint32_t)((kc + kk * 16 + (lm & 1) * 8 + lr) * ROW + d2 * 16 + (lm >> 1) * 8) * 2);
            mma_16816(dq[2 * d2], sa, kb[0], kb[1]);
            mma_16816(dq[2 * d2 + 1], sa, kb[2], kb[3]);
          }
        }
      }
    }
    bf16* dqg = p.dq + (long long)b * p.Lq * p.lddq + h * DH;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      const int c = dt * 8 + 2 * tg;
      if (r0 < p.Lq) *reinterpret_cast<uint32_t*>(dqg + (long long)r0 * p.lddq + c) = pack_bf16x2(dq[dt][0] * 0.125f, dq[dt][1] * 0.125f);
      if (r1 < p.Lq) *reinterpret_cast<uint32_t*>(dqg + (long long)r1 * p.lddq + c) = pack_bf16x2(dq[dt][2] * 0.125f, dq[dt][3] * 0.125f);
    }
  }
  if (p.pair_dist && p.d_affine) {                           // this CTA's GASA partial, summed in a fixed order
    aw = warp_sum(aw);
    ab = warp_sum(ab);
    if (lane == 0) { red[2 * warp] = aw; red[2 * warp + 1] = ab; }
    __syncthreads();
    if (tid == 0) {
      float sw = 0.f, sb = 0.f;
      for (int w = 0; w < (nthr >> 5); ++w) { sw += red[2 * w]; sb += red[2 * w + 1]; }
      const int cta = (b * p.H + h) * gridDim.x + blockIdx.x;
      p.aff_part[2 * cta] = sw;
      p.aff_part[2 * cta + 1] = sb;
    }
  }
}

__global__ void __launch_bounds__(128) attn_bwd_dkv_kernel(const AttnBwdTcParams p) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  bf16* Ks = reinterpret_cast<bf16*>(smem);                  // [64][72]
  bf16* Vs = Ks + KB * ROW;                                  // [64][72]
  bf16* Qs = Vs + KB * ROW;                                  // [2][64][72]
  bf16* Os = Qs + 2 * KB * ROW;                              // [2][64][72]   dO
  float* st = reinterpret_cast<float*>(Os + 2 * KB * ROW);   // [2][3][64]    max, 1 / sum, D of the tile's rows
  float* madd = st + 2 * 3 * KB;                             // [64]
  const int b = blockIdx.z, h = blockIdx.y, k_base = blockIdx.x * KB;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (p.pair_dist && p.d_affine && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && warp == 0) {
    float sw = 0.f, sb = 0.f;                                // the dQ kernel's partials, fixed order
    for (int i = lane; i < p.n_aff; i += 32) { sw += p.aff_part[2 * i]; sb += p.aff_part[2 * i + 1]; }
    sw = warp_sum(sw);
    sb = warp_sum(sb);
    if (lane == 0) { p.d_affine[0] += sw; p.d_affine[1] += sb; }
  }

  const bf16* kg = p.k + (long long)b * p.Lk * p.ldk + h * DH;
  const bf16* vg = p.v + (long long)b * p.Lk * p.ldv + h * DH;
  const bf16* qg = p.q + (long long)b * p.Lq * p.ldq + h * DH;
  const bf16* og = p.dout + (long long)b * p.Lq * p.ldo + h * DH;
  const long long R = (long long)p.B * p.H * p.LqP;
  const float* stg = p.stats + (long long)(b * p.H + h) * p.LqP;
  const uint32_t ks_u = smem_u32(Ks), vs_u = smem_u32(Vs), qs_u = smem_u32(Qs), os_u = smem_u32(Os), st_u = smem_u32(st);
  for (int e = tid; e < KB * 8; e += 128) {
    const int key = e >> 3, ch = e & 7;
    const bool ok = k_base + key < p.Lk;
    const int kk = ok ? k_base + key : 0;
    cp_async16(ks_u + (uint32_t)(key * ROW + ch * 8) * 2, kg + (long long)kk * p.ldk + ch * 8, ok);
    cp_async16(vs_u + (uint32_t)(key * ROW + ch * 8) * 2, vg + (long long)kk * p.ldv + ch * 8, ok);
  }
  auto load_tile = [&](int t, int buf) {                     // Q, dO and the statistics of query tile t
    const int qb = t * KB;
    for (int e = tid; e < KB * 8; e += 128) {
      const int r = e >> 3, ch = e & 7;
      const bool ok = qb + r < p.Lq;
      const int rr = ok ? qb + r : 0;
      const uint32_t so = (uint32_t)((buf * KB + r) * ROW + ch * 8) * 2;
      cp_async16(qs_u + so, qg + (long long)rr * p.ldq + ch * 8, ok);
      cp_async16(os_u + so, og + (long long)rr * p.ldo + ch * 8, ok);
    }
    if (tid < 3 * (KB / 4)) {
      const int arr = tid / (KB / 4), c = (tid % (KB / 4)) * 4;
      const bool ok = qb + c < p.LqP;
      cp_async16(st_u + (uint32_t)((buf * 3 + arr) * KB + c) * 4, stg + arr * R + (ok ? qb + c : 0), ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  load_tile(0, 0);
  if (tid < KB) {
    const int key = k_base + tid;
    float m = 0.f;
    if (key >= p.Lk) m = -INFINITY;
    else if (p.key_mask && !p.key_mask[(long long)b * p.Lk + key]) m = (p.mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f;
    madd[tid] = m;
  }

  const int g = lane >> 2, tg = lane & 3;
  const int lm = lane >> 3, lr = lane & 7;
  const int kl = warp * 16;                                  // this warp's first key in the block
  const bool active = k_base + kl < p.LkP;
  const int kr0 = k_base + kl + g, kr1 = kr0 + 8;
  float bw = 0.f, bb = 0.f;
  if (p.pair_dist) { bw = p.bias_affine[0]; bb = p.bias_affine[1]; }
  const bool drop = p.drop_thresh != 0;
  const uint32_t dkey = drop ? vi_drop_key(p.drop_seed, p.drop_site) : 0u;
  const uint32_t dbase = (uint32_t)((b * p.H + h) * p.Lq) * (uint32_t)p.LkP;
  float dv[8][4], dk[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
    dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
  }
  const int nqt = (p.Lq + KB - 1) / KB;
  for (int t = 0; t < nqt; ++t) {
    const int buf = t & 1;
    if (t + 1 < nqt) {
      load_tile(t + 1, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    if (active) {
      const uint32_t qs_b = qs_u + (uint32_t)(buf * KB * ROW) * 2, os_b = os_u + (uint32_t)(buf * KB * ROW) * 2;
      const float* sm_ = st + buf * 3 * KB;
      // S^T = K Q^T and dP^T = V dO^T: keys are the MMA rows, the tile's 64 queries the columns
      float s[8][4], dp[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
      }
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t ka[4], va[4];
        const uint32_t aoff = (uint32_t)((kl + (lm & 1) * 8 + lr) * ROW + (lm >> 1) * 8 + ks * 16) * 2;
        ldsm_x4(ka, ks_u + aoff);
        ldsm_x4(va, vs_u + aoff);
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          uint32_t qb4[4], ob[4];
          const uint32_t boff = (uint32_t)((np * 16 + (lm >> 1) * 8 + lr) * ROW + ks * 16 + (lm & 1) * 8) * 2;
          ldsm_x4(qb4, qs_b + boff);
          ldsm_x4(ob, os_b + boff);
          mma_16816(s[2 * np], ka, qb4[0], qb4[1]);
          mma_16816(s[2 * np + 1], ka, qb4[2], qb4[3]);
          mma_16816(dp[2 * np], va, ob[0], ob[1]);
          mma_16816(dp[2 * np + 1], va, ob[2], ob[3]);
        }
      }
      const float ma0 = madd[kl + g], ma1 = madd[kl + g + 8];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {                        // query column of c[j] (key kr0) and c[2 + j] (key kr1)
          const int lq = nt * 8 + 2 * tg + j, q = t * KB + lq;
          const bool qok = q < p.Lq;
          const float mq = qok ? sm_[lq] : INFINITY, iq = qok ? sm_[KB + lq] : 0.f, dd = qok ? sm_[2 * KB + lq] : 0.f;
          float b0 = 0.f, b1 = 0.f;
          if (p.pair_dist && qok) {
            const float* pd = p.pair_dist + ((long long)b * p.Lq + q) * p.Lk;
            if (kr0 < p.Lk) b0 = fmaf(bw, pd[kr0], bb);
            if (kr1 < p.Lk) b1 = fmaf(bw, pd[kr1], bb);
          }
          const float p0 = __expf(s[nt][j] * 0.125f + ma0 + b0 - mq) * iq;
          const float p1 = __expf(s[nt][2 + j] * 0.125f + ma1 + b1 - mq) * iq;
          float f0 = 1.f, f1 = 1.f;
          if (drop && qok) {
            const uint32_t eq = dbase + (uint32_t)q * (uint32_t)p.LkP;
            f0 = drop_factor(p, eq + (uint32_t)kr0, dkey);
            f1 = drop_factor(p, eq + (uint32_t)kr1, dkey);
          }
          dp[nt][j] = p0 * (dp[nt][j] * f0 - dd);
          dp[nt][2 + j] = p1 * (dp[nt][2 + j] * f1 - dd);
          s[nt][j] = p0 * f0;
          s[nt][2 + j] = p1 * f1;
        }
      }
      // dV += (P o mask / (1 - p))^T dO,  dK += dS^T Q: the accumulators re-packed as A operands, dO / Q through ldmatrix.trans
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t pa[4], sa[4];
        pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        sa[0] = pack_bf16x2(dp[2 * kk][0], dp[2 * kk][1]);
        sa[1] = pack_bf16x2(dp[2 * kk][2], dp[2 * kk][3]);
        sa[2] = pack_bf16x2(dp[2 * kk + 1][0], dp[2 * kk + 1][1]);
        sa[3] = pack_bf16x2(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
#pragma unroll
        for (int d2 = 0; d2 < 4; ++d2) {
          uint32_t ob[4], qb4[4];
          const uint32_t boff = (uint32_t)((kk * 16 + (lm & 1) * 8 + lr) * ROW + d2 * 16 + (lm >> 1) * 8) * 2;
          ldsm_x4_trans(ob, os_b + boff);
          ldsm_x4_trans(qb4, qs_b + boff);
          mma_16816(dv[2 * d2], pa, ob[0], ob[1]);
          mma_16816(dv[2 * d2 + 1], pa, ob[2], ob[3]);
          mma_16816(dk[2 * d2], sa, qb4[0], qb4[1]);
          mma_16816(dk[2 * d2 + 1], sa, qb4[2], qb4[3]);
        }
      }
    }
    __syncthreads();                                         // the next iteration's copy overwrites this buffer
  }
  if (!active) return;
  bf16* dkg = p.dk + (long long)b * p.Lk * p.lddk + h * DH;
  bf16* dvg = p.dv + (long long)b * p.Lk * p.lddv + h * DH;
#pragma unroll
  for (int dt = 0; dt < 8; ++dt) {
    const int c = dt * 8 + 2 * tg;
    if (kr0 < p.Lk) {
      *reinterpret_cast<uint32_t*>(dvg + (long long)kr0 * p.lddv + c) = pack_bf16x2(dv[dt][0], dv[dt][1]);
      *reinterpret_cast<uint32_t*>(dkg + (long long)kr0 * p.lddk + c) = pack_bf16x2(dk[dt][0] * 0.125f, dk[dt][1] * 0.125f);
    }
    if (kr1 < p.Lk) {
      *reinterpret_cast<uint32_t*>(dvg + (long long)kr1 * p.lddv + c) = pack_bf16x2(dv[dt][2], dv[dt][3]);
      *reinterpret_cast<uint32_t*>(dkg + (long long)kr1 * p.lddk + c) = pack_bf16x2(dk[dt][2] * 0.125f, dk[dt][3] * 0.125f);
    }
  }
}

int long_q_warps(int Lq) { return Lq >= 64 ? 4 : (Lq + 15) / 16; }

}  // namespace

// per device (vi_init): the dynamic shared memory the key-blocked kernels may ask for (164 KB at 512 keys)
int vi_attn_bwd_init() {
  VI_CUDA(cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  VI_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  return VI_OK;
}

// fp32 workspace of the key-blocked kernels: the row statistics [3][B * H][LqP] and the dQ kernel's GASA partials
int64_t vi_attn_bwd_long_floats(int B, int H, int Lq) {
  const int64_t LqP = (Lq + 15) & ~15, qrows = 16 * long_q_warps(Lq);
  return 3 * (int64_t)B * H * LqP + 2 * (int64_t)B * H * ((Lq + qrows - 1) / qrows);
}

// bf16 problems the single-CTA kernel does not take (more than 128 keys, more than 256 queries), up to 512 keys
int vi_attn_bwd_long(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* dout,
                     int64_t ldo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                     const uint8_t* key_mask, const float* pair_dist, const float* bias_affine, float* d_affine, int B, int H,
                     int Lq, int Lk, int mask_mode, float drop_p, uint32_t drop_site, const uint32_t* drop_seed, float* workspace,
                     int64_t workspace_floats, cudaStream_t st) {
  const int LqP = (Lq + 15) & ~15, LkP = (Lk + 15) & ~15;
  const uintptr_t al = (uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)dout;
  VI_CHECK_ARG(!(al & 15) && ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0,
               "vi_attn_bwd: bf16 q / k / v / dout must be 16-byte aligned with leading dimensions multiple of 8");
  VI_CHECK_ARG(!(((uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 3) && lddq % 2 == 0 && lddk % 2 == 0 && lddv % 2 == 0,
               "vi_attn_bwd: bf16 dq / dk / dv must be 4-byte aligned with even leading dimensions");
  const int64_t need = vi_attn_bwd_long_floats(B, H, Lq);
  VI_CHECK_ARG(workspace && workspace_floats >= need && ((uintptr_t)workspace & 15) == 0,
               "vi_attn_bwd: the workspace has %lld floats (16-byte aligned) where %lld are needed (vi_attn_bwd_workspace)",
               (long long)(workspace ? workspace_floats : 0), (long long)need);
  const int nwarp = long_q_warps(Lq), qrows = 16 * nwarp, nqt = (Lq + qrows - 1) / qrows;
  AttnBwdTcParams p;
  p.q = reinterpret_cast<const bf16*>(q); p.ldq = ldq; p.k = reinterpret_cast<const bf16*>(k); p.ldk = ldk;
  p.v = reinterpret_cast<const bf16*>(v); p.ldv = ldv; p.dout = reinterpret_cast<const bf16*>(dout); p.ldo = ldo;
  p.dq = reinterpret_cast<bf16*>(dq); p.lddq = lddq; p.dk = reinterpret_cast<bf16*>(dk); p.lddk = lddk;
  p.dv = reinterpret_cast<bf16*>(dv); p.lddv = lddv;
  p.key_mask = key_mask; p.pair_dist = pair_dist; p.bias_affine = bias_affine; p.d_affine = d_affine;
  p.B = B; p.H = H; p.Lq = Lq; p.Lk = Lk; p.LqP = LqP; p.LkP = LkP; p.mask_mode = mask_mode;
  p.drop_thresh = drop_p > 0.f ? vi_drop_threshold(drop_p) : 0u;
  if (drop_p > 0.f && p.drop_thresh == 0u) p.drop_thresh = 1u;
  p.drop_scale = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
  p.drop_site = drop_site; p.drop_seed = drop_seed;
  p.stats = workspace;
  p.aff_part = workspace + 3 * (int64_t)B * H * LqP;
  p.n_aff = B * H * nqt;
  const size_t smem_q = (size_t)(2 * LkP + 2 * qrows) * ROW * 2 + (size_t)LkP * 4 + 8 * 4;
  const size_t smem_kv = (size_t)6 * KB * ROW * 2 + (size_t)(2 * 3 * KB + KB) * 4;
  VI_CUDA(vi_launch(attn_bwd_dq_kernel, dim3(nqt, H, B), dim3(32 * nwarp), smem_q, st, p));
  VI_CUDA(vi_launch(attn_bwd_dkv_kernel, dim3((LkP + KB - 1) / KB, H, B), dim3(128), smem_kv, st, p));
  return VI_OK;
}

// Returns VI_OK after launching, or 1 when the problem does not fit the single-CTA kernel (the caller then uses the
// key-blocked kernels, vi_attn_bwd_long).
int vi_attn_bwd_tc(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* dout,
                   int64_t ldo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                   const uint8_t* key_mask, const float* pair_dist, const float* bias_affine, float* d_affine, int B, int H,
                   int Lq, int Lk, int mask_mode, float drop_p, uint32_t drop_site, const uint32_t* drop_seed, cudaStream_t st) {
  const int LqP = (Lq + 15) & ~15, LkP = (Lk + 15) & ~15;
  if (LkP > 128 || LqP > 256) return 1;
  const uintptr_t al = (uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)dout;
  if ((al & 15) || (ldq % 8) || (ldk % 8) || (ldv % 8) || (ldo % 8)) return 1;
  if ((((uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 3) || (lddq % 2) || (lddk % 2) || (lddv % 2)) return 1;
  const size_t smem = ((size_t)(2 * LkP + 2 * LqP) * ROW + (size_t)2 * LqP * (LkP + 8)) * 2 + (size_t)LkP * 4;
  if (smem > 200 * 1024) return 1;
  AttnBwdTcParams p;
  p.q = reinterpret_cast<const bf16*>(q); p.ldq = ldq; p.k = reinterpret_cast<const bf16*>(k); p.ldk = ldk;
  p.v = reinterpret_cast<const bf16*>(v); p.ldv = ldv; p.dout = reinterpret_cast<const bf16*>(dout); p.ldo = ldo;
  p.dq = reinterpret_cast<bf16*>(dq); p.lddq = lddq; p.dk = reinterpret_cast<bf16*>(dk); p.lddk = lddk;
  p.dv = reinterpret_cast<bf16*>(dv); p.lddv = lddv;
  p.key_mask = key_mask; p.pair_dist = pair_dist; p.bias_affine = bias_affine; p.d_affine = d_affine;
  p.B = B; p.H = H; p.Lq = Lq; p.Lk = Lk; p.LqP = LqP; p.LkP = LkP; p.mask_mode = mask_mode;
  p.drop_thresh = drop_p > 0.f ? vi_drop_threshold(drop_p) : 0u;
  if (drop_p > 0.f && p.drop_thresh == 0u) p.drop_thresh = 1u;
  p.drop_scale = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
  p.drop_site = drop_site; p.drop_seed = drop_seed;
  if (LkP <= 48) return launch_tc<6>(p, smem, st);
  if (LkP <= 96) return launch_tc<12>(p, smem, st);
  return launch_tc<16>(p, smem, st);
}
