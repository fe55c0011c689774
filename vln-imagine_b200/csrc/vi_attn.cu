// vi_attn.cu - fused masked multi-head attention for the navigation step (scores never reach HBM).
//
//   O = softmax(Q K^T / sqrt(64) + key_padding + (w * pair_dist + b)) V        per (episode, head)
//
// Sequence lengths on this path are tiny (<= 37 queries x <= 85 keys at cfg-2, <= 212 at cfg-5;
// SURVEY.md section 5), so a whole K/V head fits one CTA's shared memory and attention is ~1.7% of the
// step's FLOPs: the bf16 kernel uses warp-level mma.sync m16n8k16 tiles (a 16-query tile per
// warp) with an fp32 online softmax rather than 128-row tcgen05 tiles that would be >70% padding.
// The fp32 kernel is the check mode.
//
// Reference: BertSelfAttention / BertOutAttention (VLN-DUET/map_nav_src/models/vilmodel.py:118-134,
// 336-349), GASA bias (:392-394, :1145-1149), nn.MultiheadAttention with key_padding_mask
// (models/transformer.py:176-177).
#include "vi_common.cuh"

namespace {

// one attention problem = one token stream; a launch runs up to VI_ATTN_MAX_PROBLEMS of them so that the
// streams of a row-stacked activation (DUET global|local, HAMT language|vision) share one kernel launch
struct AttnProblem {
  const void* q; long long ldq;
  const void* k; long long ldk;
  const void* v; long long ldv;
  void* o; long long ldo;
  const uint8_t* key_mask;
  const float* pair_dist;
  const float* bias_affine;
  float* lse;
  int B, Lq, Lk, LkP;
  uint32_t drop_thresh;      // attention-probability dropout (training): 0 = none
  float drop_scale;
  uint32_t drop_site;
  const uint32_t* drop_seed;
};
struct AttnParams {
  AttnProblem pr[VI_ATTN_MAX_PROBLEMS];
  int n_problems, H, mask_mode;
};

constexpr int DH = 64;
constexpr int ROW = 72;            // bf16 elements per staged row (64 + 8): 144-byte pitch keeps ldmatrix conflict-free

template <bool F16>
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (F16) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  } else {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
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
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// exp(x) as one MUFU.EX2: ex2.approx.ftz skips the denormal range fix-up that __expf's ex2.approx carries (results below
// 2^-126 flush to zero, which a softmax numerator cannot tell from the 1e-38 it would otherwise be)
__device__ __forceinline__ float fast_exp(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// grid (q-tiles, H, sum of B over problems), 32..128 threads (one warp per 16 queries of the longest stream, so that
// no warp of a CTA idles on registers another CTA could use): warp w owns query rows [qrows*bx + 16w, +16).
// K, V (whole head) and the Q tile are staged with cp.async; fragments come from ldmatrix (V through .trans, so no
// explicit transpose); scores stay in registers with an fp32 online softmax over 64-key chunks.
// F16: the 16-bit operands / output are fp16 (inference on range-bounded tensors) instead of bf16.
template <bool F16>
__global__ void __launch_bounds__(128, 5) attn_fwd_bf16_kernel(const AttnParams p) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  int z = blockIdx.z, pi = 0;
  while (pi < p.n_problems - 1 && z >= p.pr[pi].B) { z -= p.pr[pi].B; ++pi; }
  const AttnProblem& pr = p.pr[pi];
  const int nthr = blockDim.x, qrows = (blockDim.x >> 5) * 16;      // 1..4 warps: a 16-query tile each
  const int q_base = blockIdx.x * qrows;
  if (q_base >= pr.Lq) return;
  const int b = z, h = blockIdx.y;
  const int LkP = pr.LkP;
  bf16* Ks = reinterpret_cast<bf16*>(smem);                 // [LkP][72]
  bf16* Vs = Ks + (size_t)LkP * ROW;                        // [LkP][72]
  bf16* Qs = Vs + (size_t)LkP * ROW;                        // [qrows][72]
  float* madd = reinterpret_cast<float*>(Qs + qrows * ROW); // [LkP]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const bf16* kg = reinterpret_cast<const bf16*>(pr.k) + (long long)b * pr.Lk * pr.ldk + h * DH;
  const bf16* vg = reinterpret_cast<const bf16*>(pr.v) + (long long)b * pr.Lk * pr.ldv + h * DH;
  const bf16* qg = reinterpret_cast<const bf16*>(pr.q) + (long long)b * pr.Lq * pr.ldq + h * DH;
  const uint32_t ks_u = smem_u32(Ks), vs_u = smem_u32(Vs), qs_u = smem_u32(Qs);
  // two cp.async groups: Q + the first 64 keys, then the remaining keys, so the first score chunk can start
  // while the tail of K / V is still in flight
  const int first = LkP < 64 ? LkP : 64;
  for (int e = tid; e < qrows * 8; e += nthr) {
    const int r = e >> 3, ch = e & 7;
    const bool ok = q_base + r < pr.Lq;
    const int rr = ok ? q_base + r : 0;
    cp_async16(qs_u + (uint32_t)(r * ROW + ch * 8) * 2, qg + (long long)rr * pr.ldq + ch * 8, ok);
  }
  for (int e = tid; e < first * 8; e += nthr) {
    const int key = e >> 3, ch = e & 7;
    const bool ok = key < pr.Lk;
    const int kk = ok ? key : 0;
    cp_async16(ks_u + (uint32_t)(key * ROW + ch * 8) * 2, kg + (long long)kk * pr.ldk + ch * 8, ok);
    cp_async16(vs_u + (uint32_t)(key * ROW + ch * 8) * 2, vg + (long long)kk * pr.ldv + ch * 8, ok);
  }
  cp_async_commit();
  for (int e = first * 8 + tid; e < LkP * 8; e += nthr) {
    const int key = e >> 3, ch = e & 7;
    const bool ok = key < pr.Lk;
    const int kk = ok ? key : 0;
    cp_async16(ks_u + (uint32_t)(key * ROW + ch * 8) * 2, kg + (long long)kk * pr.ldk + ch * 8, ok);
    cp_async16(vs_u + (uint32_t)(key * ROW + ch * 8) * 2, vg + (long long)kk * pr.ldv + ch * 8, ok);
  }
  cp_async_commit();
  for (int key = tid; key < LkP; key += nthr) {
    float m = 0.f;
    if (key >= pr.Lk) m = -INFINITY;
    else if (pr.key_mask && !pr.key_mask[(long long)b * pr.Lk + key]) m = (p.mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f;
    madd[key] = m;
  }
  cp_async_wait<1>();
  __syncthreads();

  const int q0 = q_base + warp * 16;
  if (q0 >= pr.Lq) {                                  // idle warp: still takes part in the second barrier
    if (LkP > 64) { cp_async_wait<0>(); __syncthreads(); }
    return;
  }
  const int g = lane >> 2, tg = lane & 3;
  const int r0 = q0 + g, r1 = q0 + g + 8;
  const int lm = lane >> 3, lr = lane & 7;          // ldmatrix: this lane addresses row lr of matrix lm

  const uint32_t q_frag = qs_u + (uint32_t)((warp * 16 + (lm & 1) * 8 + lr) * ROW + (lm >> 1) * 8) * 2;

  float bw = 0.f, bb = 0.f;
  const float* pd0 = nullptr;
  const float* pd1 = nullptr;
  if (pr.pair_dist) {
    bw = pr.bias_affine[0];
    bb = pr.bias_affine[1];
    pd0 = pr.pair_dist + ((long long)b * pr.Lq + (r0 < pr.Lq ? r0 : 0)) * pr.Lk;
    pd1 = pr.pair_dist + ((long long)b * pr.Lq + (r1 < pr.Lq ? r1 : 0)) * pr.Lk;
  }

  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  const bool drop = pr.drop_thresh != 0;
  const uint32_t dkey = drop ? vi_drop_key(pr.drop_seed, pr.drop_site) : 0u;
  const uint32_t dbase = (uint32_t)((b * p.H + h) * pr.Lq) * (uint32_t)LkP;     // element id = dbase + q * LkP + key

  for (int kc = 0; kc < LkP; kc += 64) {
    if (kc == 64) {                                   // (block-uniform) the second cp.async group is needed from here
      cp_async_wait<0>();
      __syncthreads();
    }
    const int npairs = min(4, (LkP - kc) >> 4);       // 16-key blocks in this chunk (LkP % 16 == 0)
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t qa[4];
      ldsm_x4(qa, q_frag + (uint32_t)(ks * 32));
#pragma unroll
      for (int np = 0; np < 4; ++np) {
        if (np < npairs) {
          uint32_t kb[4];     // (keys 0-7, d 0-7) (keys 0-7, d 8-15) (keys 8-15, d 0-7) (keys 8-15, d 8-15)
          ldsm_x4(kb, ks_u + (uint32_t)((kc + np * 16 + (lm >> 1) * 8 + lr) * ROW + ks * 16 + (lm & 1) * 8) * 2);
          mma_16816<F16>(s[2 * np], qa, kb[0], kb[1]);
          mma_16816<F16>(s[2 * np + 1], qa, kb[2], kb[3]);
        }
      }
    }
    // scale, mask, bias; chunk row max
    float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt < 2 * npairs) {
        const int key = kc + nt * 8 + 2 * tg;
        const float2 ma = *reinterpret_cast<const float2*>(madd + key);
        float b00 = 0.f, b01 = 0.f, b10 = 0.f, b11 = 0.f;
        if (pd0) {
          if (key < pr.Lk) { b00 = fmaf(bw, (*(pd0 + key)), bb); b10 = fmaf(bw, (*(pd1 + key)), bb); }
          if (key + 1 < pr.Lk) { b01 = fmaf(bw, (*(pd0 + key + 1)), bb); b11 = fmaf(bw, (*(pd1 + key + 1)), bb); }
        }
        s[nt][0] = s[nt][0] * 0.125f + ma.x + b00;
        s[nt][1] = s[nt][1] * 0.125f + ma.y + b01;
        s[nt][2] = s[nt][2] * 0.125f + ma.x + b10;
        s[nt][3] = s[nt][3] * 0.125f + ma.y + b11;
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
    const float sc0 = (m0 == -INFINITY) ? 0.f : fast_exp(m0 - mu0);
    const float sc1 = (m1 == -INFINITY) ? 0.f : fast_exp(m1 - mu1);
    m0 = mn0; m1 = mn1;
    l0 *= sc0; l1 *= sc1;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) { o[dt][0] *= sc0; o[dt][1] *= sc0; o[dt][2] *= sc1; o[dt][3] *= sc1; }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (nt < 2 * npairs) {
        s[nt][0] = fast_exp(s[nt][0] - mu0); s[nt][1] = fast_exp(s[nt][1] - mu0);
        s[nt][2] = fast_exp(s[nt][2] - mu1); s[nt][3] = fast_exp(s[nt][3] - mu1);
        l0 += s[nt][0] + s[nt][1];
        l1 += s[nt][2] + s[nt][3];
        if (drop) {      // dropout on the probabilities (vilmodel.py:128,347): the denominator keeps the undropped sum
          const uint32_t e0 = dbase + (uint32_t)r0 * (uint32_t)LkP + (uint32_t)(kc + nt * 8 + 2 * tg);
          const uint32_t e1 = dbase + (uint32_t)r1 * (uint32_t)LkP + (uint32_t)(kc + nt * 8 + 2 * tg);
          s[nt][0] *= vi_hash32(e0, dkey) >= pr.drop_thresh ? pr.drop_scale : 0.f;
          s[nt][1] *= vi_hash32(e0 + 1, dkey) >= pr.drop_thresh ? pr.drop_scale : 0.f;
          s[nt][2] *= vi_hash32(e1, dkey) >= pr.drop_thresh ? pr.drop_scale : 0.f;
          s[nt][3] *= vi_hash32(e1 + 1, dkey) >= pr.drop_thresh ? pr.drop_scale : 0.f;
        }
      }
    }
    // O += P V : P (accumulator layout) re-packed as the A operand; V fragments through ldmatrix.trans
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      if (kk < npairs) {
        uint32_t pa[4];
        pa[0] = pack_h16x2(s[2 * kk][0], s[2 * kk][1], F16);
        pa[1] = pack_h16x2(s[2 * kk][2], s[2 * kk][3], F16);
        pa[2] = pack_h16x2(s[2 * kk + 1][0], s[2 * kk + 1][1], F16);
        pa[3] = pack_h16x2(s[2 * kk + 1][2], s[2 * kk + 1][3], F16);
#pragma unroll
        for (int d2 = 0; d2 < 4; ++d2) {
          uint32_t vb[4];     // (keys 0-7, d 0-7)^T (keys 8-15, d 0-7)^T (keys 0-7, d 8-15)^T (keys 8-15, d 8-15)^T
          ldsm_x4_trans(vb, vs_u + (uint32_t)((kc + kk * 16 + (lm & 1) * 8 + lr) * ROW + d2 * 16 + (lm >> 1) * 8) * 2);
          mma_16816<F16>(o[2 * d2], pa, vb[0], vb[1]);
          mma_16816<F16>(o[2 * d2 + 1], pa, vb[2], vb[3]);
        }
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  bf16* og = reinterpret_cast<bf16*>(pr.o) + (long long)b * pr.Lq * pr.ldo + h * DH;
#pragma unroll
  for (int dt = 0; dt < 8; ++dt) {
    const int c = dt * 8 + 2 * tg;
    if (r0 < pr.Lq) *reinterpret_cast<uint32_t*>(og + (long long)r0 * pr.ldo + c) = pack_h16x2(o[dt][0] * i0, o[dt][1] * i0, F16);
    if (r1 < pr.Lq) *reinterpret_cast<uint32_t*>(og + (long long)r1 * pr.ldo + c) = pack_h16x2(o[dt][2] * i1, o[dt][3] * i1, F16);
  }
  if (pr.lse && tg == 0) {
    float* lg = pr.lse + ((long long)b * p.H + h) * pr.Lq;
    if (r0 < pr.Lq) lg[r0] = m0 + logf(l0);
    if (r1 < pr.Lq) lg[r1] = m1 + logf(l1);
  }
}

// ---------------------------------------------------------------------------------------------------------------------------
// Single-pass form for the inference shapes (every problem <= 96 keys, no dropout, no log-sum-exp output).  Same CTA mapping
// and staging as attn_fwd_bf16_kernel; what changes is the instruction count, which is what bounds this operator (ncu, cfg-2
// cross-attention: 1934 instructions per 16-query warp tile at 43 % issue utilisation, 5 - 6 warps per scheduler):
//   * the number of 16-key blocks is a template parameter chosen per problem, so every loop is exactly unrolled - the generic
//     kernel issues its 64-key chunk body with half of it predicated off for the 32-key tail of an 85-key context;
//   * all scores of a row stay in registers (<= 48 per thread), so there is one softmax pass: no running maximum, no rescaling
//     of the output accumulators, one barrier;
//   * scale, key mask and GASA bias are applied in the log2 domain: one FFMA per score, then FADD + MUFU.EX2 + FADD.
// ---------------------------------------------------------------------------------------------------------------------------
constexpr float LOG2E_F = 1.4426950408889634f;
__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <bool F16, int NB>
__device__ __forceinline__ void attn_sp_body(const AttnProblem& pr, uint32_t ks_u, uint32_t vs_u, uint32_t q_frag, const float* madd,
                                             int b, int h, int q0, int lane) {
  const int g = lane >> 2, tg = lane & 3;
  const int r0 = q0 + g, r1 = q0 + g + 8;
  const int lm = lane >> 3, lr = lane & 7;
  float s[2 * NB][4];
#pragma unroll
  for (int nt = 0; nt < 2 * NB; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
  // GASA bias operands first (graphs of <= 64 nodes): their global loads fly under the score MMAs; larger graphs load them in
  // the scoring loop
  constexpr bool PRE = NB <= 4;
  constexpr int ND = PRE ? 2 * NB : 1;
  float d0[ND][2], d1[ND][2];
  float bw2 = 0.f, bb2 = 0.f;
  const bool gasa = pr.pair_dist != nullptr;
  const float* pd0 = nullptr;
  const float* pd1 = nullptr;
  if (gasa) {
    bw2 = pr.bias_affine[0] * LOG2E_F;
    bb2 = pr.bias_affine[1] * LOG2E_F;
    pd0 = pr.pair_dist + ((long long)b * pr.Lq + (r0 < pr.Lq ? r0 : 0)) * pr.Lk;
    pd1 = pr.pair_dist + ((long long)b * pr.Lq + (r1 < pr.Lq ? r1 : 0)) * pr.Lk;
    if constexpr (PRE) {
#pragma unroll
      for (int nt = 0; nt < 2 * NB; ++nt) {
        const int key = nt * 8 + 2 * tg;
        d0[nt][0] = key < pr.Lk ? pd0[key] : 0.f;
        d1[nt][0] = key < pr.Lk ? pd1[key] : 0.f;
        d0[nt][1] = key + 1 < pr.Lk ? pd0[key + 1] : 0.f;
        d1[nt][1] = key + 1 < pr.Lk ? pd1[key + 1] : 0.f;
      }
    }
  }
  // ... and under the K / V / Q copies: the tiles are waited for only here (every warp of the CTA reaches this barrier)
  cp_async_wait<0>();
  __syncthreads();
  if (q0 >= pr.Lq) return;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t qa[4];
    ldsm_x4(qa, q_frag + (uint32_t)(ks * 32));
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) {
      uint32_t kb[4];
      ldsm_x4(kb, ks_u + (uint32_t)((nb * 16 + (lm >> 1) * 8 + lr) * ROW + ks * 16 + (lm & 1) * 8) * 2);
      mma_16816<F16>(s[2 * nb], qa, kb[0], kb[1]);
      mma_16816<F16>(s[2 * nb + 1], qa, kb[2], kb[3]);
    }
  }
  // log2-domain scores: s * (log2e / 8) + mask (+ bias); row maxima
  const float c1 = 0.125f * LOG2E_F;
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 2 * NB; ++nt) {
    const float2 ma = *reinterpret_cast<const float2*>(madd + nt * 8 + 2 * tg);
    s[nt][0] = fmaf(s[nt][0], c1, ma.x);
    s[nt][1] = fmaf(s[nt][1], c1, ma.y);
    s[nt][2] = fmaf(s[nt][2], c1, ma.x);
    s[nt][3] = fmaf(s[nt][3], c1, ma.y);
    if (gasa) {
      float e00, e01, e10, e11;
      if constexpr (PRE) {
        e00 = d0[nt][0]; e01 = d0[nt][1]; e10 = d1[nt][0]; e11 = d1[nt][1];
      } else {
        const int key = nt * 8 + 2 * tg;
        e00 = key < pr.Lk ? pd0[key] : 0.f;
        e10 = key < pr.Lk ? pd1[key] : 0.f;
        e01 = key + 1 < pr.Lk ? pd0[key + 1] : 0.f;
        e11 = key + 1 < pr.Lk ? pd1[key + 1] : 0.f;
      }
      s[nt][0] += fmaf(bw2, e00, bb2);
      s[nt][1] += fmaf(bw2, e01, bb2);
      s[nt][2] += fmaf(bw2, e10, bb2);
      s[nt][3] += fmaf(bw2, e11, bb2);
    }
    mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
    mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  const float mu0 = (mx0 == -INFINITY) ? 0.f : mx0, mu1 = (mx1 == -INFINITY) ? 0.f : mx1;
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < 2 * NB; ++nt) {
    s[nt][0] = ex2_ftz(s[nt][0] - mu0); s[nt][1] = ex2_ftz(s[nt][1] - mu0);
    s[nt][2] = ex2_ftz(s[nt][2] - mu1); s[nt][3] = ex2_ftz(s[nt][3] - mu1);
    l0 += s[nt][0] + s[nt][1];
    l1 += s[nt][2] + s[nt][3];
  }
  // O = P V
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
#pragma unroll
  for (int kk = 0; kk < NB; ++kk) {
    uint32_t pa[4];
    pa[0] = pack_h16x2(s[2 * kk][0], s[2 * kk][1], F16);
    pa[1] = pack_h16x2(s[2 * kk][2], s[2 * kk][3], F16);
    pa[2] = pack_h16x2(s[2 * kk + 1][0], s[2 * kk + 1][1], F16);
    pa[3] = pack_h16x2(s[2 * kk + 1][2], s[2 * kk + 1][3], F16);
#pragma unroll
    for (int d2 = 0; d2 < 4; ++d2) {
      uint32_t vb[4];
      ldsm_x4_trans(vb, vs_u + (uint32_t)((kk * 16 + (lm & 1) * 8 + lr) * ROW + d2 * 16 + (lm >> 1) * 8) * 2);
      mma_16816<F16>(o[2 * d2], pa, vb[0], vb[1]);
      mma_16816<F16>(o[2 * d2 + 1], pa, vb[2], vb[3]);
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  bf16* og = reinterpret_cast<bf16*>(pr.o) + (long long)b * pr.Lq * pr.ldo + h * DH + 2 * tg;
  bf16* og0 = og + (long long)r0 * pr.ldo;
  bf16* og1 = og + (long long)r1 * pr.ldo;
  if (r0 < pr.Lq) {
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) *reinterpret_cast<uint32_t*>(og0 + dt * 8) = pack_h16x2(o[dt][0] * i0, o[dt][1] * i0, F16);
  }
  if (r1 < pr.Lq) {
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) *reinterpret_cast<uint32_t*>(og1 + dt * 8) = pack_h16x2(o[dt][2] * i1, o[dt][3] * i1, F16);
  }
}

template <bool F16>
__global__ void __launch_bounds__(128, 5) attn_fwd_sp_kernel(const AttnParams p) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  int z = blockIdx.z, pi = 0;
  while (pi < p.n_problems - 1 && z >= p.pr[pi].B) { z -= p.pr[pi].B; ++pi; }
  const AttnProblem& pr = p.pr[pi];
  const int nthr = blockDim.x, qrows = (blockDim.x >> 5) * 16;
  const int q_base = blockIdx.x * qrows;
  if (q_base >= pr.Lq) return;
  const int b = z, h = blockIdx.y;
  const int LkP = pr.LkP;
  bf16* Ks = reinterpret_cast<bf16*>(smem);                 // [LkP][72]
  bf16* Vs = Ks + (size_t)LkP * ROW;                        // [LkP][72]
  bf16* Qs = Vs + (size_t)LkP * ROW;                        // [qrows][72]
  float* madd = reinterpret_cast<float*>(Qs + qrows * ROW); // [LkP], log2 domain
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ch = tid & 7, rstep = nthr >> 3;                // a thread copies 16-byte chunk `ch` of rows r, r + rstep, ...
  const uint32_t ks_u = smem_u32(Ks), vs_u = smem_u32(Vs), qs_u = smem_u32(Qs);
  {
    const bf16* qg = reinterpret_cast<const bf16*>(pr.q) + ((long long)b * pr.Lq + q_base) * pr.ldq + h * DH + ch * 8;
    const int nq = pr.Lq - q_base;
    for (int r = tid >> 3; r < qrows; r += rstep) {
      const bool ok = r < nq;
      cp_async16(qs_u + (uint32_t)(r * ROW + ch * 8) * 2, qg + (long long)(ok ? r : 0) * pr.ldq, ok);
    }
    const bf16* kg = reinterpret_cast<const bf16*>(pr.k) + (long long)b * pr.Lk * pr.ldk + h * DH + ch * 8;
    const bf16* vg = reinterpret_cast<const bf16*>(pr.v) + (long long)b * pr.Lk * pr.ldv + h * DH + ch * 8;
    for (int key = tid >> 3; key < LkP; key += rstep) {
      const bool ok = key < pr.Lk;
      const int kk = ok ? key : 0;
      cp_async16(ks_u + (uint32_t)(key * ROW + ch * 8) * 2, kg + (long long)kk * pr.ldk, ok);
      cp_async16(vs_u + (uint32_t)(key * ROW + ch * 8) * 2, vg + (long long)kk * pr.ldv, ok);
    }
    cp_async_commit();
  }
  for (int key = tid; key < LkP; key += nthr) {
    float m = 0.f;
    if (key >= pr.Lk) m = -INFINITY;
    else if (pr.key_mask && !pr.key_mask[(long long)b * pr.Lk + key]) m = (p.mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f * LOG2E_F;
    madd[key] = m;
  }
  const int q0 = q_base + warp * 16;                         // a warp without rows still joins the barrier inside the body
  const int lm = lane >> 3, lr = lane & 7;
  const uint32_t q_frag = qs_u + (uint32_t)((warp * 16 + (lm & 1) * 8 + lr) * ROW + (lm >> 1) * 8) * 2;
  switch (LkP >> 4) {
    case 1: attn_sp_body<F16, 1>(pr, ks_u, vs_u, q_frag, madd, b, h, q0, lane); break;
    case 2: attn_sp_body<F16, 2>(pr, ks_u, vs_u, q_frag, madd, b, h, q0, lane); break;
    case 3: attn_sp_body<F16, 3>(pr, ks_u, vs_u, q_frag, madd, b, h, q0, lane); break;
    case 4: attn_sp_body<F16, 4>(pr, ks_u, vs_u, q_frag, madd, b, h, q0, lane); break;
    case 5: attn_sp_body<F16, 5>(pr, ks_u, vs_u, q_frag, madd, b, h, q0, lane); break;
    default: attn_sp_body<F16, 6>(pr, ks_u, vs_u, q_frag, madd, b, h, q0, lane); break;
  }
}

// fp32 check mode: grid (H, B), 128 threads; warp w handles query rows w, w+4, ...
__global__ void __launch_bounds__(128) attn_fwd_f32_kernel(const AttnProblem p, const int H, const int mask_mode) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t smem[];
  float* Ks = reinterpret_cast<float*>(smem);            // [Lk][65]
  float* Vs = Ks + (size_t)p.Lk * 65;                    // [Lk][64]
  float* madd = Vs + (size_t)p.Lk * 64;                  // [Lk]
  float* sc = madd + p.Lk;                               // [4][Lk]
  float* qs = sc + 4 * (size_t)p.Lk;                     // [4][64]
  const int b = blockIdx.y, h = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* kg = reinterpret_cast<const float*>(p.k) + (long long)b * p.Lk * p.ldk + h * DH;
  const float* vg = reinterpret_cast<const float*>(p.v) + (long long)b * p.Lk * p.ldv + h * DH;
  for (int e = tid; e < p.Lk * DH; e += 128) {
    const int key = e >> 6, d = e & 63;
    Ks[(size_t)key * 65 + d] = kg[(long long)key * p.ldk + d];
    Vs[(size_t)key * 64 + d] = vg[(long long)key * p.ldv + d];
  }
  for (int key = tid; key < p.Lk; key += 128) {
    float m = 0.f;
    if (p.key_mask && !p.key_mask[(long long)b * p.Lk + key]) m = (mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f;
    madd[key] = m;
  }
  __syncthreads();
  float bw = 0.f, bb = 0.f;
  if (p.pair_dist) { bw = p.bias_affine[0]; bb = p.bias_affine[1]; }
  const float* qg = reinterpret_cast<const float*>(p.q) + (long long)b * p.Lq * p.ldq + h * DH;
  float* og = reinterpret_cast<float*>(p.o) + (long long)b * p.Lq * p.ldo + h * DH;
  float* myq = qs + warp * 64;
  float* mysc = sc + (size_t)warp * p.Lk;
  for (int r = warp; r < p.Lq; r += 4) {
    myq[lane] = qg[(long long)r * p.ldq + lane];
    myq[lane + 32] = qg[(long long)r * p.ldq + lane + 32];
    __syncwarp();
    float mx = -INFINITY;
    for (int key = lane; key < p.Lk; key += 32) {
      float dot = 0.f;
#pragma unroll 16
      for (int d = 0; d < DH; ++d) dot = fmaf(myq[d], Ks[(size_t)key * 65 + d], dot);
      // same association as the reference: (qk / 8 + mask) + bias  (mask+sprels is pre-added there;
      // the difference is below fp32 resolution of the -10000 term only for masked keys)
      float s = dot * 0.125f;
      float add = madd[key];
      if (p.pair_dist) add += fmaf(bw, p.pair_dist[((long long)b * p.Lq + r) * p.Lk + key], bb);
      s += add;
      mysc[key] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    const float mu = (mx == -INFINITY) ? 0.f : mx;
    float sum = 0.f;
    for (int key = lane; key < p.Lk; key += 32) {
      const float e = expf(mysc[key] - mu);
      mysc[key] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    __syncwarp();
    float a0 = 0.f, a1 = 0.f;
    for (int key = 0; key < p.Lk; ++key) {
      const float pj = mysc[key];
      a0 = fmaf(pj, Vs[(size_t)key * 64 + lane], a0);
      a1 = fmaf(pj, Vs[(size_t)key * 64 + lane + 32], a1);
    }
    const float inv = 1.0f / sum;
    og[(long long)r * p.ldo + lane] = a0 * inv;
    og[(long long)r * p.ldo + lane + 32] = a1 * inv;
    if (p.lse && lane == 0) p.lse[((long long)b * H + h) * p.Lq + r] = mx + logf(sum);
    __syncwarp();
  }
}

}  // namespace

static int check_problem(const vi_attn_problem& a, int H, int dtype, AttnProblem& o) {
  VI_CHECK_ARG(a.q && a.k && a.v && a.o, "vi_attn_fwd_multi: null operand");
  VI_CHECK_ARG(a.B > 0 && a.Lq > 0 && a.Lk > 0, "vi_attn_fwd_multi: empty problem B=%d Lq=%d Lk=%d", a.B, a.Lq, a.Lk);
  VI_CHECK_ARG(a.Lk <= 512, "vi_attn_fwd_multi: Lk=%d exceeds the single-pass limit of 512 keys", a.Lk);
  VI_CHECK_ARG(!a.pair_dist || a.bias_affine, "vi_attn_fwd_multi: pair_dist needs bias_affine {w,b}");
  const int64_t hd = (int64_t)H * DH;
  VI_CHECK_ARG(a.ldq >= hd && a.ldk >= hd && a.ldv >= hd && a.ldo >= hd, "vi_attn_fwd_multi: leading dimensions smaller than H*64");
  if (dtype != VI_DT_F32) {
    VI_CHECK_ARG(a.ldq % 8 == 0 && a.ldk % 8 == 0 && a.ldv % 8 == 0 && a.ldo % 2 == 0,
                 "vi_attn_fwd_multi: bf16 leading dims must be multiples of 8");
    VI_CHECK_ARG((((uintptr_t)a.q | (uintptr_t)a.k | (uintptr_t)a.v) & 15) == 0 && ((uintptr_t)a.o & 3) == 0,
                 "vi_attn_fwd_multi: misaligned bf16 operands");
  }
  o.q = a.q; o.ldq = a.ldq; o.k = a.k; o.ldk = a.ldk; o.v = a.v; o.ldv = a.ldv; o.o = a.o; o.ldo = a.ldo;
  o.key_mask = a.key_mask; o.pair_dist = a.pair_dist; o.bias_affine = a.bias_affine; o.lse = a.lse;
  o.B = a.B; o.Lq = a.Lq; o.Lk = a.Lk; o.LkP = (a.Lk + 15) & ~15;
  VI_CHECK_ARG(a.drop_p >= 0.f && a.drop_p < 1.f && (a.drop_p == 0.f || (a.drop_seed && dtype != VI_DT_F32)),
               "vi_attn_fwd_multi: attention dropout needs 0 <= p < 1, a device seed pointer and the bf16 kernel");
  o.drop_thresh = a.drop_p > 0.f ? vi_drop_threshold(a.drop_p) : 0u;
  if (a.drop_p > 0.f && o.drop_thresh == 0u) o.drop_thresh = 1u;
  o.drop_scale = a.drop_p > 0.f ? 1.0f / (1.0f - a.drop_p) : 1.0f;
  o.drop_site = a.drop_site; o.drop_seed = a.drop_seed;
  return VI_OK;
}

extern "C" int vi_attn_fwd_multi(const vi_attn_problem* problems, int n_problems, int H, int dtype, int mask_mode,
                                 vi_stream_t stream) {
  VI_CHECK_ARG(problems && n_problems >= 1 && n_problems <= VI_ATTN_MAX_PROBLEMS, "vi_attn_fwd_multi: 1..%d problems",
               VI_ATTN_MAX_PROBLEMS);
  VI_CHECK_ARG(H > 0, "vi_attn_fwd_multi: H must be positive");
  VI_CHECK_ARG(mask_mode == VI_MASK_ADD_NEG10000 || mask_mode == VI_MASK_NEG_INF, "vi_attn_fwd_multi: bad mask_mode");
  VI_CHECK_ARG(dtype == VI_DT_BF16 || dtype == VI_DT_F32 || dtype == VI_DT_F16, "vi_attn_fwd_multi: bad dtype %d", dtype);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.n_problems = n_problems; p.H = H; p.mask_mode = mask_mode;
  int total_b = 0, max_lq = 0, max_lkp = 0;
  for (int i = 0; i < n_problems; ++i) {
    if (int rc = check_problem(problems[i], H, dtype, p.pr[i])) return rc;
    total_b += p.pr[i].B;
    max_lq = p.pr[i].Lq > max_lq ? p.pr[i].Lq : max_lq;
    max_lkp = p.pr[i].LkP > max_lkp ? p.pr[i].LkP : max_lkp;
  }
  if (dtype != VI_DT_F32) {
    const int q_tiles = (max_lq + 15) / 16;
    const int nwarp = q_tiles < 4 ? q_tiles : 4;
    const int qrows = nwarp * 16;
    const size_t smem = (size_t)max_lkp * ROW * 2 * 2 + (size_t)qrows * ROW * 2 + (size_t)max_lkp * 4;
    dim3 grid((max_lq + qrows - 1) / qrows, H, total_b);
    // inference shapes (<= 96 keys, no dropout, no log-sum-exp): the single-pass kernel; training and longer key sets the generic one
    bool sp = max_lkp <= 96;
    for (int i = 0; i < n_problems; ++i) sp = sp && p.pr[i].drop_thresh == 0 && p.pr[i].lse == nullptr;
    if (sp && dtype == VI_DT_F16) {
      VI_CUDA(vi_launch(attn_fwd_sp_kernel<true>, dim3(grid), dim3(nwarp * 32), (size_t)(smem), st, p));
    } else if (sp) {
      VI_CUDA(vi_launch(attn_fwd_sp_kernel<false>, dim3(grid), dim3(nwarp * 32), (size_t)(smem), st, p));
    } else if (dtype == VI_DT_F16) {
      VI_CUDA(vi_launch(attn_fwd_bf16_kernel<true>, dim3(grid), dim3(nwarp * 32), (size_t)(smem), st, p));
    } else {
      VI_CUDA(vi_launch(attn_fwd_bf16_kernel<false>, dim3(grid), dim3(nwarp * 32), (size_t)(smem), st, p));
    }
    VI_LAUNCH_CHECK();
  } else {
    for (int i = 0; i < n_problems; ++i) {
      const AttnProblem& a = p.pr[i];
      const size_t smem = ((size_t)a.Lk * 65 + (size_t)a.Lk * 64 + a.Lk + 4 * (size_t)a.Lk + 4 * 64) * 4;
      dim3 grid(H, a.B);
      VI_CUDA(vi_launch(attn_fwd_f32_kernel, dim3(grid), dim3(128), (size_t)(smem), st, a, H, mask_mode));
      VI_LAUNCH_CHECK();
    }
  }
  return VI_OK;
}

int vi_attn_init() {
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_bf16_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 176 * 1024));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_bf16_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_bf16_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 176 * 1024));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_bf16_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_sp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_sp_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_sp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_sp_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  VI_CUDA(cudaFuncSetAttribute(attn_fwd_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  return VI_OK;
}
