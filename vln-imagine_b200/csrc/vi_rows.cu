// vi_rows.cu - HBM-bound row kernels: one warp per 768-wide row, fp32 statistics via warp shuffles,
// 16-byte coalesced accesses (lane l touches float4 #(l + 32 j), j = 0..5, of its row).
//
// LayerNorm / residual / embedding sums / action-logit tail / aux-loss reductions of
// VLN-DUET/map_nav_src/models/vilmodel.py and VLN-HAMT/finetune_src/models/vilmodel_cmt.py; each
// entry point cites its reference lines in include/vlnimagine.h.
#include "vi_common.cuh"
#include <cuda_fp16.h>

namespace {

constexpr int D = VI_HIDDEN;     // 768
constexpr int V4 = D / 128;      // 6 float4 per lane
constexpr int ROWS_PER_BLOCK = 4;

struct Row {
  float v[V4 * 4];
};

__device__ __forceinline__ void row_zero(Row& r) {
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) r.v[i] = 0.f;
}
__device__ __forceinline__ void row_load(Row& r, const float* src, int lane) {
  const float4* s4 = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    const float4 t = (*(s4 + lane + 32 * j));
    r.v[4 * j] = t.x; r.v[4 * j + 1] = t.y; r.v[4 * j + 2] = t.z; r.v[4 * j + 3] = t.w;
  }
}
__device__ __forceinline__ void row_add(Row& r, const float* src, int lane) {
  const float4* s4 = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    const float4 t = (*(s4 + lane + 32 * j));
    r.v[4 * j] += t.x; r.v[4 * j + 1] += t.y; r.v[4 * j + 2] += t.z; r.v[4 * j + 3] += t.w;
  }
}
__device__ __forceinline__ void row_acc(Row& r, const Row& o) {
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) r.v[i] += o.v[i];
}
// in-place LayerNorm over the 768 values held by the warp (biased variance, like torch)
__device__ __forceinline__ void row_layernorm(Row& r, const float* gamma, const float* beta,
                                              float eps, int lane) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) s += r.v[i];
  const float mean = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) { const float d = r.v[i] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    const float4 g = (*(g4 + lane + 32 * j)), b = (*(b4 + lane + 32 * j));
    r.v[4 * j] = (r.v[4 * j] - mean) * rstd * g.x + b.x;
    r.v[4 * j + 1] = (r.v[4 * j + 1] - mean) * rstd * g.y + b.y;
    r.v[4 * j + 2] = (r.v[4 * j + 2] - mean) * rstd * g.z + b.z;
    r.v[4 * j + 3] = (r.v[4 * j + 3] - mean) * rstd * g.w + b.w;
  }
}
__device__ __forceinline__ void row_store(const Row& r, float* y32, bf16* y16, long long row, int lane, bool f16 = false) {
  if (y32) {
    float4* o = reinterpret_cast<float4*>(y32 + row * D);
#pragma unroll
    for (int j = 0; j < V4; ++j) o[lane + 32 * j] = make_float4(r.v[4 * j], r.v[4 * j + 1], r.v[4 * j + 2], r.v[4 * j + 3]);
  }
  if (y16) {
    uint2* o = reinterpret_cast<uint2*>(y16 + row * D);
#pragma unroll
    for (int j = 0; j < V4; ++j)
      o[lane + 32 * j] = make_uint2(pack_h16x2(r.v[4 * j], r.v[4 * j + 1], f16), pack_h16x2(r.v[4 * j + 2], r.v[4 * j + 3], f16));
  }
}
__device__ __forceinline__ float row_dot(const Row& a, const Row& b) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) s = fmaf(a.v[i], b.v[i], s);
  return warp_sum(s);
}

#define ROW_INDEX()                                                           \
  const int lane = threadIdx.x & 31;                                          \
  const long long row = (long long)blockIdx.x * ROWS_PER_BLOCK + (threadIdx.x >> 5)

// ---------------------------------------------------------------------------------------------
struct RowGroups {
  int n;
  int end[4];
};
__device__ __forceinline__ int group_of_row(const RowGroups& g, long long row) {
  int i = 0;
  while (i < g.n - 1 && row >= g.end[i]) ++i;
  return i;
}

__global__ void __launch_bounds__(128) add_ln_kernel(const float* a, const float* b,
                                                     const float* gamma, const float* beta,
                                                     float eps, float* y32, bf16* y16, int f16, long long rows, const RowGroups grp) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const int gi = group_of_row(grp, row);
  gamma += gi * D;
  beta += gi * D;
  Row r;
  row_load(r, a + row * D, lane);
  if (b) row_add(r, b + row * D, lane);
  row_layernorm(r, gamma, beta, eps, lane);
  row_store(r, y32, y16, row, lane, f16 != 0);
}

// LN(dropout(a) + b): the hidden dropout of BertSelfOutput / BertOutput (D/models/vilmodel.py:151-155,190-194) applied on the fly -
// keep(i) = hash(i, seed, site) >= threshold with i = row * 768 + column, the same mask vi_dropout produces for a [rows, 768] tensor
__global__ void __launch_bounds__(128) add_ln_drop_kernel(const float* a, const float* b, const float* gamma, const float* beta,
                                                          float eps, float* y32, bf16* y16, int f16, long long rows,
                                                          const RowGroups grp, uint32_t thresh, float scale, const uint32_t* seed,
                                                          uint32_t site) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const int gi = group_of_row(grp, row);
  gamma += gi * D;
  beta += gi * D;
  const uint32_t key = vi_drop_key(seed, site);
  Row r;
  row_load(r, a + row * D, lane);
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    const uint32_t e0 = (uint32_t)(row * D) + (uint32_t)((lane + 32 * j) * 4);
#pragma unroll
    for (int e = 0; e < 4; ++e) r.v[4 * j + e] = vi_hash32(e0 + e, key) >= thresh ? r.v[4 * j + e] * scale : 0.f;
  }
  if (b) row_add(r, b + row * D, lane);
  row_layernorm(r, gamma, beta, eps, lane);
  row_store(r, y32, y16, row, lane, f16 != 0);
}

// One row per warp, 4 warps per CTA.  Everything a row needs PER COLUMN - the TRANSPOSED weight of the small feature
// projection ([feat_dim][768], prepared by the caller once per weight version) and up to eleven 768-wide vectors (LayerNorm
// gains / biases, the feature bias, constant rows; 33 - 76 KB in all) - is read with plain 16-byte loads through the SM's L1.
// The grid is ONE wave whose warps start together, so without help every warp walks the k-loop and the vectors as a chain of
// 20 - 30 dependent L2 round trips (ncu: 29 of 36 cycles per issued instruction on the long scoreboard); the kernel therefore
// touches every parameter line once at its top, all loads in flight, ahead of the dependency wait - measured 8.5 us per
// navigation step (3 launches), 0.8255 -> 0.8170 ms.  The row's own data (the row, its table row) is prefetched at the top
// and loaded when it is needed, which keeps the live registers at one accumulator row + one operand row.
// Measured and rejected: two rows per warp sharing every parameter load (half the L1 traffic, 150 registers, 0.4 % slower -
// the kernel is latency-, not L1-bandwidth-bound); staging the parameters in shared memory per CTA (80 KB for 8 rows: the
// L2 -> SM traffic dominates); prefetch.global.L1 for the warm-up (CCTL.PF1: no effect).
constexpr int EMBED_WARPS = 4;

__device__ __forceinline__ void prefetch_row_l1(const float* src, int lane) {       // 768 floats = 24 lines of 128 bytes
  if (lane < 24) asm volatile("prefetch.global.L1 [%0];" ::"l"(src + lane * 32));
}

// Brings the 128-byte line into the SM's L1 with a real load: prefetch.global.L1 (CCTL.PF1) measured as a no-op for this
// purpose on sm_100a, and ptxas deletes a load whose result is dead - so the values are summed and the sum is "used" by a
// harmless, practically never taken branch at the end of the kernel (warm_sink), long after the loads have landed.
__device__ __forceinline__ float touch_line(const float* src) {
  float v;
  asm volatile("ld.global.ca.f32 %0, [%1];" : "=f"(v) : "l"(src));
  return v;
}
__device__ __forceinline__ void warm_sink(float warm) {
  if (warm == -1.2345678e-30f) asm volatile("nanosleep.u32 0;");
}

__global__ void __launch_bounds__(EMBED_WARPS * 32) embed_compose_kernel(const vi_embed_args p) {
  pdl_launch_dependents();
  // Warm the L1 with every PARAMETER line the rows will read (the transposed weight and the vectors), all loads in flight at
  // once and BEFORE waiting for the previous kernel: the whole grid is one wave that starts together, so without this every
  // warp walks the k-loop and the vectors as a chain of 20 - 30 dependent L2 round trips.  Parameters are never written by a
  // kernel of this library, so reading them ahead of the dependency is safe; activations are read after pdl_wait().
  float warm = 0.f;
  {
    const int tid = threadIdx.x;
    if (p.feat)
      for (int l = tid; l < p.feat_dim * (D / 32); l += EMBED_WARPS * 32) warm += touch_line(p.feat_w + l * 32);
    if (tid < 120) {
      const int grp = tid / 24, ln = (tid % 24) * 32;
#define VI_WARM(ptr, i) if ((ptr) && grp == (i) % 5) warm += touch_line((ptr) + ln);
      VI_WARM(p.feat_b, 0) VI_WARM(p.feat_gamma, 1) VI_WARM(p.feat_beta, 2) VI_WARM(p.a_gamma, 3) VI_WARM(p.a_beta, 4)
      VI_WARM(p.const_row, 5) VI_WARM(p.const_row2, 6) VI_WARM(p.out_gamma, 7) VI_WARM(p.out_beta, 8) VI_WARM(p.ln2_gamma, 9)
      VI_WARM(p.ln2_beta, 10)
#undef VI_WARM
    }
  }
  pdl_wait();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long row = (long long)blockIdx.x * EMBED_WARPS + warp;
  const long long end = p.rows + p.zero_rows;
  if (row >= end) return;
  if (row >= p.rows) {                             // padding rows behind the stream (row-stacked activations): zeros
    Row z;
    row_zero(z);
    row_store(z, p.y32, reinterpret_cast<bf16*>(p.y16), row, lane, p.y16_dtype == VI_DT_F16);
    return;
  }

  // ---- the row's own data: small loads now, the 3 KB rows prefetched into L1
  const float fv = (p.feat && lane < p.feat_dim) ? *(p.feat + row * p.feat_dim + lane) : 0.f;
  const long long ti = p.idx ? p.idx[row] : 0;
  if (p.a) prefetch_row_l1(p.a + row * D, lane);
  if (p.idx) prefetch_row_l1(p.table + ti * D, lane);

  Row acc;
  row_zero(acc);
  if (p.feat) {
    if (p.feat_b) row_add(acc, p.feat_b, lane);
    for (int k = 0; k < p.feat_dim; ++k) {
      const float f = __shfl_sync(0xffffffffu, fv, k);
      const float4* w4 = reinterpret_cast<const float4*>(p.feat_w + (long long)k * D);       // transposed: [feat_dim][768]
#pragma unroll
      for (int j = 0; j < V4; ++j) {
        const float4 w = *(w4 + lane + 32 * j);
        acc.v[4 * j] = fmaf(f, w.x, acc.v[4 * j]);
        acc.v[4 * j + 1] = fmaf(f, w.y, acc.v[4 * j + 1]);
        acc.v[4 * j + 2] = fmaf(f, w.z, acc.v[4 * j + 2]);
        acc.v[4 * j + 3] = fmaf(f, w.w, acc.v[4 * j + 3]);
      }
    }
    if (p.feat_gamma) row_layernorm(acc, p.feat_gamma, p.feat_beta, p.eps, lane);
  }
  if (p.a) {
    Row a;
    row_load(a, p.a + row * D, lane);
    if (p.a_gamma) row_layernorm(a, p.a_gamma, p.a_beta, p.eps, lane);
    row_acc(acc, a);
  }
  if (p.a2) row_add(acc, p.a2 + row * D, lane);
  if (p.a3) row_add(acc, p.a3 + row * D, lane);
  if (p.idx) row_add(acc, p.table + ti * D, lane);
  if (p.pos_table) row_add(acc, p.pos_table + (row % p.pos_period) * D, lane);
  if (p.const_row) row_add(acc, p.const_row, lane);
  if (p.const_row2) row_add(acc, p.const_row2, lane);
  if (p.out_gamma) row_layernorm(acc, p.out_gamma, p.out_beta, p.eps, lane);
  if (p.ln2_gamma) {
    // a second LayerNorm chained on the result (norm1 of the first panorama layer, D/models/transformer.py:171): the fp32
    // output keeps the first result (the residual stream), the 16-bit output is the operand of the next contraction
    if (p.y32) row_store(acc, p.y32, nullptr, row, lane);
    row_layernorm(acc, p.ln2_gamma, p.ln2_beta, p.ln2_eps, lane);
    row_store(acc, nullptr, reinterpret_cast<bf16*>(p.y16), row, lane, p.y16_dtype == VI_DT_F16);
    warm_sink(warm);
    return;
  }
  row_store(acc, p.y32, reinterpret_cast<bf16*>(p.y16), row, lane, p.y16_dtype == VI_DT_F16);
  warm_sink(warm);
}

__global__ void __launch_bounds__(128) ln_dot_kernel(const float* h, const float* gamma,
                                                     const float* beta, float eps,
                                                     const float* w, const float* bias,
                                                     float* out, long long rows, const RowGroups grp) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const int gi = group_of_row(grp, row);
  w += gi * D;
  if (bias) bias += gi;
  Row r, wv;
  row_load(r, h + row * D, lane);
  if (gamma) row_layernorm(r, gamma + gi * D, beta + gi * D, eps, lane);       // gamma == NULL: plain dot product of the rows
  row_load(wv, w, lane);
  const float d = row_dot(r, wv);
  if (lane == 0) out[row] = d + (bias ? (*(bias)) : 0.f);
}

__global__ void __launch_bounds__(128) mul_bcast_kernel(const float* x, long long x_bs,
                                                        const float* s, long long lds, float* y32,
                                                        bf16* y16, int f16, long long rows, int rows_per_batch) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const long long b = row / rows_per_batch;
  Row r, m;
  row_load(r, x + b * x_bs + (row - b * rows_per_batch) * D, lane);
  row_load(m, s + b * lds, lane);
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) r.v[i] *= m.v[i];
  row_store(r, y32, y16, row, lane, f16 != 0);
}

// One warp per episode.  Viewpoint-id strings are interned to int32 on the host (gmap_ids: -1 = padding,
// cand_ids: -2 = padding); set membership / dictionary look-ups of the reference become id comparisons here,
// so no mask has to travel back to the host.  bw is accumulated sequentially in candidate order like the
// reference's Python loop (same fp32 association).
constexpr int FUSE_MAX = 512;
__global__ void __launch_bounds__(32) duet_fuse_logits_kernel(const float* g_raw, const float* l_raw,
                                                              const float* fuse_raw,
                                                              const uint8_t* gmap_masks,
                                                              const uint8_t* gmap_visited,
                                                              const uint8_t* vp_nav,
                                                              const int32_t* gmap_ids,
                                                              const int32_t* cand_ids, float* global_logits,
                                                              float* local_logits, float* fused_logits, int G, int P) {
  pdl_enter();
  __shared__ float ll[FUSE_MAX];
  __shared__ int gid[FUSE_MAX];
  __shared__ int cid[FUSE_MAX];
  __shared__ int vid[FUSE_MAX];           // gid of the visited nodes, -1 elsewhere
  __shared__ uint8_t gvis[FUSE_MAX];      // node id is in the reference's `visited_nodes` set
  __shared__ uint8_t cvis[FUSE_MAX];      // candidate id is in `visited_nodes`
  __shared__ float bw_s;
  const int b = blockIdx.x, lane = threadIdx.x;
  const float fw = fuse_raw ? 1.0f / (1.0f + expf(-fuse_raw[b])) : 0.5f;
  const float ninf = -INFINITY;
  for (int v = lane; v < P; v += 32) {
    const long long i = (long long)b * P + v;
    const float x = vp_nav[i] ? l_raw[i] * (1.0f - fw) : ninf;
    ll[v] = x;
    local_logits[i] = x;
    cid[v] = cand_ids[i];
  }
  // ids of the VISITED nodes only (-1 otherwise): the set look-ups below then run on shared memory alone (they used to read
  // gmap_visited from global memory inside the inner loops: one latency chain per comparison hit)
  for (int j = lane; j < G; j += 32) {
    const int id = gmap_ids[(long long)b * G + j];
    gid[j] = id;
    vid[j] = (id != -1 && gmap_visited[(long long)b * G + j]) ? id : -1;
  }
  __syncwarp();
  for (int j = lane; j < G; j += 32) {
    bool in_set = false;
    const int id = gid[j];
    if (id != -1)
      for (int k = 0; k < G; ++k) in_set |= vid[k] == id;
    gvis[j] = in_set;
  }
  for (int v = lane; v < P; v += 32) {
    bool in_set = false;
    const int id = cid[v];
    if (id != -2 && id != -1)
      for (int k = 0; k < G; ++k) in_set |= vid[k] == id;
    cvis[v] = in_set;
  }
  __syncwarp();
  if (lane == 0) {
    float bw = 0.f;
    for (int v = 1; v < P; ++v)
      if (cid[v] != -2 && cvis[v]) bw += ll[v];
    bw_s = bw;
  }
  __syncwarp();
  const float bw = bw_s;
  for (int j = lane; j < G; j += 32) {
    const long long i = (long long)b * G + j;
    float x = g_raw[i] * fw;
    if (gmap_visited[i] || !gmap_masks[i]) x = ninf;
    global_logits[i] = x;
    float f = x;
    if (j == 0) f += ll[0];
    else if (gid[j] != -1 && !gvis[j]) {
      int hit = -1;
      for (int v = 1; v < P; ++v)
        if (cid[v] != -2 && !cvis[v] && cid[v] == gid[j]) hit = v;      // dict semantics: the last one wins
      f += hit >= 0 ? ll[hit] : bw;
    }
    fused_logits[i] = f;
  }
}

__global__ void mask_logits_navtype_kernel(const float* raw, const int64_t* nav_types,
                                           float* out, long long n) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = nav_types[i] == 0 ? -INFINITY : raw[i];
}

__global__ void __launch_bounds__(128) gather_mean_kernel(const float* src, const int32_t* offsets,
                                                          const int32_t* row_idx, float* out32, bf16* out16, int f16,
                                                          long long rows) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  Row acc;
  row_zero(acc);
  const int s = offsets[row], e = offsets[row + 1];
  // four member rows in flight at a time (a segment of 36 views used to be 36 serialised DRAM round trips = 30 us for the
  // history panorama mean of HAMT); they are still ADDED in member order, so the fp32 sum is unchanged
  int t = s;
  for (; t + 4 <= e; t += 4) {
    Row r0, r1, r2, r3;
    const long long i0 = row_idx[t], i1 = row_idx[t + 1], i2 = row_idx[t + 2], i3 = row_idx[t + 3];
    row_load(r0, src + i0 * D, lane);
    row_load(r1, src + i1 * D, lane);
    row_load(r2, src + i2 * D, lane);
    row_load(r3, src + i3 * D, lane);
    row_acc(acc, r0); row_acc(acc, r1); row_acc(acc, r2); row_acc(acc, r3);
  }
  for (; t < e; ++t) row_add(acc, src + (long long)row_idx[t] * D, lane);
  // torch.mean = sum / n (true division); n == 0 never reaches the kernel (host filters empty rows)
  const float n = (float)(e - s);
#pragma unroll
  for (int i = 0; i < V4 * 4; ++i) acc.v[i] = acc.v[i] / n;
  row_store(acc, out32, out16, row, lane, f16 != 0);
}

__global__ void __launch_bounds__(128) scatter_rows_kernel(const float* src, const int32_t* dst_rows,
                                                           float* dst, long long rows) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  Row r;
  row_load(r, src + row * D, lane);
  row_store(r, dst, nullptr, dst_rows[row], lane);
}

// 1 - cos(p, t) with torch's cosine_similarity clamping: x.y / (max(|x|,eps) * max(|y|,eps))
__global__ void __launch_bounds__(128) cosine_loss_kernel(const float* proj, const float* tgt,
                                                          float* loss_rows, long long rows) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  Row a, b;
  row_load(a, proj + row * D, lane);
  row_load(b, tgt + row * D, lane);
  const float ab = row_dot(a, b), aa = row_dot(a, a), bb = row_dot(b, b);
  if (lane == 0) loss_rows[row] = 1.0f - ab / (fmaxf(sqrtf(aa), 1e-8f) * fmaxf(sqrtf(bb), 1e-8f));
}

// single-block deterministic mean of n floats (n <= a few thousand)
__global__ void __launch_bounds__(256) mean_kernel(const float* x, float* out, int n) {
  pdl_enter();
  __shared__ float sh[8];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) s += x[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += sh[i];
    *out = n > 0 ? t / (float)n : 0.f;
  }
}

// sims[r, 0] = cos(proj r, tgt r)/T ; sims[r, 1+n] = cos(proj r, negs n)/T ; one warp per (r, column)
__global__ void __launch_bounds__(128) infonce_sims_kernel(const float* proj, const float* tgt,
                                                           const float* negs, float inv_t, float* sims,
                                                           int R, int n_negs) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long item = (long long)blockIdx.x * ROWS_PER_BLOCK + (threadIdx.x >> 5);
  const int cols = n_negs + 1;
  if (item >= (long long)R * cols) return;
  const int r = (int)(item / cols), c = (int)(item % cols);
  Row a, b;
  row_load(a, proj + (long long)r * D, lane);
  row_load(b, c == 0 ? tgt + (long long)r * D : negs + (long long)(c - 1) * D, lane);
  const float ab = row_dot(a, b), aa = row_dot(a, a), bb = row_dot(b, b);
  if (lane == 0) sims[item] = ab / (fmaxf(sqrtf(aa), 1e-8f) * fmaxf(sqrtf(bb), 1e-8f)) * inv_t;
}
// loss_r = logsumexp over {col 0} U {negatives of other episodes} - sims[r,0]; one warp per row
__global__ void __launch_bounds__(128) infonce_rows_kernel(const float* sims, const int32_t* row_ep,
                                                           const int32_t* neg_ep, float* loss_rows, int R,
                                                           int n_negs) {
  pdl_enter();
  ROW_INDEX();
  if (row >= R) return;
  const int cols = n_negs + 1;
  const float* s = sims + row * cols;
  const int ep = row_ep[row];
  float mx = s[0];
  for (int c = 1 + lane; c < cols; c += 32)
    if (neg_ep[c - 1] != ep) mx = fmaxf(mx, s[c]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int c = 1 + lane; c < cols; c += 32)
    if (neg_ep[c - 1] != ep) sum += expf(s[c] - mx);
  sum = warp_sum(sum) + expf(s[0] - mx);
  if (lane == 0) loss_rows[row] = mx + logf(sum) - s[0];
}

// margin form (H/models/vilmodel_cmt.py:825-856): loss_r = (1 - cos_pos) + mean over the negatives of OTHER episodes of
// relu(margin + cos_neg - cos_pos); `sims` holds plain cosines (inv_t = 1).  No admissible negative -> 0 / 0 = NaN, as
// torch.mean of an empty tensor in the reference.
__global__ void __launch_bounds__(128) margin_rows_kernel(const float* sims, const int32_t* row_ep, const int32_t* neg_ep,
                                                          float margin, float* loss_rows, int R, int n_negs) {
  pdl_enter();
  ROW_INDEX();
  if (row >= R) return;
  const int cols = n_negs + 1;
  const float* s = sims + row * cols;
  const int ep = row_ep[row];
  const float pos = s[0];
  float sum = 0.f, cnt = 0.f;
  for (int c = 1 + lane; c < cols; c += 32)
    if (neg_ep[c - 1] != ep) { sum += fmaxf(margin + s[c] - pos, 0.f); cnt += 1.f; }
  sum = warp_sum(sum);
  cnt = warp_sum(cnt);
  if (lane == 0) loss_rows[row] = (1.0f - pos) + sum / cnt;
}

__global__ void cast_bf16_kernel(const float* src, bf16* dst, int f16, long long n4, long long n) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) {
    const float4 t = (*(reinterpret_cast<const float4*>(src) + i));
    reinterpret_cast<uint2*>(dst)[i] = make_uint2(pack_h16x2(t.x, t.y, f16 != 0), pack_h16x2(t.z, t.w, f16 != 0));
  }
  if (i == 0)
    for (long long j = n4 * 4; j < n; ++j)
      reinterpret_cast<uint16_t*>(dst)[j] = (uint16_t)(pack_h16x2(src[j], 0.f, f16 != 0) & 0xFFFFu);
}

// dst[r, :] = dropout(store[idx[r], 0:F]) for a device-resident feature store: 8 elements (16 bytes of a 16-bit store, two
// float4 of an fp32 one) per thread.  Values, mask and rounding are those of the dense path store[idx].float() ->
// vi_dropout (element id r * F + c) -> vi_cast_h16; an index outside [0, n_store) gives a zero row and reads nothing.
template <typename T> struct StoreVec;
template <> struct StoreVec<float> {
  static __device__ __forceinline__ void load(const float* p, float (&f)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
};
template <> struct StoreVec<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&f)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      f[2 * j] = __uint_as_float(w[j] << 16);
      f[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
    }
  }
};
template <> struct StoreVec<__half> {
  static __device__ __forceinline__ void load(const __half* p, float (&f)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
      f[2 * j] = t.x;
      f[2 * j + 1] = t.y;
    }
  }
};

// One warp per output row, 8 rows per CTA: the row index is read once, then every 16-byte load of the row is issued before the
// first store (up to 4 per lane), so a row costs two dependent memory round trips (index, then data); a thread per 8 elements
// would repeat the index load and a 64-bit division for every 16 bytes.
constexpr int GATHER_UNROLL = 4;
template <typename T>
__global__ void __launch_bounds__(256) gather_rows_kernel(const T* store, long long ld_store, long long n_store, const int32_t* idx,
                                                          long long n_rows, int F, float* dst32, bf16* dst16, int f16,
                                                          uint32_t thresh, float scale, const uint32_t* seed, uint32_t site) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const long long s = idx[r];
  const bool ok = s >= 0 && s < n_store;
  const T* src = store + (ok ? s : 0LL) * ld_store;
  const uint32_t key = seed ? vi_drop_key(seed, site) : 0u;
  for (int c0 = lane * 8; c0 < F; c0 += 256 * GATHER_UNROLL) {
    float f[GATHER_UNROLL][8];
#pragma unroll
    for (int u = 0; u < GATHER_UNROLL; ++u) {
      const int c = c0 + u * 256;
      if (ok && c < F) {
        StoreVec<T>::load(src + c, f[u]);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[u][j] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < GATHER_UNROLL; ++u) {
      const int c = c0 + u * 256;
      if (c >= F) break;
      const long long o = r * F + c;
      if (seed) {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[u][j] = vi_hash32((uint32_t)(o + j), key) >= thresh ? f[u][j] * scale : 0.f;
      }
      if (dst32) {
        float4* d = reinterpret_cast<float4*>(dst32 + o);
        d[0] = make_float4(f[u][0], f[u][1], f[u][2], f[u][3]);
        d[1] = make_float4(f[u][4], f[u][5], f[u][6], f[u][7]);
      }
      if (dst16)
        *reinterpret_cast<uint4*>(dst16 + o) = make_uint4(pack_h16x2(f[u][0], f[u][1], f16 != 0), pack_h16x2(f[u][2], f[u][3], f16 != 0),
                                                          pack_h16x2(f[u][4], f[u][5], f16 != 0), pack_h16x2(f[u][6], f[u][7], f16 != 0));
    }
  }
}

// dst[b, r, :] = src[b, r, :] for nb batches of `rpb` 768-wide rows with independent batch / row strides
// (token concatenation [txt; imagine], token-0 gathers, fp32 -> bf16 operand copies)
__global__ void __launch_bounds__(128) copy_rows_kernel(const float* src, long long src_bs, long long src_rs,
                                                        float* dst32, bf16* dst16, int f16, long long dst_bs, long long dst_rs,
                                                        long long rows, int rpb) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const long long b = row / rpb, r = row % rpb;
  Row v;
  row_load(v, src + b * src_bs + r * src_rs, lane);
  const long long off = b * dst_bs + r * dst_rs;
  if (dst32) {
    float4* o = reinterpret_cast<float4*>(dst32 + off);
#pragma unroll
    for (int j = 0; j < V4; ++j) o[lane + 32 * j] = make_float4(v.v[4 * j], v.v[4 * j + 1], v.v[4 * j + 2], v.v[4 * j + 3]);
  }
  if (dst16) {
    uint2* o = reinterpret_cast<uint2*>(dst16 + off);
#pragma unroll
    for (int j = 0; j < V4; ++j)
      o[lane + 32 * j] = make_uint2(pack_h16x2(v.v[4 * j], v.v[4 * j + 1], f16 != 0), pack_h16x2(v.v[4 * j + 2], v.v[4 * j + 3], f16 != 0));
  }
}

// ---- loss rows of the pre-training proxy tasks (VLN-DUET/pretrain_src/model/pretrain_cmt.py:150,198-204) -----------------
// out[r] = logsumexp(logits[r, 0:n]) - logits[r, label[r]]          (F.cross_entropy, reduction='none'); one warp per row
__global__ void __launch_bounds__(128) ce_rows_kernel(const float* logits, long long ld, const int64_t* labels, int n,
                                                      float* out, long long rows) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const float* x = logits + row * ld;
  float mx = -INFINITY;
  for (int c = lane; c < n; c += 32) mx = fmaxf(mx, x[c]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int c = lane; c < n; c += 32) sum += expf(x[c] - mx);
  sum = warp_sum(sum);
  if (lane == 0) out[row] = mx + logf(sum) - x[labels[row]];
}
// out[r] = sum_c t[r, c] * (log t[r, c] - log_softmax(logits[r])[c]), terms with t == 0 dropped   (F.kl_div(..., 'none').sum(1))
__global__ void __launch_bounds__(128) kl_rows_kernel(const float* logits, long long ld, const float* targets, long long ldt, int n,
                                                      float* out, long long rows) {
  pdl_enter();
  ROW_INDEX();
  if (row >= rows) return;
  const float* x = logits + row * ld;
  const float* t = targets + row * ldt;
  float mx = -INFINITY;
  for (int c = lane; c < n; c += 32) mx = fmaxf(mx, x[c]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int c = lane; c < n; c += 32) sum += expf(x[c] - mx);
  const float lse = mx + logf(warp_sum(sum));
  float acc = 0.f;
  for (int c = lane; c < n; c += 32) {
    const float tc = t[c];
    if (tc > 0.f) acc += tc * (logf(tc) - (x[c] - lse));
  }
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

inline unsigned row_grid(long long rows) { return (unsigned)((rows + ROWS_PER_BLOCK - 1) / ROWS_PER_BLOCK); }
inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }
inline bool make_groups(RowGroups& g, int n_groups, const int32_t* ends, long long rows) {
  if (n_groups < 1 || n_groups > 4 || (n_groups > 1 && !ends)) return false;
  g.n = n_groups;
  for (int i = 0; i < 4; ++i) g.end[i] = 0x7fffffff;
  for (int i = 0; i < n_groups && n_groups > 1; ++i) {
    if (ends[i] <= 0 || (i > 0 && ends[i] <= ends[i - 1])) return false;
    g.end[i] = ends[i];
  }
  (void)rows;
  return true;
}

}  // namespace

#define ST(s) reinterpret_cast<cudaStream_t>(s)

inline bool dt16_ok(int dt) { return dt == VI_DT_BF16 || dt == VI_DT_F16; }

extern "C" int vi_add_ln(const float* a, const float* b, const float* gamma, const float* beta, float eps, float* y32,
                         void* y16, int y16_dtype, int64_t rows, int n_groups, const int32_t* group_row_end, vi_stream_t stream) {
  RowGroups grp;
  VI_CHECK_ARG(dt16_ok(y16_dtype), "vi_add_ln: y16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(make_groups(grp, n_groups, group_row_end, rows), "vi_add_ln: bad row groups");
  VI_CHECK_ARG(a && gamma && beta && (y32 || y16), "vi_add_ln: null operand");
  VI_CHECK_ARG(aligned16(a) && aligned16(b) && aligned16(gamma) && aligned16(beta) && aligned16(y32) && ((uintptr_t)y16 & 7) == 0,
               "vi_add_ln: operands must be 16-byte aligned");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(add_ln_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), a, b, gamma, beta, eps, y32, reinterpret_cast<bf16*>(y16), (int)(y16_dtype == VI_DT_F16), rows, grp));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_add_ln_drop(const float* a, const float* b, const float* gamma, const float* beta, float eps, float* y32, void* y16,
                              int y16_dtype, int64_t rows, int n_groups, const int32_t* group_row_end, float p, const uint32_t* seed,
                              uint32_t site, vi_stream_t stream) {
  RowGroups grp;
  VI_CHECK_ARG(dt16_ok(y16_dtype), "vi_add_ln_drop: y16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(make_groups(grp, n_groups, group_row_end, rows), "vi_add_ln_drop: bad row groups");
  VI_CHECK_ARG(a && gamma && beta && (y32 || y16) && seed && p >= 0.f && p < 1.f, "vi_add_ln_drop: bad operands (0 <= p < 1, device seed)");
  VI_CHECK_ARG(aligned16(a) && aligned16(b) && aligned16(gamma) && aligned16(beta) && aligned16(y32) && ((uintptr_t)y16 & 7) == 0,
               "vi_add_ln_drop: operands must be 16-byte aligned");
  VI_CHECK_ARG(rows * D < (1LL << 32), "vi_add_ln_drop: the dropout mask is indexed with 32 bits");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(add_ln_drop_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), a, b, gamma, beta, eps, y32,
                    reinterpret_cast<bf16*>(y16), (int)(y16_dtype == VI_DT_F16), rows, grp, vi_drop_threshold(p), 1.0f / (1.0f - p), seed, site));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_embed_compose(const vi_embed_args* args, vi_stream_t stream) {
  VI_CHECK_ARG(args, "vi_embed_compose: null args");
  const vi_embed_args& p = *args;
  VI_CHECK_ARG(p.y32 || p.y16, "vi_embed_compose: no output");
  VI_CHECK_ARG(!p.feat || (p.feat_dim > 0 && p.feat_dim <= 16 && p.feat_w), "vi_embed_compose: feat_dim=%d out of range (1..16)", p.feat_dim);
  VI_CHECK_ARG(!p.idx || p.table, "vi_embed_compose: idx without table");
  VI_CHECK_ARG(!p.pos_table || p.pos_period > 0, "vi_embed_compose: pos_table without pos_period");
  VI_CHECK_ARG(!p.a_gamma || p.a_beta, "vi_embed_compose: a_gamma without a_beta");
  VI_CHECK_ARG(!p.feat_gamma || p.feat_beta, "vi_embed_compose: feat_gamma without feat_beta");
  VI_CHECK_ARG(!p.out_gamma || p.out_beta, "vi_embed_compose: out_gamma without out_beta");
  VI_CHECK_ARG(!p.ln2_gamma || (p.ln2_beta && p.y16), "vi_embed_compose: the chained LayerNorm needs ln2_beta and a 16-bit output");
  VI_CHECK_ARG(dt16_ok(p.y16_dtype), "vi_embed_compose: y16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(aligned16(p.a2) && aligned16(p.a3), "vi_embed_compose: a2 / a3 must be 16-byte aligned");
  VI_CHECK_ARG(aligned16(p.a) && aligned16(p.table) && aligned16(p.pos_table) && aligned16(p.const_row) &&
                   aligned16(p.const_row2) && aligned16(p.y32) && ((uintptr_t)p.y16 & 7) == 0,
               "vi_embed_compose: row operands must be 16-byte aligned");
  VI_CHECK_ARG(aligned16(p.feat_b) && aligned16(p.feat_w), "vi_embed_compose: feat_b / feat_w must be 16-byte aligned");
  VI_CHECK_ARG(p.zero_rows >= 0, "vi_embed_compose: negative zero_rows");
  if (p.rows <= 0) return VI_OK;
  const long long blocks = (p.rows + p.zero_rows + EMBED_WARPS - 1) / EMBED_WARPS;
  VI_CUDA(vi_launch(embed_compose_kernel, dim3((unsigned)blocks), dim3(EMBED_WARPS * 32), (size_t)0, ST(stream), p));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_ln_dot(const float* h, const float* gamma, const float* beta, float eps, const float* w, const float* b,
                         float* out, int64_t rows, int n_groups, const int32_t* group_row_end, vi_stream_t stream) {
  RowGroups grp;
  VI_CHECK_ARG(make_groups(grp, n_groups, group_row_end, rows), "vi_ln_dot: bad row groups");
  VI_CHECK_ARG(h && w && out && ((gamma != nullptr) == (beta != nullptr)), "vi_ln_dot: null operand");
  VI_CHECK_ARG(aligned16(h) && aligned16(gamma) && aligned16(beta) && aligned16(w), "vi_ln_dot: operands must be 16-byte aligned");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(ln_dot_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), h, gamma, beta, eps, w, b, out, rows, grp));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_mul_bcast(const float* x, int64_t x_batch_stride, const float* s, int64_t lds, float* y32, void* y16,
                            int y16_dtype, int64_t rows, int rows_per_batch, vi_stream_t stream) {
  VI_CHECK_ARG(dt16_ok(y16_dtype), "vi_mul_bcast: y16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(x && s && (y32 || y16) && rows_per_batch > 0, "vi_mul_bcast: bad operands");
  VI_CHECK_ARG(aligned16(x) && aligned16(s) && lds % 4 == 0 && x_batch_stride % 4 == 0 && aligned16(y32) &&
                   ((uintptr_t)y16 & 7) == 0, "vi_mul_bcast: misaligned operands");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(mul_bcast_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), x, x_batch_stride, s, lds, y32, reinterpret_cast<bf16*>(y16), (int)(y16_dtype == VI_DT_F16), rows,
                                                          rows_per_batch));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_duet_fuse_logits(const float* g_raw, const float* l_raw, const float* fuse_raw, const uint8_t* gmap_masks,
                                   const uint8_t* gmap_visited, const uint8_t* vp_nav_masks, const int32_t* gmap_ids,
                                   const int32_t* cand_ids, float* global_logits, float* local_logits,
                                   float* fused_logits, int B, int G, int P, vi_stream_t stream) {
  VI_CHECK_ARG(g_raw && l_raw && gmap_masks && gmap_visited && vp_nav_masks && gmap_ids && cand_ids &&
                   global_logits && local_logits && fused_logits, "vi_duet_fuse_logits: null operand");
  VI_CHECK_ARG(B > 0 && G > 0 && P > 0, "vi_duet_fuse_logits: empty problem");
  VI_CHECK_ARG(G <= FUSE_MAX && P <= FUSE_MAX, "vi_duet_fuse_logits: G=%d / P=%d exceed %d", G, P, FUSE_MAX);
  VI_CUDA(vi_launch(duet_fuse_logits_kernel, dim3(B), dim3(32), (size_t)(0), ST(stream), g_raw, l_raw, fuse_raw, gmap_masks, gmap_visited, vp_nav_masks, gmap_ids,
                                                   cand_ids, global_logits, local_logits, fused_logits, G, P));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_mask_logits_navtype(const float* raw, const int64_t* nav_types, float* out, int64_t n, vi_stream_t stream) {
  VI_CHECK_ARG(raw && nav_types && out, "vi_mask_logits_navtype: null operand");
  if (n <= 0) return VI_OK;
  VI_CUDA(vi_launch(mask_logits_navtype_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)(0), ST(stream), raw, nav_types, out, n));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_gather_mean(const float* src, const int32_t* offsets, const int32_t* row_idx, float* out32, void* out16,
                              int out16_dtype, int R, vi_stream_t stream) {
  VI_CHECK_ARG(dt16_ok(out16_dtype), "vi_gather_mean: out16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(src && offsets && row_idx && (out32 || out16), "vi_gather_mean: null operand");
  VI_CHECK_ARG(aligned16(src) && aligned16(out32) && ((uintptr_t)out16 & 7) == 0, "vi_gather_mean: misaligned operands");
  if (R <= 0) return VI_OK;
  VI_CUDA(vi_launch(gather_mean_kernel, dim3(row_grid(R)), dim3(128), (size_t)(0), ST(stream), src, offsets, row_idx, out32, reinterpret_cast<bf16*>(out16), (int)(out16_dtype == VI_DT_F16), (long long)R));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_scatter_rows(const float* src, const int32_t* dst_rows, float* dst, int R, vi_stream_t stream) {
  VI_CHECK_ARG(src && dst_rows && dst, "vi_scatter_rows: null operand");
  VI_CHECK_ARG(aligned16(src) && aligned16(dst), "vi_scatter_rows: misaligned operands");
  if (R <= 0) return VI_OK;
  VI_CUDA(vi_launch(scatter_rows_kernel, dim3(row_grid(R)), dim3(128), (size_t)(0), ST(stream), src, dst_rows, dst, R));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_cosine_loss(const float* proj, const float* tgt, float* loss_rows, float* loss_mean, int R,
                              vi_stream_t stream) {
  VI_CHECK_ARG(loss_mean && (R == 0 || (proj && tgt && loss_rows)), "vi_cosine_loss: null operand");
  VI_CHECK_ARG(aligned16(proj) && aligned16(tgt), "vi_cosine_loss: misaligned operands");
  if (R > 0) VI_CUDA(vi_launch(cosine_loss_kernel, dim3(row_grid(R)), dim3(128), (size_t)(0), ST(stream), proj, tgt, loss_rows, R));
  VI_CUDA(vi_launch(mean_kernel, dim3(1), dim3(256), (size_t)(0), ST(stream), loss_rows, loss_mean, R));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_infonce_loss(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                               const int32_t* neg_episode, float temperature, float* loss_rows, float* loss_mean, int R,
                               int n_negs, vi_stream_t stream) {
  // loss_rows doubles as scratch: it must hold R * (n_negs + 1) + R floats (sims first, losses after)
  VI_CHECK_ARG(loss_mean && (R == 0 || (proj && tgt && loss_rows && row_episode)), "vi_infonce_loss: null operand");
  VI_CHECK_ARG(n_negs == 0 || (negs && neg_episode), "vi_infonce_loss: negatives missing");
  VI_CHECK_ARG(temperature > 0.f, "vi_infonce_loss: temperature must be positive");
  float* sims = loss_rows;
  float* rows_out = loss_rows + (long long)R * (n_negs + 1);
  if (R > 0) {
    const long long items = (long long)R * (n_negs + 1);
    VI_CUDA(vi_launch(infonce_sims_kernel, dim3(row_grid(items)), dim3(128), (size_t)(0), ST(stream), proj, tgt, negs, 1.0f / temperature, sims, R, n_negs));
    VI_CUDA(vi_launch(infonce_rows_kernel, dim3(row_grid(R)), dim3(128), (size_t)(0), ST(stream), sims, row_episode, neg_episode, rows_out, R, n_negs));
  }
  VI_CUDA(vi_launch(mean_kernel, dim3(1), dim3(256), (size_t)(0), ST(stream), rows_out, loss_mean, R));
  VI_LAUNCH_CHECK();
  return VI_OK;
}


extern "C" int vi_margin_loss(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                              const int32_t* neg_episode, float margin, float* loss_rows, float* loss_mean, int R, int n_negs,
                              vi_stream_t stream) {
  // loss_rows doubles as scratch exactly as in vi_infonce_loss: R * (n_negs + 1) cosines first, the R losses after
  VI_CHECK_ARG(loss_mean && (R == 0 || (proj && tgt && loss_rows && row_episode)), "vi_margin_loss: null operand");
  VI_CHECK_ARG(n_negs == 0 || (negs && neg_episode), "vi_margin_loss: negatives missing");
  float* sims = loss_rows;
  float* rows_out = loss_rows + (long long)R * (n_negs + 1);
  if (R > 0) {
    const long long items = (long long)R * (n_negs + 1);
    VI_CUDA(vi_launch(infonce_sims_kernel, dim3(row_grid(items)), dim3(128), (size_t)(0), ST(stream), proj, tgt, negs, 1.0f, sims, R, n_negs));
    VI_CUDA(vi_launch(margin_rows_kernel, dim3(row_grid(R)), dim3(128), (size_t)(0), ST(stream), sims, row_episode, neg_episode, margin, rows_out, R, n_negs));
  }
  VI_CUDA(vi_launch(mean_kernel, dim3(1), dim3(256), (size_t)(0), ST(stream), rows_out, loss_mean, R));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_copy_rows(const float* src, int64_t src_batch_stride, int64_t src_row_stride, float* dst32, void* dst16,
                            int dst16_dtype, int64_t dst_batch_stride, int64_t dst_row_stride, int64_t n_batches,
                            int rows_per_batch, vi_stream_t stream) {
  VI_CHECK_ARG(dt16_ok(dst16_dtype), "vi_copy_rows: dst16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(src && (dst32 || dst16) && rows_per_batch > 0, "vi_copy_rows: bad operands");
  VI_CHECK_ARG(aligned16(src) && aligned16(dst32) && ((uintptr_t)dst16 & 7) == 0 && src_batch_stride % 4 == 0 &&
                   src_row_stride % 4 == 0 && dst_batch_stride % 4 == 0 && dst_row_stride % 4 == 0,
               "vi_copy_rows: pointers must be 16-byte aligned and strides multiples of 4 elements");
  const long long rows = (long long)n_batches * rows_per_batch;
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(copy_rows_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), src, src_batch_stride, src_row_stride, dst32,
                                                          reinterpret_cast<bf16*>(dst16), (int)(dst16_dtype == VI_DT_F16), dst_batch_stride,
                                                          dst_row_stride, rows, rows_per_batch));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_cast_h16(const float* src, void* dst, int dst_dtype, int64_t n, vi_stream_t stream) {
  VI_CHECK_ARG(src && dst, "vi_cast_h16: null operand");
  VI_CHECK_ARG(dt16_ok(dst_dtype), "vi_cast_h16: dst_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(aligned16(src) && ((uintptr_t)dst & 7) == 0, "vi_cast_h16: misaligned operands");
  if (n <= 0) return VI_OK;
  const long long n4 = n / 4;
  const long long threads = n4 > 0 ? n4 : 1;
  VI_CUDA(vi_launch(cast_bf16_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), (size_t)(0), ST(stream), src, reinterpret_cast<bf16*>(dst), (int)(dst_dtype == VI_DT_F16), n4, n));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_gather_rows(const void* store, int store_dtype, int64_t ld_store, int64_t n_store_rows, const int32_t* idx,
                              int64_t n_rows, int F, float* dst32, void* dst16, int dst16_dtype, float drop_p,
                              const uint32_t* drop_seed, uint32_t drop_site, vi_stream_t stream) {
  VI_CHECK_ARG(store_dtype == VI_DT_F32 || dt16_ok(store_dtype), "vi_gather_rows: store_dtype must be VI_DT_F32, VI_DT_F16 or VI_DT_BF16");
  VI_CHECK_ARG(!dst16 || dt16_ok(dst16_dtype), "vi_gather_rows: dst16_dtype must be VI_DT_BF16 or VI_DT_F16");
  if (n_rows <= 0) return VI_OK;                  // an empty selection (e.g. imagination slots of width 0) has no pointers
  VI_CHECK_ARG((store || n_store_rows == 0) && idx && (dst32 || dst16), "vi_gather_rows: null operand");
  VI_CHECK_ARG(F > 0 && F % 8 == 0 && ld_store >= F && ld_store % 8 == 0 && n_store_rows >= 0,
               "vi_gather_rows: F=%d must be a positive multiple of 8, ld_store a multiple of 8 >= F", F);
  VI_CHECK_ARG(aligned16(store) && aligned16(dst32) && aligned16(dst16), "vi_gather_rows: operands must be 16-byte aligned");
  VI_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_seed), "vi_gather_rows: 0 <= drop_p < 1, with a device seed");
  const uint32_t thresh = vi_drop_threshold(drop_p);
  const float scale = 1.0f / (1.0f - drop_p);
  const uint32_t* seed = drop_p > 0.f ? drop_seed : nullptr;
  const dim3 grid((unsigned)((n_rows + 7) / 8));
  bf16* d16 = reinterpret_cast<bf16*>(dst16);
  const int f16 = dst16_dtype == VI_DT_F16;
  if (store_dtype == VI_DT_F32)
    VI_CUDA(vi_launch(gather_rows_kernel<float>, grid, dim3(256), (size_t)0, ST(stream), reinterpret_cast<const float*>(store),
                      (long long)ld_store, (long long)n_store_rows, idx, (long long)n_rows, F, dst32, d16, f16, thresh, scale, seed, drop_site));
  else if (store_dtype == VI_DT_F16)
    VI_CUDA(vi_launch(gather_rows_kernel<__half>, grid, dim3(256), (size_t)0, ST(stream), reinterpret_cast<const __half*>(store),
                      (long long)ld_store, (long long)n_store_rows, idx, (long long)n_rows, F, dst32, d16, f16, thresh, scale, seed, drop_site));
  else
    VI_CUDA(vi_launch(gather_rows_kernel<bf16>, grid, dim3(256), (size_t)0, ST(stream), reinterpret_cast<const bf16*>(store),
                      (long long)ld_store, (long long)n_store_rows, idx, (long long)n_rows, F, dst32, d16, f16, thresh, scale, seed, drop_site));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_ce_rows(const float* logits, int64_t ld, const int64_t* labels, int n_cols, float* out, int64_t rows,
                          vi_stream_t stream) {
  VI_CHECK_ARG(logits && labels && out && n_cols > 0 && ld >= n_cols, "vi_ce_rows: bad operands");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(ce_rows_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), logits, (long long)ld, labels, n_cols, out, (long long)rows));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_kl_rows(const float* logits, int64_t ld, const float* targets, int64_t ldt, int n_cols, float* out, int64_t rows,
                          vi_stream_t stream) {
  VI_CHECK_ARG(logits && targets && out && n_cols > 0 && ld >= n_cols && ldt >= n_cols, "vi_kl_rows: bad operands");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(kl_rows_kernel, dim3(row_grid(rows)), dim3(128), (size_t)(0), ST(stream), logits, (long long)ld, targets, (long long)ldt, n_cols, out,
                    (long long)rows));
  VI_LAUNCH_CHECK();
  return VI_OK;
}
