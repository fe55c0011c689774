// vi_bwd.cu - backward-pass kernels of the navigation hot path (fine-tuning, BASELINE.json cfg-4).
//
// The dense gradients (dgrad / wgrad) reuse the tcgen05 GEMM of vi_gemm_tc.cu on transposed operands; this file
// holds everything around them: transposes, bias / LayerNorm parameter reductions, LayerNorm / GELU / ReLU input
// gradients, the attention backward, gather / scatter adjoints, and the adjoints of the logit heads and of the
// alignment loss.  Reductions over rows are deterministic (fixed summation order, no floating-point atomics) except
// where noted.  Reference semantics: torch.autograd of the reference modules (VLN-DUET/map_nav_src/models/
// vilmodel.py, transformer.py; VLN-HAMT/finetune_src/models/vilmodel_cmt.py).
#include "vi_common.cuh"

namespace {

constexpr int D = VI_HIDDEN;

template <typename T> __device__ __forceinline__ float ldf(const T* p, long long i) { return to_f32<T>(p[i]); }

struct RowGroups {
  int n;
  int end[4];
};
__device__ __forceinline__ int group_of_row(const RowGroups& g, long long row) {
  int i = 0;
  while (i < g.n - 1 && row >= g.end[i]) ++i;
  return i;
}

// ---------------------------------------------------------------------------------------------
// dst[c, r] = src[r, c]  (rows x cols -> cols x ldd, columns r >= rows of dst are zero up to pad_rows)
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) transpose_kernel(const T* src, long long ld, T* __restrict__ dst,
                                                        long long ldd, int rows, int cols, int pad_rows) {
  pdl_enter();
  __shared__ T tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 x 8
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + 8 * i, c = c0 + tx;
    tile[ty + 8 * i][tx] = (r < rows && c < cols) ? src[(long long)r * ld + c] : from_f32<T>(0.f);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + 8 * i, r = r0 + tx;
    if (c < cols && r < pad_rows) dst[(long long)c * ldd + r] = tile[tx][ty + 8 * i];
  }
}

// ---------------------------------------------------------------------------------------------
// Column reductions over rows, deterministic and parallel over the rows: stage 1 reduces RED_CHUNK-row chunks into a
// caller-provided scratch [n_out][n_chunks][cols]; stage 2 sums the chunks of each output (of each row group) in a
// fixed order.  Row groups end on multiples of 128 rows (host contract), so a chunk never straddles two groups.
// ---------------------------------------------------------------------------------------------
constexpr int RED_CHUNK = 128;

__device__ __forceinline__ float2 ld2f(const float* p) { return *reinterpret_cast<const float2*>(p); }
__device__ __forceinline__ float2 ld2f(const bf16* p) {
  const __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(p);
  return __bfloat1622float2(t);
}

// out[c] = sum_r x[r, c]; grid (cols / 64, n_chunks), 256 threads: warp w takes rows w, w+8, ... of the chunk, a lane 2 columns
template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const T* x, long long ld, float* __restrict__ part,
                                                             long long rows, int cols) {
  pdl_enter();
  __shared__ float2 red[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + 2 * lane;
  const long long r0 = (long long)blockIdx.y * RED_CHUNK;
  const long long r1 = r0 + RED_CHUNK < rows ? r0 + RED_CHUNK : rows;
  float2 s = make_float2(0.f, 0.f);
  if (c < cols)
    for (long long r = r0 + warp; r < r1; r += 8) {
      const float2 v = ld2f(x + r * ld + c);
      s.x += v.x; s.y += v.y;
    }
  red[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && c < cols) {
    float2 t = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) { t.x += red[i][lane].x; t.y += red[i][lane].y; }
    *reinterpret_cast<float2*>(part + (long long)blockIdx.y * cols + c) = t;
  }
}

// out[o][g][c] = sum over the chunks of group g of part[o][chunk][c]; grid (ceil(cols / 256), n_groups, n_out)
__global__ void __launch_bounds__(256) chunk_sum_kernel(const float* part, float* __restrict__ out, int n_chunks,
                                                        int cols, long long rows, const RowGroups grp, long long out_stride) {
  pdl_enter();
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= cols) return;
  const int gi = blockIdx.y, o = blockIdx.z;
  const long long g0 = gi == 0 ? 0 : grp.end[gi - 1];
  long long g1 = gi == grp.n - 1 ? rows : grp.end[gi];
  if (g1 > rows) g1 = rows;
  const int k0 = (int)(g0 / RED_CHUNK), k1 = (int)((g1 + RED_CHUNK - 1) / RED_CHUNK);
  const float* pp = part + ((long long)o * n_chunks) * cols + c;
  float t = 0.f;
  for (int k = k0; k < k1; ++k) t += pp[(long long)k * cols];
  out[o * out_stride + (long long)gi * cols + c] = t;
}

// ---------------------------------------------------------------------------------------------
// elementwise activations on [rows, cols] views
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_grad(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
  return cdf + x * pdf;
}
// The 16-bit instances (results rounded to 8 mantissa bits) use erf(z) = 1 - (a1 t + ... + a5 t^5) exp(-z^2), t = 1 / (1 + p z)
// (Abramowitz & Stegun 7.1.26, |error| <= 1.5e-7): one MUFU.RCP + one MUFU.EX2 + a dozen FMAs per element, and the exponential
// is the one the density needs anyway - erff + expf made these kernels instruction-bound (ncu: 23 us for 41 MB).  The fp32
// instances (check mode) keep erff / expf.
__device__ __forceinline__ void gelu_terms(float x, float& cdf, float& e) {
  const float ax = fabsf(x);
  float ex;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex) : "f"(x * x * -0.72134752044448170368f));       // exp(-x^2 / 2)
  const float t = __fdividef(1.0f, fmaf(ax, 0.3275911f * 0.70710678118654752440f, 1.0f));
  float q = fmaf(t, 1.061405429f, -1.453152027f);
  q = fmaf(q, t, 1.421413741f);
  q = fmaf(q, t, -0.284496736f);
  q = fmaf(q, t, 0.254829592f);
  const float h = 0.5f * q * t * ex;                                                           // 0.5 * (1 - erf(|x| / sqrt 2))
  cdf = x >= 0.f ? 1.0f - h : h;
  e = ex;
}
__device__ __forceinline__ float gelu_fast(float x) {
  float cdf, e;
  gelu_terms(x, cdf, e);
  return x * cdf;
}
__device__ __forceinline__ float gelu_grad_fast(float x) {
  float cdf, e;
  gelu_terms(x, cdf, e);
  return fmaf(x * 0.39894228040143267794f, e, cdf);
}
template <typename T> __device__ __forceinline__ float gelu_fwd_t(float x) { return sizeof(T) == 2 ? gelu_fast(x) : gelu_erf(x); }
template <typename T> __device__ __forceinline__ float gelu_grad_t(float x) { return sizeof(T) == 2 ? gelu_grad_fast(x) : gelu_grad(x); }
// 8 elements per thread (16-byte accesses for bf16, 2 x 16 for fp32); n is a multiple of 8 on this path (768 / 3072 wide
// rows); a scalar tail covers anything else
template <typename T> struct Vec8;
template <> struct Vec8<bf16> {
  uint4 raw;
  __device__ __forceinline__ void load(const bf16* p) { raw = *reinterpret_cast<const uint4*>(p); }
  __device__ __forceinline__ void store(bf16* p) const { *reinterpret_cast<uint4*>(p) = raw; }
  __device__ __forceinline__ void get(float (&f)[8]) const {
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
      f[2 * i] = t.x; f[2 * i + 1] = t.y;
    }
  }
  __device__ __forceinline__ void set(const float (&f)[8]) {
    raw.x = pack_bf16x2(f[0], f[1]); raw.y = pack_bf16x2(f[2], f[3]);
    raw.z = pack_bf16x2(f[4], f[5]); raw.w = pack_bf16x2(f[6], f[7]);
  }
};
template <> struct Vec8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p) { a = *reinterpret_cast<const float4*>(p); b = *reinterpret_cast<const float4*>(p + 4); }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = a; *reinterpret_cast<float4*>(p + 4) = b; }
  __device__ __forceinline__ void get(float (&f)[8]) const {
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
  __device__ __forceinline__ void set(const float (&f)[8]) {
    a = make_float4(f[0], f[1], f[2], f[3]); b = make_float4(f[4], f[5], f[6], f[7]);
  }
};

template <typename T>
__global__ void __launch_bounds__(256) act_fwd_kernel(const T* x, T* __restrict__ y, long long n, int act) {
  pdl_enter();
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i >= n) return;
  if (i + 8 <= n) {
    Vec8<T> v;
    v.load(x + i);
    float f[8];
    v.get(f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = act == VI_EPI_GELU ? gelu_fwd_t<T>(f[j]) : fmaxf(f[j], 0.f);
    v.set(f);
    v.store(y + i);
  } else {
    for (long long j = i; j < n; ++j) {
      const float v = ldf(x, j);
      y[j] = from_f32<T>(act == VI_EPI_GELU ? gelu_fwd_t<T>(v) : fmaxf(v, 0.f));
    }
  }
}
// dx = dy * act'(x)
template <typename T>
__global__ void __launch_bounds__(256) act_bwd_kernel(const T* x, const T* dy, T* __restrict__ dx,
                                                      long long n, int act) {
  pdl_enter();
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i >= n) return;
  if (i + 8 <= n) {
    Vec8<T> vx, vg;
    vx.load(x + i);
    vg.load(dy + i);
    float f[8], g[8];
    vx.get(f);
    vg.get(g);
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] = act == VI_EPI_GELU ? g[j] * gelu_grad_t<T>(f[j]) : (f[j] > 0.f ? g[j] : 0.f);
    vg.set(g);
    vg.store(dx + i);
  } else {
    for (long long j = i; j < n; ++j) {
      const float v = ldf(x, j), g = ldf(dy, j);
      dx[j] = from_f32<T>(act == VI_EPI_GELU ? g * gelu_grad_t<T>(v) : (v > 0.f ? g : 0.f));
    }
  }
}

// y = x * keep / (1 - p); 8 elements per thread, the mask is a pure function of (element index, seed, site)
template <typename T>
__global__ void __launch_bounds__(256) dropout_kernel(const T* x, T* __restrict__ y, long long n, uint32_t thresh, float scale,
                                                      const uint32_t* seed, uint32_t site) {
  pdl_enter();
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i >= n) return;
  const uint32_t key = vi_drop_key(seed, site);
  if (i + 8 <= n) {
    Vec8<T> v;
    v.load(x + i);
    float f[8];
    v.get(f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = vi_hash32((uint32_t)(i + j), key) >= thresh ? f[j] * scale : 0.f;
    v.set(f);
    v.store(y + i);
  } else {
    for (long long j = i; j < n; ++j) y[j] = from_f32<T>(vi_hash32((uint32_t)j, key) >= thresh ? ldf(x, j) * scale : 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm backward.  y = LN(a [+ b]) * gamma + beta;  dy = dy32 [+ dy16].
//   dx[r] = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma      (one warp per row)
//   dgamma[c] = sum_r dy * xhat,  dbeta[c] = sum_r dy;  stats[r] = {mean, rstd}
// ---------------------------------------------------------------------------------------------

// dx AND the parameter-gradient partials in ONE pass over the rows: a CTA of
// 8 warps owns chunk_rows = 8 / 16 / 32 consecutive rows (1 / 2 / 4 per warp), every lane keeps the dgamma / dbeta contributions of its
// 24 columns in registers, the 8 warps are summed through shared memory in a fixed order and the chunk's partial row goes to
// part[2][n_chunks][768]; ln_param_sum_kernel then adds the chunks of each row group (fixed order: deterministic).
// The chunk is sized by the row count (ln_chunk_rows): the streams of this path have 1.3k - 5k rows, and at 32 rows per CTA the
// grid was 40 - 160 CTAs of 8 warps walking 4 dependent row round trips each on a 148-SM part.
constexpr int LN_CHUNK_MAX = 32;
static int ln_chunk_rows(int64_t rows, int64_t scratch_elems) {
  int chunk = rows <= 296 * 8 ? 8 : rows <= 296 * 16 ? 16 : LN_CHUNK_MAX;
  while (chunk < LN_CHUNK_MAX && (int64_t)2 * ((rows + chunk - 1) / chunk) * D > scratch_elems) chunk *= 2;     // caller's workspace decides
  return chunk;
}
// DropArgs: the forward pass normalised dropout(a) + b (vi_add_ln_drop); then dxa16 receives dropout(dx) - the gradient of a - as the
// 16-bit operand of the weight / input gradient GEMMs of the dense layer that produced a, and dx32 stays the gradient of b.
struct DropArgs { uint32_t thresh; float scale; const uint32_t* seed; uint32_t site; bf16* dxa16; };
__global__ void __launch_bounds__(256, 2) ln_bwd_fused_kernel(const float* a, const float* b, const float* gamma, float eps,
                                                           const float* dy32, const bf16* dy16, float* __restrict__ dx32,
                                                           bf16* __restrict__ dx16, float* __restrict__ stats,
                                                           float* __restrict__ part, long long rows, int n_chunks,
                                                           int chunk_rows, const RowGroups grp, const DropArgs dr) {
  pdl_enter();
  const bool drop = dr.seed != nullptr;
  const uint32_t dkey = drop ? vi_drop_key(dr.seed, dr.site) : 0u;
  __shared__ float red[8][D];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long r0 = (long long)blockIdx.x * chunk_rows;
  float ag[24], ab[24];
#pragma unroll
  for (int i = 0; i < 24; ++i) { ag[i] = 0.f; ab[i] = 0.f; }
  const float* gm_base = gamma + group_of_row(grp, r0) * D;         // a chunk never straddles two row groups
  for (int it = 0; it < chunk_rows / 8; ++it) {
    const long long row = r0 + it * 8 + warp;
    if (row >= rows) break;
    float x[24], dv[24];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const int c = (lane + 32 * j) * 4;
      float4 t = *reinterpret_cast<const float4*>(a + row * D + c);
      if (drop) {
        const uint32_t e0 = (uint32_t)(row * D) + (uint32_t)c;
        t.x = vi_hash32(e0, dkey) >= dr.thresh ? t.x * dr.scale : 0.f;
        t.y = vi_hash32(e0 + 1, dkey) >= dr.thresh ? t.y * dr.scale : 0.f;
        t.z = vi_hash32(e0 + 2, dkey) >= dr.thresh ? t.z * dr.scale : 0.f;
        t.w = vi_hash32(e0 + 3, dkey) >= dr.thresh ? t.w * dr.scale : 0.f;
      }
      if (b) {
        const float4 u = *reinterpret_cast<const float4*>(b + row * D + c);
        t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
      }
      x[4 * j] = t.x; x[4 * j + 1] = t.y; x[4 * j + 2] = t.z; x[4 * j + 3] = t.w;
      s += t.x + t.y + t.z + t.w;
      float4 d4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (dy32) d4 = *reinterpret_cast<const float4*>(dy32 + row * D + c);
      if (dy16) {
        const uint2 h = *reinterpret_cast<const uint2*>(dy16 + row * D + c);
        const float2 h0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&h.x));
        const float2 h1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&h.y));
        d4.x += h0.x; d4.y += h0.y; d4.z += h1.x; d4.w += h1.y;
      }
      dv[4 * j] = d4.x; dv[4 * j + 1] = d4.y; dv[4 * j + 2] = d4.z; dv[4 * j + 3] = d4.w;
    }
    const float mean = warp_sum(s) * (1.0f / D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) { const float d = x[i] - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const float4 gm = *reinterpret_cast<const float4*>(gm_base + (lane + 32 * j) * 4);
      const float gmv[4] = {gm.x, gm.y, gm.z, gm.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float xh = (x[4 * j + e] - mean) * rstd;
        const float gg = dv[4 * j + e] * gmv[e];
        x[4 * j + e] = xh;
        sg += gg;
        sgx = fmaf(gg, xh, sgx);
        ag[4 * j + e] = fmaf(dv[4 * j + e], xh, ag[4 * j + e]);
        ab[4 * j + e] += dv[4 * j + e];
      }
    }
    const float mg = warp_sum(sg) * (1.0f / D), mgx = warp_sum(sgx) * (1.0f / D);
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const int c = (lane + 32 * j) * 4;
      const float4 gm = *reinterpret_cast<const float4*>(gm_base + c);      // dy * gamma again (an L1 hit) instead of 24 live registers
      const float gmv[4] = {gm.x, gm.y, gm.z, gm.w};
      float o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = rstd * (dv[4 * j + e] * gmv[e] - mg - x[4 * j + e] * mgx);
      if (dx32) *reinterpret_cast<float4*>(dx32 + row * D + c) = make_float4(o[0], o[1], o[2], o[3]);
      if (dx16) *reinterpret_cast<uint2*>(dx16 + row * D + c) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
      if (dr.dxa16) {
        if (drop) {
          const uint32_t e0 = (uint32_t)(row * D) + (uint32_t)c;
#pragma unroll
          for (int e = 0; e < 4; ++e) o[e] = vi_hash32(e0 + e, dkey) >= dr.thresh ? o[e] * dr.scale : 0.f;
        }
        *reinterpret_cast<uint2*>(dr.dxa16 + row * D + c) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
      }
    }
    if (lane == 0) { stats[2 * row] = mean; stats[2 * row + 1] = rstd; }
  }
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const int c = (lane + 32 * j) * 4;
      const float* v = pass ? ab : ag;
      *reinterpret_cast<float4*>(&red[warp][c]) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += 256) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += red[w][c];
      part[((long long)pass * n_chunks + blockIdx.x) * D + c] = t;
    }
  }
}
// dgamma[g][c] / dbeta[g][c] = sum over the chunks of group g; grid (768 / 128, n_groups, 2), 256 threads = 32 lanes of four
// columns x 8 chunk lanes: lane k adds the chunks k0 + k, k0 + k + 8, ... (two loads in flight), then the 8 lanes are added in
// order - a fixed order for a given chunk size, so the result is deterministic.
__global__ void __launch_bounds__(256) ln_param_sum_kernel(const float* part, float* dgamma, float* dbeta, int n_chunks,
                                                           int chunk_rows, long long rows, const RowGroups grp, int accumulate) {
  pdl_enter();
  __shared__ float4 red[8][32];
  const int cl = threadIdx.x & 31, kl = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + cl * 4;
  const int gi = blockIdx.y, o = blockIdx.z;
  const long long g0 = gi == 0 ? 0 : grp.end[gi - 1];
  long long g1 = gi == grp.n - 1 ? rows : grp.end[gi];
  if (g1 > rows) g1 = rows;
  const int k0 = (int)(g0 / chunk_rows), k1 = (int)((g1 + chunk_rows - 1) / chunk_rows);
  const float* pp = part + ((long long)o * n_chunks) * D + c;
  float4 t0 = make_float4(0.f, 0.f, 0.f, 0.f), t1 = t0;
  int k = k0 + kl;
  for (; k + 8 < k1; k += 16) {
    const float4 u = *reinterpret_cast<const float4*>(pp + (long long)k * D);
    const float4 v = *reinterpret_cast<const float4*>(pp + (long long)(k + 8) * D);
    t0.x += u.x; t0.y += u.y; t0.z += u.z; t0.w += u.w;
    t1.x += v.x; t1.y += v.y; t1.z += v.z; t1.w += v.w;
  }
  if (k < k1) {
    const float4 u = *reinterpret_cast<const float4*>(pp + (long long)k * D);
    t0.x += u.x; t0.y += u.y; t0.z += u.z; t0.w += u.w;
  }
  red[kl][cl] = make_float4(t0.x + t1.x, t0.y + t1.y, t0.z + t1.z, t0.w + t1.w);
  __syncthreads();
  if (kl == 0) {
    float4 t = red[0][cl];
#pragma unroll
    for (int w = 1; w < 8; ++w) { const float4 u = red[w][cl]; t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
    float4* dst = reinterpret_cast<float4*>((o ? dbeta : dgamma) + (long long)gi * D + c);
    if (accumulate) { const float4 u = *dst; t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
    *dst = t;
  }
}

// ---------------------------------------------------------------------------------------------
// small-feature linear  t = feat W^T + b  (feat_dim <= 16):  dW[c, k] = sum_r dt[r, c] feat[r, k], db[c] = sum_r dt[r, c]
// stage 1: part[17][n_chunks][768] (k = 16 is the bias), grid (768 / 32, n_chunks), 256 threads; stage 2 sums the chunks
// and writes dW (transposed to [768, fd]) / db
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) feat_wgrad_partial_kernel(const float* dt, const float* feat, int fd,
                                                                 float* __restrict__ part, long long rows, int n_chunks) {
  pdl_enter();
  __shared__ float red[8][17][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const long long r0 = (long long)blockIdx.y * RED_CHUNK;
  const long long r1 = r0 + RED_CHUNK < rows ? r0 + RED_CHUNK : rows;
  float acc[17];
#pragma unroll
  for (int k = 0; k < 17; ++k) acc[k] = 0.f;
  for (long long r = r0 + ty; r < r1; r += 8) {
    const float d = dt[r * D + c];
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < fd) acc[k] = fmaf(d, (*(feat + r * fd + k)), acc[k]);
    acc[16] += d;
  }
#pragma unroll
  for (int k = 0; k < 17; ++k) red[ty][k][tx] = acc[k];
  __syncthreads();
  if (ty == 0) {
    for (int k = 0; k < 17; ++k) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red[i][k][tx];
      part[((long long)k * n_chunks + blockIdx.y) * D + c] = t;
    }
  }
}
__global__ void __launch_bounds__(256) feat_wgrad_final_kernel(const float* part, int fd, float* __restrict__ dW,
                                                               float* __restrict__ db, int n_chunks) {
  pdl_enter();
  const int c = blockIdx.x * 256 + threadIdx.x;
  const int k = blockIdx.y;                      // 0..16
  if (c >= D || (k < 16 && k >= fd) || (k == 16 && !db)) return;
  float t = 0.f;
  for (int i = 0; i < n_chunks; ++i) t += part[((long long)k * n_chunks + i) * D + c];
  if (k < 16) dW[(long long)c * fd + k] = t; else db[c] = t;
}

// ---------------------------------------------------------------------------------------------
// dst[idx[r]] += src[r]   (embedding-table adjoint; fp32 atomics: rows may repeat)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) scatter_add_rows_kernel(const float* src, const int64_t* idx,
                                                               float* __restrict__ dst, long long rows, int period) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const long long d = idx ? idx[row] : (row % period);
  for (int c = lane; c < D; c += 32) atomicAdd(dst + d * D + c, src[row * D + c]);
}

// ---------------------------------------------------------------------------------------------
// out[r] = x[r] . w + b  adjoint:  dx[r, :] = dout[r] * w[g],  dw[g, c] = sum_r dout[r] x[r, c],  db[g] = sum_r dout[r]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rowdot_bwd_dx_kernel(const float* dout, const float* w,
                                                            float* __restrict__ dx, long long rows, const RowGroups grp) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* wg = w + group_of_row(grp, row) * D;
  const float g = dout[row];
  for (int c = lane; c < D; c += 32) dx[row * D + c] = g * wg[c];
}
// stage 1 of dw[g, c] = sum_r dout[r] x[r, c], db[g] = sum_r dout[r]: part[2][n_chunks][768] (the bias partial is replicated
// over the columns so that stage 2 is the shared chunk_sum_kernel); grid (768 / 64, n_chunks)
__global__ void __launch_bounds__(256) rowdot_bwd_w_partial_kernel(const float* dout, const float* x,
                                                                   float* __restrict__ part, long long rows, int n_chunks) {
  pdl_enter();
  __shared__ float2 rw[8][32];
  __shared__ float rbias[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + 2 * lane;
  const long long r0 = (long long)blockIdx.y * RED_CHUNK;
  const long long r1 = r0 + RED_CHUNK < rows ? r0 + RED_CHUNK : rows;
  float2 sw = make_float2(0.f, 0.f);
  float sb = 0.f;
  for (long long r = r0 + warp; r < r1; r += 8) {
    const float g = dout[r];
    const float2 v = ld2f(x + r * D + c);
    sw.x = fmaf(g, v.x, sw.x);
    sw.y = fmaf(g, v.y, sw.y);
    sb += g;
  }
  rw[warp][lane] = sw;
  if (lane == 0) rbias[warp] = sb;
  __syncthreads();
  if (warp == 0) {
    float2 t = make_float2(0.f, 0.f);
    float u = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { t.x += rw[i][lane].x; t.y += rw[i][lane].y; u += rbias[i]; }
    *reinterpret_cast<float2*>(part + (long long)blockIdx.y * D + c) = t;
    *reinterpret_cast<float2*>(part + ((long long)n_chunks + blockIdx.y) * D + c) = make_float2(u, u);
  }
}

// ---------------------------------------------------------------------------------------------
// attention backward, one CTA (8 warps) per (episode, head); fp32 arithmetic on fp32 or bf16 tensors.
//   S = Q K^T / 8 + mask + (w dist + b);  P = softmax(S);  dP = dO V^T;  Dr = rowsum(dO o O);
//   dS = P o (dP - Dr);  dQ = dS K / 8;  dK = dS^T Q / 8;  dV = P^T dO;
//   GASA:  dw += sum dS dist,  db += sum dS  (two fp32 atomics per CTA).
// K, V and the dK / dV accumulators live in shared memory; each warp walks query rows; the accumulators take
// shared-memory atomics (rows of different warps collide), so dK / dV sums are order-dependent in the last bits.
// ---------------------------------------------------------------------------------------------
struct AttnBwdParams {
  const void* q; long long ldq;
  const void* k; long long ldk;
  const void* v; long long ldv;
  const void* dout; long long ldo;
  void* dq; long long lddq;
  void* dk; long long lddk;
  void* dv; long long lddv;
  const uint8_t* key_mask;
  const float* pair_dist;
  const float* bias_affine;
  float* d_affine;
  int B, H, Lq, Lk, mask_mode;
};

template <typename T>
__global__ void __launch_bounds__(256) attn_bwd_kernel(const AttnBwdParams p) {
  pdl_enter();
  extern __shared__ __align__(16) float sm[];
  const int Lk = p.Lk;
  float* Ks = sm;                        // [Lk][65]
  float* Vs = Ks + (size_t)Lk * 65;      // [Lk][65]
  float* dKs = Vs + (size_t)Lk * 65;     // [Lk][64]
  float* dVs = dKs + (size_t)Lk * 64;    // [Lk][64]
  float* madd = dVs + (size_t)Lk * 64;   // [Lk]
  float* wbuf = madd + Lk;               // per warp: q[64], do[64], prob[Lk], ds[Lk]
  const int b = blockIdx.y, h = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const T* kg = reinterpret_cast<const T*>(p.k) + (long long)b * Lk * p.ldk + h * 64;
  const T* vg = reinterpret_cast<const T*>(p.v) + (long long)b * Lk * p.ldv + h * 64;
  for (int e = tid; e < Lk * 64; e += 256) {
    const int key = e >> 6, d = e & 63;
    Ks[(size_t)key * 65 + d] = ldf(kg, (long long)key * p.ldk + d);
    Vs[(size_t)key * 65 + d] = ldf(vg, (long long)key * p.ldv + d);
    dKs[e] = 0.f;
    dVs[e] = 0.f;
  }
  for (int key = tid; key < Lk; key += 256) {
    float m = 0.f;
    if (p.key_mask && !p.key_mask[(long long)b * Lk + key]) m = (p.mask_mode == VI_MASK_NEG_INF) ? -INFINITY : -10000.0f;
    madd[key] = m;
  }
  __syncthreads();
  float bw = 0.f, bb = 0.f;
  if (p.pair_dist) { bw = p.bias_affine[0]; bb = p.bias_affine[1]; }
  float* myq = wbuf + (size_t)warp * (128 + 2 * Lk);
  float* mydo = myq + 64;
  float* prob = mydo + 64;
  float* ds = prob + Lk;
  const T* qg = reinterpret_cast<const T*>(p.q) + (long long)b * p.Lq * p.ldq + h * 64;
  const T* dog = reinterpret_cast<const T*>(p.dout) + (long long)b * p.Lq * p.ldo + h * 64;
  T* dqg = reinterpret_cast<T*>(p.dq) + (long long)b * p.Lq * p.lddq + h * 64;
  float aw = 0.f, ab = 0.f;              // GASA affine gradients of this warp
  for (int r = warp; r < p.Lq; r += 8) {
    myq[lane] = ldf(qg, (long long)r * p.ldq + lane);
    myq[lane + 32] = ldf(qg, (long long)r * p.ldq + lane + 32);
    mydo[lane] = ldf(dog, (long long)r * p.ldo + lane);
    mydo[lane + 32] = ldf(dog, (long long)r * p.ldo + lane + 32);
    __syncwarp();
    const float* pd = p.pair_dist ? p.pair_dist + ((long long)b * p.Lq + r) * Lk : nullptr;
    float mx = -INFINITY;
    for (int key = lane; key < Lk; key += 32) {
      float dot = 0.f, dp = 0.f;
#pragma unroll 16
      for (int d = 0; d < 64; ++d) {
        dot = fmaf(myq[d], Ks[(size_t)key * 65 + d], dot);
        dp = fmaf(mydo[d], Vs[(size_t)key * 65 + d], dp);
      }
      float add = madd[key];
      if (pd) add += fmaf(bw, pd[key], bb);
      const float s = dot * 0.125f + add;
      prob[key] = s;
      ds[key] = dp;                      // dP for now
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    const float mu = (mx == -INFINITY) ? 0.f : mx;
    float sum = 0.f;
    for (int key = lane; key < Lk; key += 32) {
      const float e = expf(prob[key] - mu);
      prob[key] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    // Dr = sum_j P_j dP_j  (= rowsum(dO o O))
    float dr = 0.f;
    for (int key = lane; key < Lk; key += 32) {
      const float pj = prob[key] * inv;
      prob[key] = pj;
      dr = fmaf(pj, ds[key], dr);
    }
    dr = warp_sum(dr);
    for (int key = lane; key < Lk; key += 32) {
      const float g = prob[key] * (ds[key] - dr);
      ds[key] = g;
      if (pd) { aw = fmaf(g, pd[key], aw); ab += g; }
    }
    __syncwarp();
    float q0 = 0.f, q1 = 0.f;
    const float qa = myq[lane] * 0.125f, qb = myq[lane + 32] * 0.125f;
    const float oa = mydo[lane], ob = mydo[lane + 32];
    for (int key = 0; key < Lk; ++key) {
      const float g = ds[key], pj = prob[key];
      q0 = fmaf(g, Ks[(size_t)key * 65 + lane], q0);
      q1 = fmaf(g, Ks[(size_t)key * 65 + lane + 32], q1);
      atomicAdd(dKs + (size_t)key * 64 + lane, g * qa);
      atomicAdd(dKs + (size_t)key * 64 + lane + 32, g * qb);
      atomicAdd(dVs + (size_t)key * 64 + lane, pj * oa);
      atomicAdd(dVs + (size_t)key * 64 + lane + 32, pj * ob);
    }
    dqg[(long long)r * p.lddq + lane] = from_f32<T>(q0 * 0.125f);
    dqg[(long long)r * p.lddq + lane + 32] = from_f32<T>(q1 * 0.125f);
    __syncwarp();
  }
  if (p.pair_dist && p.d_affine) {
    aw = warp_sum(aw);
    ab = warp_sum(ab);
    if (lane == 0) { atomicAdd(p.d_affine, aw); atomicAdd(p.d_affine + 1, ab); }
  }
  __syncthreads();
  T* dkg = reinterpret_cast<T*>(p.dk) + (long long)b * Lk * p.lddk + h * 64;
  T* dvg = reinterpret_cast<T*>(p.dv) + (long long)b * Lk * p.lddv + h * 64;
  for (int e = tid; e < Lk * 64; e += 256) {
    const int key = e >> 6, d = e & 63;
    dkg[(long long)key * p.lddk + d] = from_f32<T>(dKs[e]);
    dvg[(long long)key * p.lddv + d] = from_f32<T>(dVs[e]);
  }
}

// ---------------------------------------------------------------------------------------------
// adjoint of vi_mul_bcast w.r.t. the broadcast row:  ds[b, c] = sum_r dy[b, r, c] * x[b, r, c]   (one CTA per episode)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mul_bcast_bwd_s_kernel(const float* dy, const float* x, float* __restrict__ ds,
                                                              int rows_per_batch) {
  pdl_enter();
  const long long b = blockIdx.x;
  for (int c = threadIdx.x; c < D; c += 256) {
    float t = 0.f;
    for (int r = 0; r < rows_per_batch; ++r) {
      const long long i = (b * rows_per_batch + r) * D + c;
      t = fmaf(dy[i], x[i], t);
    }
    ds[b * D + c] = t;
  }
}

// ---------------------------------------------------------------------------------------------
// adjoint of vi_duet_fuse_logits (one warp per episode, same id matching as the forward kernel)
// ---------------------------------------------------------------------------------------------
constexpr int FUSE_MAX = 512;
__global__ void __launch_bounds__(32) duet_fuse_logits_bwd_kernel(
    const float* g_raw, const float* l_raw, const float* fuse_raw,
    const uint8_t* gmap_masks, const uint8_t* gmap_visited, const uint8_t* vp_nav,
    const int32_t* gmap_ids, const int32_t* cand_ids, const float* d_global,
    const float* d_local, const float* d_fused, float* __restrict__ dg_raw,
    float* __restrict__ dl_raw, float* __restrict__ dfuse_raw, int G, int P) {
  pdl_enter();
  __shared__ float dll[FUSE_MAX];          // gradient w.r.t. the masked local logits
  __shared__ int gid[FUSE_MAX], cid[FUSE_MAX];
  __shared__ uint8_t gvis[FUSE_MAX], cvis[FUSE_MAX];
  __shared__ float dbw_s;
  const int b = blockIdx.x, lane = threadIdx.x;
  const float fw = fuse_raw ? 1.0f / (1.0f + expf(-fuse_raw[b])) : 0.5f;
  for (int v = lane; v < P; v += 32) {
    cid[v] = cand_ids[(long long)b * P + v];
    dll[v] = d_local ? d_local[(long long)b * P + v] : 0.f;
  }
  for (int j = lane; j < G; j += 32) gid[j] = gmap_ids[(long long)b * G + j];
  __syncwarp();
  for (int j = lane; j < G; j += 32) {
    bool in_set = false;
    if (gid[j] != -1)
      for (int k = 0; k < G; ++k) in_set |= (gid[k] == gid[j]) && gid[k] != -1 && gmap_visited[(long long)b * G + k];
    gvis[j] = in_set;
  }
  for (int v = lane; v < P; v += 32) {
    bool in_set = false;
    if (cid[v] != -2)
      for (int k = 0; k < G; ++k) in_set |= (gid[k] == cid[v]) && gid[k] != -1 && gmap_visited[(long long)b * G + k];
    cvis[v] = in_set;
  }
  __syncwarp();
  // fused[j] = global[j] + (j == 0 ? local[0] : hit >= 0 ? local[hit] : bw) -> scatter d_fused into dll / dbw (lane 0, in order)
  float dfw = 0.f;                          // d loss / d fuse weight
  if (lane == 0) {
    float dbw = 0.f;
    for (int j = 0; j < G; ++j) {
      const float df = d_fused ? d_fused[(long long)b * G + j] : 0.f;
      if (j == 0) { dll[0] += df; continue; }
      if (gid[j] == -1 || gvis[j]) continue;
      int hit = -1;
      for (int v = 1; v < P; ++v)
        if (cid[v] != -2 && !cvis[v] && cid[v] == gid[j]) hit = v;
      if (hit >= 0) dll[hit] += df; else dbw += df;
    }
    for (int v = 1; v < P; ++v)
      if (cid[v] != -2 && cvis[v]) dll[v] += dbw;
    dbw_s = dbw;
  }
  __syncwarp();
  for (int v = lane; v < P; v += 32) {
    const long long i = (long long)b * P + v;
    float g = 0.f;
    if (vp_nav[i]) {                        // masked positions are constants (-inf)
      g = dll[v] * (1.0f - fw);
      dfw -= dll[v] * l_raw[i];
    }
    dl_raw[i] = g;
  }
  for (int j = lane; j < G; j += 32) {
    const long long i = (long long)b * G + j;
    float g = 0.f;
    if (!(gmap_visited[i] || !gmap_masks[i])) {
      const float dgl = (d_global ? d_global[i] : 0.f) + (d_fused ? d_fused[i] : 0.f);
      g = dgl * fw;
      dfw += dgl * g_raw[i];
    }
    dg_raw[i] = g;
  }
  dfw = warp_sum(dfw);
  if (lane == 0 && dfuse_raw) dfuse_raw[b] = dfw * fw * (1.0f - fw);
}

// ---------------------------------------------------------------------------------------------
// cosine alignment loss adjoint:  loss = mean_r (1 - cos(p_r, t_r));  dp_r = -(dloss / R) d cos / d p_r
// (torch clamps each norm at eps = 1e-8; the clamp is inactive for non-degenerate rows and is treated as such)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) cosine_loss_bwd_kernel(const float* proj, const float* tgt,
                                                              const float* dloss, float* __restrict__ dproj,
                                                              float* __restrict__ dtgt, long long rows) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= rows) return;
  float a[24], t[24];
  float ab = 0.f, aa = 0.f, bb = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) {
    a[i] = proj[row * D + lane + 32 * i];
    t[i] = tgt[row * D + lane + 32 * i];
    ab = fmaf(a[i], t[i], ab); aa = fmaf(a[i], a[i], aa); bb = fmaf(t[i], t[i], bb);
  }
  ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
  const float na = fmaxf(sqrtf(aa), 1e-8f), nb = fmaxf(sqrtf(bb), 1e-8f);
  const float cosv = ab / (na * nb);
  const float scale = -dloss[0] / (float)rows;
#pragma unroll
  for (int i = 0; i < 24; ++i) {
    if (dproj) dproj[row * D + lane + 32 * i] = scale * (t[i] / (na * nb) - cosv * a[i] / (na * na));
    if (dtgt) dtgt[row * D + lane + 32 * i] = scale * (a[i] / (na * nb) - cosv * t[i] / (nb * nb));
  }
}

// InfoNCE alignment loss adjoint (vilmodel.py:657-687):  loss = mean_r [ logsumexp_{c valid} s_rc - s_r0 ],
// s_rc = cos(p_r, t_c) / tau with t_0 = the row's own noun-phrase mean and t_c (c >= 1) the noun-phrase means of OTHER
// episodes.  With w_rc = softmax_c(s_rc) - [c == 0] and g_rc = dloss w_rc / (R tau) = dloss / dcos_rc:
//     dp_r = sum_c g_rc ( t_c / (|p_r| |t_c|) - cos_rc p_r / |p_r|^2 )
//     dt_r = g_r0 ( p_r / (|p_r| |t_r|) - cos_r0 t_r / |t_r|^2 )                       (dtgt, optional)
// With `gneg` given, g_rc of every negative column (0 for the row's own episode) goes to gneg[r, c - 1] and 1 / |p_r| to
// inv_np[r]: the operands of contrastive_negs_bwd_kernel.  dproj does not depend on either option.
// `sims` is what the forward pass left in its scratch (s_rc for every column, valid or not).  One warp per row.
__global__ void __launch_bounds__(128) infonce_loss_bwd_kernel(const float* proj, const float* tgt, const float* negs,
                                                               const int32_t* row_ep, const int32_t* neg_ep, float inv_t,
                                                               const float* sims, const float* dloss,
                                                               float* __restrict__ dproj, float* __restrict__ dtgt,
                                                               float* __restrict__ gneg, float* __restrict__ inv_np,
                                                               int R, int n_negs, int margin_mode, float margin) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= R) return;
  const int cols = n_negs + 1;
  const float* s = sims + row * cols;
  const int ep = row_ep[row];
  // margin form (H/models/vilmodel_cmt.py:825-856): loss_r = (1 - cos_0) + mean_c relu(margin + cos_c - cos_0) over the admissible
  // negatives, so w_rc = [hinge c active] / count for c >= 1 and w_r0 = -1 - (active hinges) / count   (sims hold plain cosines)
  float mx = s[0];
  float sum = 0.f, cnt = 0.f, nact = 0.f;
  if (margin_mode) {
    for (int c = 1 + lane; c < cols; c += 32)
      if (neg_ep[c - 1] != ep) { cnt += 1.f; nact += (margin + s[c] - s[0] > 0.f) ? 1.f : 0.f; }
    cnt = warp_sum(cnt); nact = warp_sum(nact);
  } else {
    for (int c = 1 + lane; c < cols; c += 32)
      if (neg_ep[c - 1] != ep) mx = fmaxf(mx, s[c]);
    mx = warp_max(mx);
    for (int c = 1 + lane; c < cols; c += 32)
      if (neg_ep[c - 1] != ep) sum += expf(s[c] - mx);
    sum = warp_sum(sum) + expf(s[0] - mx);
  }
  const float inv_sum = 1.0f / sum;
  float a[24], acc[24];
  float aa = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) { a[i] = proj[row * D + lane + 32 * i]; aa = fmaf(a[i], a[i], aa); acc[i] = 0.f; }
  aa = warp_sum(aa);
  const float na = fmaxf(sqrtf(aa), 1e-8f);
  const float scale = dloss[0] * inv_t / (float)R;
  float wcos = 0.f;                                    // sum_c w_rc cos_rc
  for (int c = 0; c < cols; ++c) {
    if (c > 0 && neg_ep[c - 1] == ep) continue;        // warp-uniform
    float w;
    if (margin_mode) {
      w = c == 0 ? -1.f - nact / cnt : ((margin + s[c] - s[0] > 0.f) ? 1.f / cnt : 0.f);
      if (w == 0.f) continue;                          // warp-uniform
    } else {
      w = expf(s[c] - mx) * inv_sum - (c == 0 ? 1.f : 0.f);
    }
    const float* t = c == 0 ? tgt + row * D : negs + (long long)(c - 1) * D;
    float tv[24];
    float bb = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) { tv[i] = t[lane + 32 * i]; bb = fmaf(tv[i], tv[i], bb); }
    bb = warp_sum(bb);
    const float k = w / fmaxf(sqrtf(bb), 1e-8f);
#pragma unroll
    for (int i = 0; i < 24; ++i) acc[i] = fmaf(k, tv[i], acc[i]);
    wcos = fmaf(w, s[c], wcos);                        // s = cos / tau
    if (c == 0 && dtgt) {
      const float nt = fmaxf(sqrtf(bb), 1e-8f), g0 = scale * w, cos0 = s[0] / inv_t;
#pragma unroll
      for (int i = 0; i < 24; ++i) dtgt[row * D + lane + 32 * i] = g0 * (a[i] / (na * nt) - cos0 * tv[i] / (nt * nt));
    }
  }
  wcos /= inv_t;
#pragma unroll
  for (int i = 0; i < 24; ++i) dproj[row * D + lane + 32 * i] = scale * (acc[i] / na - wcos * a[i] / (na * na));
  if (gneg) {
    for (int c = 1 + lane; c < cols; c += 32) {
      float w = 0.f;
      if (neg_ep[c - 1] != ep)
        w = margin_mode ? ((margin + s[c] - s[0] > 0.f) ? 1.f / cnt : 0.f) : expf(s[c] - mx) * inv_sum;
      gneg[row * n_negs + c - 1] = scale * w;
    }
    if (lane == 0) inv_np[row] = 1.0f / na;
  }
}

// Adjoint of the alignment losses w.r.t. the negatives (the noun-phrase means of the other episodes):
//     dneg_n = (1 / |t_n|) sum_r g_rn p_r / |p_r|  -  (sum_r g_rn cos_rn / |t_n|^2) t_n
// with g_rn = gneg[r, n] and 1 / |p_r| = inv_np[r] from infonce_loss_bwd_kernel, cos_rn = cos_scale * sims[r, 1 + n].  The sum
// over rows is G^T P-hat ([n_negs, R] x [R, 768]): a CTA owns NEG_TILE negatives x 256 columns, each thread 4 columns of all
// NEG_TILE negatives, so every row of proj is read once per NEG_TILE negatives.  Rows are summed in a fixed order and every
// output element has one writer: two calls are bit-identical.
constexpr int NEG_TILE = 8, NEG_ROWS = 32;
__global__ void __launch_bounds__(64) contrastive_negs_bwd_kernel(const float* proj, const float* negs, const float* sims,
                                                                  const float* gneg, const float* inv_np, float cos_scale,
                                                                  float* __restrict__ dnegs, int R, int n_negs) {
  pdl_enter();
  __shared__ __align__(16) float wt[NEG_ROWS][NEG_TILE];
  __shared__ float nrm[NEG_TILE], gcos[NEG_TILE];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n0 = blockIdx.x * NEG_TILE;
  const int col = blockIdx.y * 256 + tid * 4;
  const long long cols = n_negs + 1;
  // per negative: |t_n| and sum_r g_rn cos_rn (lane-strided partial sums, then the butterfly: a fixed order)
  for (int k = warp; k < NEG_TILE; k += 2) {
    const int n = n0 + k;
    float tt = 0.f, gc = 0.f;
    if (n < n_negs) {
      for (int i = lane; i < D; i += 32) { const float t = negs[(long long)n * D + i]; tt = fmaf(t, t, tt); }
      for (int r = lane; r < R; r += 32) gc = fmaf(gneg[(long long)r * n_negs + n], sims[r * cols + 1 + n], gc);
    }
    tt = warp_sum(tt); gc = warp_sum(gc);
    if (lane == 0) { nrm[k] = fmaxf(sqrtf(tt), 1e-8f); gcos[k] = gc * cos_scale; }
  }
  float4 acc[NEG_TILE];
#pragma unroll
  for (int k = 0; k < NEG_TILE; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r0 = 0; r0 < R; r0 += NEG_ROWS) {
    __syncthreads();                                   // the previous tile is consumed
    for (int e = tid; e < NEG_ROWS * NEG_TILE; e += 64) {
      const int j = e / NEG_TILE, k = e % NEG_TILE, r = r0 + j, n = n0 + k;
      wt[j][k] = (r < R && n < n_negs) ? gneg[(long long)r * n_negs + n] * inv_np[r] : 0.f;
    }
    __syncthreads();
    const int rows = min(NEG_ROWS, R - r0);
#pragma unroll 4
    for (int j = 0; j < rows; ++j) {
      const float4 p = *reinterpret_cast<const float4*>(proj + (long long)(r0 + j) * D + col);
#pragma unroll
      for (int k = 0; k < NEG_TILE; ++k) {
        const float w = wt[j][k];
        acc[k].x = fmaf(w, p.x, acc[k].x); acc[k].y = fmaf(w, p.y, acc[k].y);
        acc[k].z = fmaf(w, p.z, acc[k].z); acc[k].w = fmaf(w, p.w, acc[k].w);
      }
    }
  }
  __syncthreads();                                     // nrm / gcos
#pragma unroll
  for (int k = 0; k < NEG_TILE; ++k) {
    const int n = n0 + k;
    if (n >= n_negs) break;
    const float inv = 1.0f / nrm[k], coef = gcos[k] * inv * inv;
    const float4 t = *reinterpret_cast<const float4*>(negs + (long long)n * D + col);
    *reinterpret_cast<float4*>(dnegs + (long long)n * D + col) =
        make_float4(acc[k].x * inv - coef * t.x, acc[k].y * inv - coef * t.y, acc[k].z * inv - coef * t.z, acc[k].w * inv - coef * t.w);
  }
}

inline bool make_groups(RowGroups& g, int n_groups, const int32_t* ends) {
  if (n_groups < 1 || n_groups > 4 || (n_groups > 1 && !ends)) return false;
  g.n = n_groups;
  for (int i = 0; i < 4; ++i) g.end[i] = 0x7fffffff;
  for (int i = 0; i < n_groups && n_groups > 1; ++i) {
    if (ends[i] <= 0 || (i > 0 && ends[i] <= ends[i - 1])) return false;
    g.end[i] = ends[i];
  }
  return true;
}
inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace

#define ST(s) reinterpret_cast<cudaStream_t>(s)

// vi_attn_bwd.cu: tensor-core kernel for bf16 operands; returns 1 when the problem does not fit it
int vi_attn_bwd_tc(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* dout,
                   int64_t ldo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                   const uint8_t* key_mask, const float* pair_dist, const float* bias_affine, float* d_affine, int B, int H,
                   int Lq, int Lk, int mask_mode, float drop_p, uint32_t drop_site, const uint32_t* drop_seed, cudaStream_t st);

extern "C" int vi_transpose(const void* src, int64_t ld, void* dst, int64_t ldd, int rows, int cols, int pad_rows, int dtype,
                            vi_stream_t stream) {
  VI_CHECK_ARG(src && dst && rows > 0 && cols > 0 && pad_rows >= rows && ld >= cols && ldd >= pad_rows, "vi_transpose: bad operands");
  dim3 grid((cols + 31) / 32, (pad_rows + 31) / 32);
  if (dtype == VI_DT_BF16)
    VI_CUDA(vi_launch(transpose_kernel<bf16>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const bf16*>(src), (long long)ld,
                      reinterpret_cast<bf16*>(dst), (long long)ldd, rows, cols, pad_rows));
  else
    VI_CUDA(vi_launch(transpose_kernel<float>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const float*>(src), (long long)ld,
                      reinterpret_cast<float*>(dst), (long long)ldd, rows, cols, pad_rows));
  return VI_OK;
}

inline int red_chunks(long long rows) { return (int)((rows + RED_CHUNK - 1) / RED_CHUNK); }
inline RowGroups one_group() {
  RowGroups g;
  g.n = 1;
  for (int i = 0; i < 4; ++i) g.end[i] = 0x7fffffff;
  return g;
}

extern "C" int vi_colsum(const void* x, int64_t ld, int dtype, float* out, int64_t rows, int cols, float* scratch,
                         int64_t scratch_elems, vi_stream_t stream) {
  VI_CHECK_ARG(x && out && scratch && rows > 0 && cols > 0 && ld >= cols, "vi_colsum: bad operands");
  VI_CHECK_ARG(cols % 2 == 0 && ld % 2 == 0 && ((uintptr_t)x & 7) == 0, "vi_colsum: columns / leading dimension must be even, x 8-byte aligned");
  const int nch = red_chunks(rows);
  VI_CHECK_ARG(scratch_elems >= (int64_t)nch * cols, "vi_colsum: scratch too small (%lld < %lld)", (long long)scratch_elems,
               (long long)nch * cols);
  dim3 grid((cols + 63) / 64, nch);
  if (dtype == VI_DT_BF16)
    VI_CUDA(vi_launch(colsum_partial_kernel<bf16>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const bf16*>(x), (long long)ld,
                      scratch, (long long)rows, cols));
  else
    VI_CUDA(vi_launch(colsum_partial_kernel<float>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const float*>(x), (long long)ld,
                      scratch, (long long)rows, cols));
  VI_CUDA(vi_launch(chunk_sum_kernel, dim3((cols + 255) / 256, 1, 1), dim3(256), 0, ST(stream), (const float*)scratch, out, nch, cols,
                    (long long)rows, one_group(), (long long)0));
  return VI_OK;
}

extern "C" int vi_dropout(const void* x, void* y, int64_t n, float p, const uint32_t* seed, uint32_t site, int dtype,
                          vi_stream_t stream) {
  VI_CHECK_ARG(x && y && seed && p >= 0.f && p < 1.f, "vi_dropout: bad operands (0 <= p < 1, seed must be a device pointer)");
  VI_CHECK_ARG((((uintptr_t)x | (uintptr_t)y) & 15) == 0, "vi_dropout: operands must be 16-byte aligned");
  if (n <= 0) return VI_OK;
  const uint32_t thresh = vi_drop_threshold(p);
  const float scale = 1.0f / (1.0f - p);
  dim3 grid((unsigned)((n + 2047) / 2048));
  if (dtype == VI_DT_BF16)
    VI_CUDA(vi_launch(dropout_kernel<bf16>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const bf16*>(x),
                      reinterpret_cast<bf16*>(y), (long long)n, thresh, scale, seed, site));
  else
    VI_CUDA(vi_launch(dropout_kernel<float>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const float*>(x),
                      reinterpret_cast<float*>(y), (long long)n, thresh, scale, seed, site));
  return VI_OK;
}

extern "C" int vi_act_fwd(const void* x, void* y, int64_t n, int act, int dtype, vi_stream_t stream) {
  VI_CHECK_ARG(x && y && (act == VI_EPI_GELU || act == VI_EPI_RELU), "vi_act_fwd: bad operands");
  if (n <= 0) return VI_OK;
  VI_CHECK_ARG((((uintptr_t)x | (uintptr_t)y) & 15) == 0, "vi_act_fwd: operands must be 16-byte aligned");
  dim3 grid((unsigned)((n + 2047) / 2048));
  if (dtype == VI_DT_BF16)
    VI_CUDA(vi_launch(act_fwd_kernel<bf16>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const bf16*>(x),
                      reinterpret_cast<bf16*>(y), (long long)n, act));
  else
    VI_CUDA(vi_launch(act_fwd_kernel<float>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const float*>(x),
                      reinterpret_cast<float*>(y), (long long)n, act));
  return VI_OK;
}

extern "C" int vi_act_bwd(const void* x, const void* dy, void* dx, int64_t n, int act, int dtype, vi_stream_t stream) {
  VI_CHECK_ARG(x && dy && dx && (act == VI_EPI_GELU || act == VI_EPI_RELU), "vi_act_bwd: bad operands");
  if (n <= 0) return VI_OK;
  VI_CHECK_ARG((((uintptr_t)x | (uintptr_t)dy | (uintptr_t)dx) & 15) == 0, "vi_act_bwd: operands must be 16-byte aligned");
  dim3 grid((unsigned)((n + 2047) / 2048));
  if (dtype == VI_DT_BF16)
    VI_CUDA(vi_launch(act_bwd_kernel<bf16>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const bf16*>(x),
                      reinterpret_cast<const bf16*>(dy), reinterpret_cast<bf16*>(dx), (long long)n, act));
  else
    VI_CUDA(vi_launch(act_bwd_kernel<float>, grid, dim3(256), 0, ST(stream), reinterpret_cast<const float*>(x),
                      reinterpret_cast<const float*>(dy), reinterpret_cast<float*>(dx), (long long)n, act));
  return VI_OK;
}

extern "C" int vi_add_ln_drop_bwd(const float* a, const float* b, const float* gamma, float eps, const float* dy32, const void* dy16,
                                  float* dx32, void* dx16, void* dxa16, float* dgamma, float* dbeta, float* stats, int64_t rows,
                                  int n_groups, const int32_t* group_row_end, float* scratch, int64_t scratch_elems, int accumulate,
                                  float p, const uint32_t* seed, uint32_t site, vi_stream_t stream) {
  VI_CHECK_ARG(p >= 0.f && p < 1.f && (p == 0.f || seed), "vi_add_ln_drop_bwd: 0 <= p < 1 and a device seed pointer");
  VI_CHECK_ARG(((uintptr_t)dxa16 & 7) == 0, "vi_add_ln_drop_bwd: dxa16 must be 8-byte aligned");
  VI_CHECK_ARG(p == 0.f || rows * D < (1LL << 32), "vi_add_ln_drop_bwd: dropout needs < 2^32 elements");
  DropArgs dr;
  dr.thresh = vi_drop_threshold(p); dr.scale = 1.0f / (1.0f - p); dr.seed = p > 0.f ? seed : nullptr; dr.site = site;
  dr.dxa16 = reinterpret_cast<bf16*>(dxa16);
  RowGroups grp;
  VI_CHECK_ARG(make_groups(grp, n_groups, group_row_end), "vi_add_ln_drop_bwd: bad row groups");
  for (int g = 0; g + 1 < n_groups; ++g)
    VI_CHECK_ARG(group_row_end[g] % RED_CHUNK == 0, "vi_add_ln_drop_bwd: row groups must end on multiples of %d rows", RED_CHUNK);
  VI_CHECK_ARG(a && gamma && (dy32 || dy16) && (dx32 || dx16) && dgamma && dbeta && stats, "vi_add_ln_drop_bwd: null operand");
  VI_CHECK_ARG(aligned16(a) && aligned16(b) && aligned16(gamma) && aligned16(dy32) && aligned16(dx32) &&
                   ((uintptr_t)dx16 & 7) == 0, "vi_add_ln_drop_bwd: misaligned operands");
  if (rows <= 0) return VI_OK;
  // one pass: dx + per-chunk partials of dgamma / dbeta, then the fixed-order sum of the chunks of every row group
  VI_CHECK_ARG(aligned16(dgamma) && aligned16(dbeta) && aligned16(scratch), "vi_add_ln_drop_bwd: dgamma / dbeta / scratch must be 16-byte aligned");
  const int chunk = scratch ? ln_chunk_rows(rows, scratch_elems) : LN_CHUNK_MAX;
  const int nch = (int)((rows + chunk - 1) / chunk);
  VI_CHECK_ARG(scratch && scratch_elems >= (int64_t)2 * nch * D, "vi_add_ln_drop_bwd: scratch too small (need 2 x ceil(rows / %d) x %d floats)",
               LN_CHUNK_MAX, D);
  VI_CUDA(vi_launch(ln_bwd_fused_kernel, dim3((unsigned)nch), dim3(256), 0, ST(stream), a, b, gamma, eps, dy32,
                    reinterpret_cast<const bf16*>(dy16), dx32, reinterpret_cast<bf16*>(dx16), stats, scratch, (long long)rows, nch, chunk,
                    grp, dr));
  VI_CUDA(vi_launch(ln_param_sum_kernel, dim3(D / 128, n_groups, 2), dim3(256), 0, ST(stream), (const float*)scratch, dgamma, dbeta, nch,
                    chunk, (long long)rows, grp, (int)(accumulate != 0)));
  return VI_OK;
}

extern "C" int vi_feat_wgrad(const float* dt, const float* feat, int feat_dim, float* dW, float* db, int64_t rows,
                             float* scratch, int64_t scratch_elems, vi_stream_t stream) {
  VI_CHECK_ARG(dt && feat && dW && feat_dim > 0 && feat_dim <= 16 && rows > 0, "vi_feat_wgrad: bad operands");
  const int nch = red_chunks(rows);
  VI_CHECK_ARG(scratch && scratch_elems >= (int64_t)17 * nch * D, "vi_feat_wgrad: scratch too small");
  VI_CUDA(vi_launch(feat_wgrad_partial_kernel, dim3(D / 32, nch), dim3(256), 0, ST(stream), dt, feat, feat_dim, scratch,
                    (long long)rows, nch));
  VI_CUDA(vi_launch(feat_wgrad_final_kernel, dim3(D / 256, 17), dim3(256), 0, ST(stream), (const float*)scratch, feat_dim, dW, db, nch));
  return VI_OK;
}

extern "C" int vi_scatter_add_rows(const float* src, const int64_t* idx, int period, float* dst, int64_t rows, vi_stream_t stream) {
  VI_CHECK_ARG(src && dst && (idx || period > 0), "vi_scatter_add_rows: bad operands");
  if (rows <= 0) return VI_OK;
  VI_CUDA(vi_launch(scatter_add_rows_kernel, dim3((unsigned)((rows + 3) / 4)), dim3(128), 0, ST(stream), src, idx, dst,
                    (long long)rows, period));
  return VI_OK;
}

extern "C" int vi_rowdot_bwd(const float* dout, const float* x, const float* w, float* dx, float* dw, float* db_cols, int64_t rows,
                             int n_groups, const int32_t* group_row_end, float* scratch, int64_t scratch_elems,
                             vi_stream_t stream) {
  RowGroups grp;
  VI_CHECK_ARG(make_groups(grp, n_groups, group_row_end), "vi_rowdot_bwd: bad row groups");
  for (int g = 0; g + 1 < n_groups; ++g)
    VI_CHECK_ARG(group_row_end[g] % RED_CHUNK == 0, "vi_rowdot_bwd: row groups must end on multiples of %d rows", RED_CHUNK);
  VI_CHECK_ARG(dout && x && w && dx && dw && db_cols, "vi_rowdot_bwd: null operand");
  if (rows <= 0) return VI_OK;
  const int nch = red_chunks(rows);
  VI_CHECK_ARG(scratch && scratch_elems >= (int64_t)2 * nch * D, "vi_rowdot_bwd: scratch too small");
  VI_CUDA(vi_launch(rowdot_bwd_dx_kernel, dim3((unsigned)((rows + 3) / 4)), dim3(128), 0, ST(stream), dout, w, dx, (long long)rows, grp));
  VI_CUDA(vi_launch(rowdot_bwd_w_partial_kernel, dim3(D / 64, nch), dim3(256), 0, ST(stream), dout, x, scratch, (long long)rows, nch));
  VI_CUDA(vi_launch(chunk_sum_kernel, dim3(D / 256, n_groups, 1), dim3(256), 0, ST(stream), (const float*)scratch, dw, nch, D,
                    (long long)rows, grp, (long long)0));
  // db_cols[g, c] = sum_r dout[r] for every column c (replicated); the caller reads column 0
  VI_CUDA(vi_launch(chunk_sum_kernel, dim3(D / 256, n_groups, 1), dim3(256), 0, ST(stream),
                    (const float*)(scratch + (long long)nch * D), db_cols, nch, D, (long long)rows, grp, (long long)0));
  return VI_OK;
}

extern "C" int vi_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* dout,
                           int64_t ldo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, int dtype,
                           const uint8_t* key_mask, const float* pair_dist, const float* bias_affine, float* d_affine, int B,
                           int H, int Lq, int Lk, int mask_mode, float drop_p, uint32_t drop_site, const uint32_t* drop_seed,
                           vi_stream_t stream) {
  VI_CHECK_ARG(q && k && v && dout && dq && dk && dv, "vi_attn_bwd: null operand");
  VI_CHECK_ARG(B > 0 && H > 0 && Lq > 0 && Lk > 0, "vi_attn_bwd: bad sizes B=%d H=%d Lq=%d Lk=%d", B, H, Lq, Lk);
  VI_CHECK_ARG(((size_t)Lk * (65 * 2 + 64 * 2 + 1) + 8 * (size_t)(128 + 2 * Lk)) * sizeof(float) <= 220 * 1024,
               "vi_attn_bwd: Lk=%d keys do not fit the 220 KB shared-memory tile", Lk);
  VI_CHECK_ARG(!pair_dist || bias_affine, "vi_attn_bwd: pair_dist needs bias_affine");
  VI_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_seed), "vi_attn_bwd: bad dropout arguments");
  VI_CHECK_ARG(H * 64 <= ldq && H * 64 <= ldk && H * 64 <= ldv && H * 64 <= ldo, "vi_attn_bwd: leading dimensions smaller than H*64");
  if (dtype == VI_DT_BF16) {
    const int rc = vi_attn_bwd_tc(q, ldq, k, ldk, v, ldv, dout, ldo, dq, lddq, dk, lddk, dv, lddv, key_mask, pair_dist,
                                  bias_affine, d_affine, B, H, Lq, Lk, mask_mode, drop_p, drop_site, drop_seed, ST(stream));
    if (rc <= 0) return rc;            // launched (0) or failed (< 0); 1 = does not fit -> fp32-arithmetic kernel below
  }
  VI_CHECK_ARG(drop_p == 0.f, "vi_attn_bwd: attention dropout is implemented by the bf16 tensor-core kernel only");
  AttnBwdParams p;
  p.q = q; p.ldq = ldq; p.k = k; p.ldk = ldk; p.v = v; p.ldv = ldv; p.dout = dout; p.ldo = ldo;
  p.dq = dq; p.lddq = lddq; p.dk = dk; p.lddk = lddk; p.dv = dv; p.lddv = lddv;
  p.key_mask = key_mask; p.pair_dist = pair_dist; p.bias_affine = bias_affine; p.d_affine = d_affine;
  p.B = B; p.H = H; p.Lq = Lq; p.Lk = Lk; p.mask_mode = mask_mode;
  const size_t smem = ((size_t)Lk * (65 * 2 + 64 * 2 + 1) + 8 * (size_t)(128 + 2 * Lk)) * sizeof(float);
  if (dtype == VI_DT_BF16) {
    static bool set = false;
    if (!set) { VI_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024)); set = true; }
    VI_CUDA(vi_launch(attn_bwd_kernel<bf16>, dim3(H, B), dim3(256), smem, ST(stream), p));
  } else {
    static bool set = false;
    if (!set) { VI_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024)); set = true; }
    VI_CUDA(vi_launch(attn_bwd_kernel<float>, dim3(H, B), dim3(256), smem, ST(stream), p));
  }
  return VI_OK;
}

extern "C" int vi_duet_fuse_logits_bwd(const float* g_raw, const float* l_raw, const float* fuse_raw, const uint8_t* gmap_masks,
                                       const uint8_t* gmap_visited, const uint8_t* vp_nav_masks, const int32_t* gmap_ids,
                                       const int32_t* cand_ids, const float* d_global, const float* d_local,
                                       const float* d_fused, float* dg_raw, float* dl_raw, float* dfuse_raw, int B, int G, int P,
                                       vi_stream_t stream) {
  VI_CHECK_ARG(g_raw && l_raw && gmap_masks && gmap_visited && vp_nav_masks && gmap_ids && cand_ids && dg_raw && dl_raw,
               "vi_duet_fuse_logits_bwd: null operand");
  VI_CHECK_ARG(B > 0 && G > 0 && P > 0 && G <= FUSE_MAX && P <= FUSE_MAX, "vi_duet_fuse_logits_bwd: bad sizes");
  VI_CUDA(vi_launch(duet_fuse_logits_bwd_kernel, dim3(B), dim3(32), 0, ST(stream), g_raw, l_raw, fuse_raw, gmap_masks,
                    gmap_visited, vp_nav_masks, gmap_ids, cand_ids, d_global, d_local, d_fused, dg_raw, dl_raw, dfuse_raw, G, P));
  return VI_OK;
}

extern "C" int vi_mul_bcast_bwd_s(const float* dy, const float* x, float* ds, int64_t n_batches, int rows_per_batch,
                                  vi_stream_t stream) {
  VI_CHECK_ARG(dy && x && ds && n_batches > 0 && rows_per_batch > 0, "vi_mul_bcast_bwd_s: bad operands");
  VI_CUDA(vi_launch(mul_bcast_bwd_s_kernel, dim3((unsigned)n_batches), dim3(256), 0, ST(stream), dy, x, ds, rows_per_batch));
  return VI_OK;
}

extern "C" int vi_cosine_loss_bwd(const float* proj, const float* tgt, const float* dloss, float* dproj, float* dtgt, int R,
                                  vi_stream_t stream) {
  VI_CHECK_ARG(proj && tgt && dloss && (dproj || dtgt), "vi_cosine_loss_bwd: null operand");
  if (R <= 0) return VI_OK;
  VI_CUDA(vi_launch(cosine_loss_bwd_kernel, dim3((unsigned)((R + 3) / 4)), dim3(128), 0, ST(stream), proj, tgt, dloss, dproj, dtgt,
                    (long long)R));
  return VI_OK;
}

// the two contrastive loss adjoints: one launch for dproj (and dtgt), a second one for dnegs when it is asked for
static int contrastive_loss_bwd(const char* name, const float* proj, const float* tgt, const float* negs,
                                const int32_t* row_episode, const int32_t* neg_episode, float inv_t, const float* sims,
                                const float* dloss, float* dproj, float* dtgt, float* dnegs, float* scratch, int R, int n_negs,
                                int margin_mode, float margin, vi_stream_t stream) {
  VI_CHECK_ARG(proj && tgt && row_episode && sims && dloss && dproj, "%s: null operand", name);
  VI_CHECK_ARG(n_negs == 0 || (negs && neg_episode), "%s: negatives missing", name);
  const bool want_negs = dnegs && n_negs > 0;
  VI_CHECK_ARG(!want_negs || scratch, "%s: dnegs needs the R * (n_negs + 1) float scratch", name);
  VI_CHECK_ARG(!want_negs || (aligned16(proj) && aligned16(negs) && aligned16(dnegs)), "%s: misaligned operands", name);
  if (R <= 0) return VI_OK;
  float* gneg = want_negs ? scratch : nullptr;
  float* inv_np = want_negs ? scratch + (long long)R * n_negs : nullptr;
  VI_CUDA(vi_launch(infonce_loss_bwd_kernel, dim3((unsigned)((R + 3) / 4)), dim3(128), 0, ST(stream), proj, tgt, negs, row_episode,
                    neg_episode, inv_t, sims, dloss, dproj, dtgt, gneg, inv_np, R, n_negs, margin_mode, margin));
  if (want_negs)
    VI_CUDA(vi_launch(contrastive_negs_bwd_kernel, dim3((unsigned)((n_negs + NEG_TILE - 1) / NEG_TILE), D / 256), dim3(64), 0,
                      ST(stream), proj, negs, sims, (const float*)gneg, (const float*)inv_np, 1.0f / inv_t, dnegs, R, n_negs));
  return VI_OK;
}

extern "C" int vi_infonce_loss_bwd(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                                   const int32_t* neg_episode, float temperature, const float* sims, const float* dloss,
                                   float* dproj, float* dtgt, float* dnegs, float* scratch, int R, int n_negs,
                                   vi_stream_t stream) {
  VI_CHECK_ARG(temperature > 0.f, "vi_infonce_loss_bwd: temperature must be positive");
  return contrastive_loss_bwd("vi_infonce_loss_bwd", proj, tgt, negs, row_episode, neg_episode, 1.0f / temperature, sims, dloss,
                              dproj, dtgt, dnegs, scratch, R, n_negs, 0, 0.f, stream);
}

extern "C" int vi_margin_loss_bwd(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                                  const int32_t* neg_episode, float margin, const float* sims, const float* dloss,
                                  float* dproj, float* dtgt, float* dnegs, float* scratch, int R, int n_negs,
                                  vi_stream_t stream) {
  return contrastive_loss_bwd("vi_margin_loss_bwd", proj, tgt, negs, row_episode, neg_episode, 1.0f, sims, dloss, dproj, dtgt,
                              dnegs, scratch, R, n_negs, 1, margin, stream);
}
