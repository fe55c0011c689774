// vi_xent.cu - backward of the per-row loss kernels vi_ce_rows / vi_kl_rows (the pre-training heads,
// VLN-DUET/pretrain_src/model/pretrain_cmt.py:150 MLM, :198-204 MRC, :244-254 SAP).
//
// dx[r, c] = dloss[r] * (softmax(x[r, 0:n])[c] * T[r] - t[r, c])   for c < n, exact 0 for n <= c < ld_out
//   cross-entropy: t = one-hot(label[r]), T = 1;   KL: t = the soft targets, T = sum_c t[r, c].
// dx goes out as fp32 and / or 16-bit: the latter is the A operand of the dgrad and wgrad GEMMs of the layer that made
// the logits, so the padded vocabulary columns must be zeros (they then add nothing to either product).
//
// Two layouts, picked from the shape:
//   * wide rows (the 30522-word vocabulary, the 1000-class MRC head): one CTA per row (128 - 1024 threads by width).  Pass 1 is an online (max, sum exp)
//     over 16-byte loads; pass 2 re-reads the row (mostly from L2) and writes 8 columns per thread per step with 16-byte
//     stores.  The forward's warp-per-row layout would run three dependent 120 KB sweeps per warp at a few hundred rows.
//   * narrow rows (the SAP logits: 10 - 40 columns, leading dimensions that are not multiples of 4): one warp per row,
//     scalar accesses.
// Reductions run in a fixed order (no atomics): results are bit-identical run to run.
#include "vi_common.cuh"

namespace {

constexpr int WIDE_MIN_COLS = 256;       // below this a CTA per row is mostly idle
constexpr int WIDE_MAX_THREADS = 1024;    // enough loads in flight for one row per SM at a few hundred rows
constexpr int VEC = 8;                   // columns per thread and step: two 16-byte fp32 loads, one 16-byte 16-bit store
constexpr int NARROW_ROWS = 4;           // warps (rows) per CTA of the narrow layout

enum { MODE_CE = 0, MODE_KL = 1 };

// running (max m, sum of exp(x - m)); m == -inf is the empty state (also for rows whose entries are all -inf)
__device__ __forceinline__ void ms_merge(float& m, float& s, float m2, float s2) {
  const float mn = fmaxf(m, m2);
  if (mn == -INFINITY) return;
  s = s * expf(m - mn) + s2 * expf(m2 - mn);     // commutative: both lanes of a butterfly get the same bits
  m = mn;
}

__device__ __forceinline__ void load8(float (&v)[VEC], const float* p, int c, int n) {
  if (c + VEC <= n) {
    const float4 a = *reinterpret_cast<const float4*>(p + c);
    const float4 b = *reinterpret_cast<const float4*>(p + c + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < VEC; ++i) v[i] = c + i < n ? p[c + i] : -INFINITY;
  }
}

template <int MODE>
__global__ void __launch_bounds__(WIDE_MAX_THREADS) xent_bwd_wide_kernel(const float* x, long long ld, const int64_t* labels,
                                                                         const float* t, long long ldt, int n, const float* dloss,
                                                                         float* dx32, bf16* dx16, int f16, long long ld_out) {
  __shared__ float red[3][WIDE_MAX_THREADS / 32];
  pdl_enter();
  const long long row = blockIdx.x;
  const float* xr = x + row * ld;
  const float* tr = MODE == MODE_KL ? t + row * ldt : nullptr;
  const int step = blockDim.x * VEC;

  // pass 1: online max / sum of exponentials (+ the target mass for KL)
  float m = -INFINITY, s = 0.f, ts = 0.f;
  for (int c = threadIdx.x * VEC; c < n; c += step) {
    float v[VEC];
    load8(v, xr, c, n);
    float m8 = v[0];
#pragma unroll
    for (int i = 1; i < VEC; ++i) m8 = fmaxf(m8, v[i]);
    if (m8 != -INFINITY) {
      float s8 = 0.f;
#pragma unroll
      for (int i = 0; i < VEC; ++i) s8 += expf(v[i] - m8);
      ms_merge(m, s, m8, s8);
    }
    if (MODE == MODE_KL) {
      float tv[VEC];
      load8(tv, tr, c, n);
#pragma unroll
      for (int i = 0; i < VEC; ++i) ts += c + i < n ? tv[i] : 0.f;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    ms_merge(m, s, m2, s2);
    if (MODE == MODE_KL) ts += __shfl_xor_sync(0xffffffffu, ts, o);
  }
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) { red[0][warp] = m; red[1][warp] = s; red[2][warp] = ts; }
  __syncthreads();
  m = red[0][0]; s = red[1][0]; ts = red[2][0];
  for (int w = 1; w < nw; ++w) {                 // every thread merges the warps in the same order
    ms_merge(m, s, red[0][w], red[1][w]);
    if (MODE == MODE_KL) ts += red[2][w];
  }
  const float inv = 1.0f / s;
  const float g = dloss[row];
  const float T = MODE == MODE_KL ? ts : 1.f;
  const long long label = MODE == MODE_CE ? labels[row] : -1;

  // pass 2: the gradient row, padding columns included
  for (long long c = threadIdx.x * VEC; c < ld_out; c += step) {
    float o[VEC];
    if (c < n) {
      float v[VEC], tv[VEC];
      load8(v, xr, (int)c, n);
      if (MODE == MODE_KL) load8(tv, tr, (int)c, n);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float p = expf(v[i] - m) * inv;    // -inf logits and the columns past n: exp(-inf) = 0
        const float tc = MODE == MODE_KL ? (c + i < n ? tv[i] : 0.f) : (c + i == label ? 1.f : 0.f);
        o[i] = c + i < n ? g * (p * T - tc) : 0.f;
      }
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) o[i] = 0.f;
    }
    if (dx32) {
      float4* d = reinterpret_cast<float4*>(dx32 + row * ld_out + c);
      d[0] = make_float4(o[0], o[1], o[2], o[3]);
      d[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
    if (dx16) {
      *reinterpret_cast<uint4*>(dx16 + row * ld_out + c) =
          make_uint4(pack_h16x2(o[0], o[1], f16 != 0), pack_h16x2(o[2], o[3], f16 != 0), pack_h16x2(o[4], o[5], f16 != 0),
                     pack_h16x2(o[6], o[7], f16 != 0));
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(NARROW_ROWS * 32) xent_bwd_narrow_kernel(const float* x, long long ld, const int64_t* labels,
                                                                           const float* t, long long ldt, int n, const float* dloss,
                                                                           float* dx32, bf16* dx16, int f16, long long ld_out,
                                                                           long long rows) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * NARROW_ROWS + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * ld;
  const float* tr = MODE == MODE_KL ? t + row * ldt : nullptr;
  float m = -INFINITY, ts = 0.f;
  for (int c = lane; c < n; c += 32) {
    m = fmaxf(m, xr[c]);
    if (MODE == MODE_KL) ts += tr[c];
  }
  m = warp_max(m);
  float s = 0.f;
  if (m != -INFINITY)
    for (int c = lane; c < n; c += 32) s += expf(xr[c] - m);
  s = warp_sum(s);
  const float inv = 1.0f / s;
  const float g = dloss[row];
  const float T = MODE == MODE_KL ? warp_sum(ts) : 1.f;
  const long long label = MODE == MODE_CE ? labels[row] : -1;
  for (long long c = lane; c < ld_out; c += 32) {
    float o = 0.f;
    if (c < n) {
      const float tc = MODE == MODE_KL ? tr[c] : (c == label ? 1.f : 0.f);
      o = g * (expf(xr[c] - m) * inv * T - tc);
    }
    if (dx32) dx32[row * ld_out + c] = o;
    if (dx16) reinterpret_cast<uint16_t*>(dx16)[row * ld_out + c] = (uint16_t)(pack_h16x2(o, 0.f, f16 != 0) & 0xFFFFu);
  }
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

template <int MODE>
int xent_bwd(const float* logits, int64_t ld, const int64_t* labels, const float* targets, int64_t ldt, int n_cols,
             const float* dloss, float* dx32, void* dx16, int dx16_dtype, int64_t ld_out, int64_t rows, cudaStream_t st) {
  const bool wide = n_cols >= WIDE_MIN_COLS && ld % 4 == 0 && ld_out % VEC == 0 && aligned16(logits) && aligned16(dx32) &&
                    aligned16(dx16) && (MODE == MODE_CE || (ldt % 4 == 0 && aligned16(targets)));
  const int f16 = dx16_dtype == VI_DT_F16;
  if (wide) {
    int threads = 128;                           // >= 4 steps of 8 columns per thread (30522 columns: 1024 threads; 1000: 128)
    while (threads < WIDE_MAX_THREADS && threads * VEC * 4 < n_cols) threads *= 2;
    VI_CUDA(vi_launch(xent_bwd_wide_kernel<MODE>, dim3((unsigned)rows), dim3(threads), (size_t)0, st, logits, (long long)ld, labels,
                      targets, (long long)ldt, n_cols, dloss, dx32, reinterpret_cast<bf16*>(dx16), f16, (long long)ld_out));
  } else {
    VI_CUDA(vi_launch(xent_bwd_narrow_kernel<MODE>, dim3((unsigned)((rows + NARROW_ROWS - 1) / NARROW_ROWS)), dim3(NARROW_ROWS * 32),
                      (size_t)0, st, logits, (long long)ld, labels, targets, (long long)ldt, n_cols, dloss, dx32,
                      reinterpret_cast<bf16*>(dx16), f16, (long long)ld_out, (long long)rows));
  }
  VI_LAUNCH_CHECK();
  return VI_OK;
}

}  // namespace

extern "C" int vi_ce_rows_bwd(const float* logits, int64_t ld, const int64_t* labels, int n_cols, const float* dloss, float* dx32,
                              void* dx16, int dx16_dtype, int64_t ld_out, int64_t rows, vi_stream_t stream) {
  VI_CHECK_ARG(rows >= 0 && rows < (1LL << 31), "vi_ce_rows_bwd: rows=%lld out of range", (long long)rows);
  VI_CHECK_ARG(dx16_dtype == VI_DT_BF16 || dx16_dtype == VI_DT_F16, "vi_ce_rows_bwd: dx16_dtype must be VI_DT_BF16 or VI_DT_F16");
  if (rows == 0) return VI_OK;
  VI_CHECK_ARG(logits && labels && dloss && (dx32 || dx16) && n_cols > 0 && ld >= n_cols && ld_out >= n_cols,
               "vi_ce_rows_bwd: bad operands");
  return xent_bwd<MODE_CE>(logits, ld, labels, nullptr, 0, n_cols, dloss, dx32, dx16, dx16_dtype, ld_out, rows,
                           reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vi_kl_rows_bwd(const float* logits, int64_t ld, const float* targets, int64_t ldt, int n_cols, const float* dloss,
                              float* dx32, void* dx16, int dx16_dtype, int64_t ld_out, int64_t rows, vi_stream_t stream) {
  VI_CHECK_ARG(rows >= 0 && rows < (1LL << 31), "vi_kl_rows_bwd: rows=%lld out of range", (long long)rows);
  VI_CHECK_ARG(dx16_dtype == VI_DT_BF16 || dx16_dtype == VI_DT_F16, "vi_kl_rows_bwd: dx16_dtype must be VI_DT_BF16 or VI_DT_F16");
  if (rows == 0) return VI_OK;
  VI_CHECK_ARG(logits && targets && dloss && (dx32 || dx16) && n_cols > 0 && ld >= n_cols && ldt >= n_cols && ld_out >= n_cols,
               "vi_kl_rows_bwd: bad operands");
  return xent_bwd<MODE_KL>(logits, ld, nullptr, targets, ldt, n_cols, dloss, dx32, dx16, dx16_dtype, ld_out, rows,
                           reinterpret_cast<cudaStream_t>(stream));
}
