// vi_rl.cu - the reinforcement-learning tail of HAMT fine-tuning (IL + A2C, H/r2r/agent_cmt.py:544-577 sampling, :661-744 loss)
// and the Critic's value head (H/models/model_HAMT.py:289-300).
//
//   vi_policy_sample   one warp per episode: masked softmax over the O observation logits, entropy, an inverse-CDF sample keyed
//                      by the counter-based dropout hash, log p[a], the running `ended` flags and the step mask
//   vi_policy_bwd      d logits of  g_logp * log p[a] + g_H * H  (softmax recomputed from the logits)
//   vi_a2c_loss[_bwd]  the discounted-return scan and the A2C loss over [T, B], one CTA
//   vi_value_head[_bwd] v = dropout(h) . w2 + b2 over 512-wide rows (the last Linear of the critic) and its adjoint
//
// Every reduction runs in a fixed order with no atomics: two calls give identical bits.
#include "vi_common.cuh"

namespace {

constexpr int POLICY_WARPS = 4;          // episodes per CTA of the policy kernels
constexpr int A2C_THREADS = 256;         // the one CTA of the loss kernels
constexpr int VH_WIDTH = 512;            // critic hidden width
constexpr int VH_ROWS = 8;               // rows (warps) per CTA of the value-head kernels
constexpr int VH_COL_THREADS = 256;      // threads of a column-reduction CTA of the value-head adjoint

// (max, sum of exp(x - max)) of one warp's row; masked entries are -inf and add nothing
__device__ __forceinline__ void row_stats(const float* x, int O, int lane, float& m, float& s) {
  m = -INFINITY;
  for (int j = lane; j < O; j += 32) m = fmaxf(m, x[j]);
  m = warp_max(m);
  s = 0.f;
  if (m != -INFINITY)
    for (int j = lane; j < O; j += 32) s += expf(x[j] - m);
  s = warp_sum(s);
}

// H = -sum_j p_j log p_j over the entries with p_j > 0, log p_j = x_j - m - log s
__device__ __forceinline__ float row_entropy(const float* x, int O, int lane, float m, float s, float lse) {
  float h = 0.f;
  for (int j = lane; j < O; j += 32) {
    const float e = x[j] == -INFINITY ? 0.f : expf(x[j] - m) / s;
    if (e > 0.f) h -= e * (x[j] - lse);
  }
  return warp_sum(h);
}

__global__ void __launch_bounds__(POLICY_WARPS * 32) policy_sample_kernel(const float* logits, long long ld, int O, int B,
                                                                          const int64_t* stop_idx, const uint32_t* seed,
                                                                          uint32_t site, int64_t* actions, float* logp,
                                                                          float* entropy, uint8_t* ended, float* step_mask) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * POLICY_WARPS + (threadIdx.x >> 5);
  if (b >= B) return;
  const float* x = logits + (long long)b * ld;
  float m, s;
  row_stats(x, O, lane, m, s);
  const bool was_ended = ended[b] != 0;
  if (m == -INFINITY) {                          // no admissible token: no action, nothing to learn from
    if (lane == 0) {
      actions[b] = -1; logp[b] = 0.f; entropy[b] = 0.f;
      step_mask[b] = was_ended ? 0.f : 1.f;
    }
    return;
  }
  const float lse = m + logf(s);
  const float H = row_entropy(x, O, lane, m, s, lse);

  // inverse CDF: u in [0, 1) from the hash of (episode, key(seed, site)); first j with cumsum(e) > u * s and e_j > 0
  const uint32_t key = vi_drop_key(seed, site);
  const float target = (float)(vi_hash32((uint32_t)b, key) >> 8) * (1.0f / 16777216.0f) * s;
  int a = -1, last_ok = -1;
  float carry = 0.f;
  for (int j0 = 0; j0 < O; j0 += 32) {
    const int j = j0 + lane;
    const float e = (j < O && x[j] != -INFINITY) ? expf(x[j] - m) : 0.f;
    float c = e;                                 // inclusive warp scan, fixed order
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float t = __shfl_up_sync(0xffffffffu, c, o);
      if (lane >= o) c += t;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, e > 0.f && carry + c > target);
    const unsigned ok = __ballot_sync(0xffffffffu, e > 0.f);
    if (ok) last_ok = j0 + 31 - __clz(ok);
    if (hit) { a = j0 + __ffs(hit) - 1; break; }
    carry += __shfl_sync(0xffffffffu, c, 31);
  }
  if (a < 0) a = last_ok;                        // rounding left the target above the total: the last admissible token
  if (lane == 0) {
    actions[b] = a;
    logp[b] = x[a] - lse;
    entropy[b] = H;
    step_mask[b] = was_ended ? 0.f : 1.f;
    if (!was_ended && a == stop_idx[b]) ended[b] = 1;
  }
}

__global__ void __launch_bounds__(POLICY_WARPS * 32) policy_bwd_kernel(const float* logits, long long ld, int O, int B,
                                                                       const int64_t* actions, const float* g_logp,
                                                                       const float* g_ent, float* dlogits, long long ldd) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * POLICY_WARPS + (threadIdx.x >> 5);
  if (b >= B) return;
  const float* x = logits + (long long)b * ld;
  float* d = dlogits + (long long)b * ldd;
  float m, s;
  row_stats(x, O, lane, m, s);
  const long long a = actions[b];
  if (m == -INFINITY || a < 0) {
    for (int j = lane; j < O; j += 32) d[j] = 0.f;
    return;
  }
  const float lse = m + logf(s);
  const float H = row_entropy(x, O, lane, m, s, lse);
  const float gl = g_logp ? g_logp[b] : 0.f, gh = g_ent ? g_ent[b] : 0.f;
  for (int j = lane; j < O; j += 32) {
    float v = 0.f;
    if (x[j] != -INFINITY) {
      const float lp = x[j] - lse;
      const float p = expf(x[j] - m) / s;
      v = gl * ((j == a ? 1.f : 0.f) - p) - gh * p * (lp + H);
    }
    d[j] = v;
  }
}

// R_T = ended_last ? 0 : boot;  R_t = gamma R_{t+1} + r_t;  A_t = R_t - v_t (constant);  per-episode sums of the three terms
struct A2CArgs {
  const float *values, *logp, *ent, *masks, *rewards, *boot;
  const uint8_t* ended;
  int T, B, norm;
  float gamma, w_ent;
};

// fixed-order block sum of n_vals per-thread values; thread 0 ends with the totals in tot[]
template <int N>
__device__ __forceinline__ void block_sums(float (&v)[N], float (*red)[A2C_THREADS], float* tot) {
#pragma unroll
  for (int i = 0; i < N; ++i) red[i][threadIdx.x] = v[i];
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      float acc = 0.f;
      for (int t = 0; t < A2C_THREADS; ++t) acc += red[i][t];
      tot[i] = acc;
    }
  }
  __syncthreads();
}

__device__ __forceinline__ float a2c_scale(const A2CArgs& a, float msum) {
  return a.norm == VI_A2C_NORM_TOTAL ? 1.0f / fmaxf(msum, 1.0f) : a.norm == VI_A2C_NORM_BATCH ? 1.0f / (float)a.B : 1.0f;
}

__global__ void __launch_bounds__(A2C_THREADS) a2c_loss_kernel(A2CArgs a, float* out) {
  __shared__ float red[4][A2C_THREADS];
  __shared__ float tot[4];
  pdl_enter();
  float acc[4] = {0.f, 0.f, 0.f, 0.f};           // policy, critic, entropy, mask sum
  for (int b = threadIdx.x; b < a.B; b += A2C_THREADS) {
    float R = (a.boot && !a.ended[b]) ? a.boot[b] : 0.f;
    for (int t = a.T - 1; t >= 0; --t) {
      const long long i = (long long)t * a.B + b;
      R = R * a.gamma + a.rewards[i];
      const float m = a.masks[i], v = a.values[i], adv = R - v;
      acc[0] += -a.logp[i] * adv * m;
      acc[1] += 0.5f * adv * adv * m;
      acc[2] += -a.w_ent * a.ent[i] * m;
      acc[3] += m;
    }
  }
  block_sums<4>(acc, red, tot);
  if (threadIdx.x == 0) {
    const float k = a2c_scale(a, tot[3]);
    out[1] = tot[0] * k;
    out[2] = tot[1] * k;
    out[3] = tot[2] * k;
    out[0] = (tot[0] + tot[1] + tot[2]) * k;
  }
}

__global__ void __launch_bounds__(A2C_THREADS) a2c_loss_bwd_kernel(A2CArgs a, const float* gout, float* dvalues, float* dlogp,
                                                                   float* dent) {
  __shared__ float red[1][A2C_THREADS];
  __shared__ float tot[1];
  pdl_enter();
  float ms[1] = {0.f};
  for (int b = threadIdx.x; b < a.B; b += A2C_THREADS)
    for (int t = 0; t < a.T; ++t) ms[0] += a.masks[(long long)t * a.B + b];
  block_sums<1>(ms, red, tot);
  const float k = a2c_scale(a, tot[0]);
  const float gp = (gout[0] + gout[1]) * k, gc = (gout[0] + gout[2]) * k, ge = (gout[0] + gout[3]) * k;
  for (int b = threadIdx.x; b < a.B; b += A2C_THREADS) {
    float R = (a.boot && !a.ended[b]) ? a.boot[b] : 0.f;
    for (int t = a.T - 1; t >= 0; --t) {
      const long long i = (long long)t * a.B + b;
      R = R * a.gamma + a.rewards[i];
      const float m = a.masks[i], adv = R - a.values[i];
      if (dlogp) dlogp[i] = -gp * adv * m;
      if (dvalues) dvalues[i] = -gc * adv * m;
      if (dent) dent[i] = -ge * a.w_ent * m;
    }
  }
}

// element (r, c) of the critic's dropout: kept iff hash(r * 512 + c, key) >= threshold (vi_dropout's rule)
__device__ __forceinline__ float drop_scale(long long r, int c, uint32_t key, uint32_t thr, float inv_keep) {
  return vi_hash32((uint32_t)(r * VH_WIDTH + c), key) >= thr ? inv_keep : 0.f;
}

__global__ void __launch_bounds__(VH_ROWS * 32) value_head_kernel(const float* h, long long rows, const float* w2, const float* b2,
                                                                  float p, const uint32_t* seed, uint32_t site, float* v) {
  pdl_enter();
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * VH_ROWS + (threadIdx.x >> 5);
  if (r >= rows) return;
  const uint32_t key = p > 0.f ? vi_drop_key(seed, site) : 0u, thr = vi_drop_threshold(p);
  const float inv_keep = p > 0.f ? 1.0f / (1.0f - p) : 1.f;
  const float* hr = h + r * VH_WIDTH;
  float acc = 0.f;
  for (int c = lane; c < VH_WIDTH; c += 32) {
    const float x = p > 0.f ? hr[c] * drop_scale(r, c, key, thr, inv_keep) : hr[c];
    acc += x * w2[c];
  }
  acc = warp_sum(acc);
  if (lane == 0) v[r] = acc + b2[0];
}

// blocks [0, row_blocks): dh rows; the next VH_WIDTH / VH_COL_THREADS blocks: dw2 columns; the last one also db2
__global__ void __launch_bounds__(VH_COL_THREADS) value_head_bwd_kernel(const float* dv, const float* h, long long rows,
                                                                        const float* w2, float p, const uint32_t* seed,
                                                                        uint32_t site, float* dh32, bf16* dh16, int f16,
                                                                        float* dw2, float* db2, int row_blocks) {
  pdl_enter();
  const uint32_t key = p > 0.f ? vi_drop_key(seed, site) : 0u, thr = vi_drop_threshold(p);
  const float inv_keep = p > 0.f ? 1.0f / (1.0f - p) : 1.f;
  if ((int)blockIdx.x < row_blocks) {
    const int lane = threadIdx.x & 31;
    const long long r = (long long)blockIdx.x * (VH_COL_THREADS / 32) + (threadIdx.x >> 5);
    if (r >= rows) return;
    const float g = dv[r];
    const float* hr = h + r * VH_WIDTH;
    for (int c = 2 * lane; c < VH_WIDTH; c += 64) {
      float o[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float ds = p > 0.f ? drop_scale(r, c + i, key, thr, inv_keep) : 1.f;
        o[i] = hr[c + i] > 0.f ? g * w2[c + i] * ds : 0.f;     // ReLU: h is the rectified output
      }
      if (dh32) { dh32[r * VH_WIDTH + c] = o[0]; dh32[r * VH_WIDTH + c + 1] = o[1]; }
      if (dh16) *reinterpret_cast<uint32_t*>(dh16 + r * VH_WIDTH + c) = pack_h16x2(o[0], o[1], f16 != 0);
    }
    return;
  }
  const int c = ((int)blockIdx.x - row_blocks) * VH_COL_THREADS + threadIdx.x;
  float acc = 0.f, accb = 0.f;
  for (long long r = 0; r < rows; ++r) {
    const float g = dv[r];
    const float x = p > 0.f ? h[r * VH_WIDTH + c] * drop_scale(r, c, key, thr, inv_keep) : h[r * VH_WIDTH + c];
    acc += g * x;
    accb += g;
  }
  dw2[c] = acc;
  if (c == 0 && db2) db2[0] = accb;
}

}  // namespace

extern "C" int vi_policy_sample(const float* logits, int64_t ld, int O, int B, const int64_t* stop_idx, const uint32_t* seed,
                                uint32_t site, int64_t* actions, float* logp, float* entropy, uint8_t* ended, float* step_mask,
                                vi_stream_t stream) {
  VI_CHECK_ARG(B >= 0 && O >= 0 && ld >= O, "vi_policy_sample: bad shape B=%d O=%d ld=%lld", B, O, (long long)ld);
  if (B == 0) return VI_OK;
  VI_CHECK_ARG(logits && stop_idx && seed && actions && logp && entropy && ended && step_mask && O > 0,
               "vi_policy_sample: bad operands");
  VI_CUDA(vi_launch(policy_sample_kernel, dim3((unsigned)((B + POLICY_WARPS - 1) / POLICY_WARPS)), dim3(POLICY_WARPS * 32), (size_t)0,
                    reinterpret_cast<cudaStream_t>(stream), logits, (long long)ld, O, B, stop_idx, seed, site, actions, logp, entropy,
                    ended, step_mask));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_policy_bwd(const float* logits, int64_t ld, int O, int B, const int64_t* actions, const float* g_logp,
                             const float* g_entropy, float* dlogits, int64_t ldd, vi_stream_t stream) {
  VI_CHECK_ARG(B >= 0 && O >= 0 && ld >= O && ldd >= O, "vi_policy_bwd: bad shape B=%d O=%d", B, O);
  if (B == 0) return VI_OK;
  VI_CHECK_ARG(logits && actions && dlogits && O > 0, "vi_policy_bwd: bad operands");
  VI_CUDA(vi_launch(policy_bwd_kernel, dim3((unsigned)((B + POLICY_WARPS - 1) / POLICY_WARPS)), dim3(POLICY_WARPS * 32), (size_t)0,
                    reinterpret_cast<cudaStream_t>(stream), logits, (long long)ld, O, B, actions, g_logp, g_entropy, dlogits,
                    (long long)ldd));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

static int a2c_args(A2CArgs& a, const float* values, const float* logp, const float* entropy, const float* masks,
                    const float* rewards, const float* boot, const uint8_t* ended, int T, int B, float gamma, float w_ent, int norm) {
  VI_CHECK_ARG(T >= 0 && B >= 0, "vi_a2c_loss: bad shape T=%d B=%d", T, B);
  VI_CHECK_ARG(norm == VI_A2C_NORM_NONE || norm == VI_A2C_NORM_BATCH || norm == VI_A2C_NORM_TOTAL, "vi_a2c_loss: bad norm %d", norm);
  VI_CHECK_ARG((T == 0 || B == 0) || (values && logp && entropy && masks && rewards), "vi_a2c_loss: bad operands");
  VI_CHECK_ARG(!boot || ended, "vi_a2c_loss: a bootstrap value needs the ended flags");
  a.values = values; a.logp = logp; a.ent = entropy; a.masks = masks; a.rewards = rewards; a.boot = boot; a.ended = ended;
  a.T = T; a.B = B; a.norm = norm; a.gamma = gamma; a.w_ent = w_ent;
  return VI_OK;
}

extern "C" int vi_a2c_loss(const float* values, const float* logp, const float* entropy, const float* masks, const float* rewards,
                           const float* boot, const uint8_t* ended, int T, int B, float gamma, float entropy_weight, int norm,
                           float* out, vi_stream_t stream) {
  A2CArgs a;
  const int rc = a2c_args(a, values, logp, entropy, masks, rewards, boot, ended, T, B, gamma, entropy_weight, norm);
  if (rc != VI_OK) return rc;
  VI_CHECK_ARG(out, "vi_a2c_loss: out is NULL");
  VI_CUDA(vi_launch(a2c_loss_kernel, dim3(1), dim3(A2C_THREADS), (size_t)0, reinterpret_cast<cudaStream_t>(stream), a, out));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_a2c_loss_bwd(const float* values, const float* logp, const float* entropy, const float* masks, const float* rewards,
                               const float* boot, const uint8_t* ended, int T, int B, float gamma, float entropy_weight, int norm,
                               const float* gout, float* dvalues, float* dlogp, float* dentropy, vi_stream_t stream) {
  A2CArgs a;
  const int rc = a2c_args(a, values, logp, entropy, masks, rewards, boot, ended, T, B, gamma, entropy_weight, norm);
  if (rc != VI_OK) return rc;
  VI_CHECK_ARG(gout, "vi_a2c_loss_bwd: gout is NULL");
  if (T == 0 || B == 0) return VI_OK;
  VI_CUDA(vi_launch(a2c_loss_bwd_kernel, dim3(1), dim3(A2C_THREADS), (size_t)0, reinterpret_cast<cudaStream_t>(stream), a, gout,
                    dvalues, dlogp, dentropy));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_value_head(const float* h, int64_t rows, const float* w2, const float* b2, float drop_p, const uint32_t* drop_seed,
                             uint32_t drop_site, float* v, vi_stream_t stream) {
  VI_CHECK_ARG(rows >= 0 && rows * VH_WIDTH < (1LL << 32), "vi_value_head: rows=%lld out of range", (long long)rows);
  VI_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_seed), "vi_value_head: bad dropout");
  if (rows == 0) return VI_OK;
  VI_CHECK_ARG(h && w2 && b2 && v, "vi_value_head: bad operands");
  VI_CUDA(vi_launch(value_head_kernel, dim3((unsigned)((rows + VH_ROWS - 1) / VH_ROWS)), dim3(VH_ROWS * 32), (size_t)0,
                    reinterpret_cast<cudaStream_t>(stream), h, (long long)rows, w2, b2, drop_p, drop_seed, drop_site, v));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

extern "C" int vi_value_head_bwd(const float* dv, const float* h, int64_t rows, const float* w2, float drop_p,
                                 const uint32_t* drop_seed, uint32_t drop_site, float* dh32, void* dh16, int dh16_dtype, float* dw2,
                                 float* db2, vi_stream_t stream) {
  VI_CHECK_ARG(rows >= 0 && rows * VH_WIDTH < (1LL << 32), "vi_value_head_bwd: rows=%lld out of range", (long long)rows);
  VI_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_seed), "vi_value_head_bwd: bad dropout");
  VI_CHECK_ARG(dh16_dtype == VI_DT_BF16 || dh16_dtype == VI_DT_F16, "vi_value_head_bwd: dh16_dtype must be VI_DT_BF16 or VI_DT_F16");
  VI_CHECK_ARG(dv && h && w2 && dw2, "vi_value_head_bwd: bad operands");
  const int row_blocks = (int)((rows + VH_COL_THREADS / 32 - 1) / (VH_COL_THREADS / 32));
  VI_CUDA(vi_launch(value_head_bwd_kernel, dim3((unsigned)(row_blocks + VH_WIDTH / VH_COL_THREADS)), dim3(VH_COL_THREADS), (size_t)0,
                    reinterpret_cast<cudaStream_t>(stream), dv, h, (long long)rows, w2, drop_p, drop_seed, drop_site, dh32,
                    reinterpret_cast<bf16*>(dh16), dh16_dtype == VI_DT_F16 ? 1 : 0, dw2, db2, row_blocks));
  VI_LAUNCH_CHECK();
  return VI_OK;
}
