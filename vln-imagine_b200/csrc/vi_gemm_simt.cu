// vi_gemm_simt.cu - the fp32 check-mode GEMM (FFMA, no tensor cores): Y = epi(X W^T + bias) + residual.
// Same contract and grouped form as vi_gemm16; used for the 1e-4 parity mode that BASELINE.json
// asks for and to cross-check the tcgen05 kernel.  64x64 output tile, 16x16 threads, 4x4 micro-tile,
// K staged through shared memory in blocks of 16.
#include "vi_common.cuh"

namespace {

constexpr int TM = 64, TN = 64, TK = 16;
constexpr int MAX_GROUPS = 4;

struct SimtParams {
  const float* x; long long ldx;
  const float* w;
  const float* bias;
  const float* residual; long long ldr;
  float* y; long long ldy;
  int M, N, K, epilogue, n_groups;
  int group_row_end[MAX_GROUPS];
};

__global__ void __launch_bounds__(256) gemm_f32_simt_kernel(const SimtParams p) {
  pdl_enter();
  __shared__ float xs[TK][TM + 4];
  __shared__ float ws[TK][TN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int row0 = blockIdx.y * TM, col0 = blockIdx.x * TN;
  int g = 0;
  while (g < p.n_groups - 1 && row0 >= p.group_row_end[g]) ++g;
  const float* wg = p.w + (long long)g * p.N * p.K;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < p.K; k0 += TK) {
    // 64 rows x 16 k of X and W: 1024 elements each, 256 threads -> 4 each
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = threadIdx.x + i * 256;
      const int r = e >> 4, k = e & 15;
      const long long xr = row0 + r;
      xs[k][r] = (xr < p.M && k0 + k < p.K) ? p.x[xr * p.ldx + k0 + k] : 0.f;
      const int wc = col0 + r;
      ws[k][r] = (wc < p.N && k0 + k < p.K) ? wg[(long long)wc * p.K + k0 + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = xs[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = ws[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long r = row0 + ty * 4 + i;
    if (r >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = col0 + tx * 4 + j;
      if (c >= p.N) continue;
      float v = acc[i][j];
      if (p.bias) v += p.bias[(long long)g * p.N + c];
      if (p.epilogue == VI_EPI_GELU) v = gelu_erf(v);
      else if (p.epilogue == VI_EPI_RELU) v = fmaxf(v, 0.f);
      if (p.residual) v += p.residual[r * p.ldr + c];
      p.y[r * p.ldy + c] = v;
    }
  }
}

}  // namespace

extern "C" int vi_gemm_f32(const float* x, int64_t ldx, const float* w, const float* bias, const float* residual,
                           int64_t ldr, float* y, int64_t ldy, int M, int N, int K, int epilogue, int n_groups,
                           const int32_t* group_row_end, vi_stream_t stream) {
  VI_CHECK_ARG(x && w && y, "vi_gemm_f32: null operand");
  VI_CHECK_ARG(M > 0 && N > 0 && K > 0, "vi_gemm_f32: empty problem M=%d N=%d K=%d", M, N, K);
  VI_CHECK_ARG(ldx >= K && ldy >= N, "vi_gemm_f32: leading dimensions too small");
  VI_CHECK_ARG(epilogue >= VI_EPI_NONE && epilogue <= VI_EPI_RELU, "vi_gemm_f32: bad epilogue %d", epilogue);
  VI_CHECK_ARG(n_groups >= 1 && n_groups <= MAX_GROUPS, "vi_gemm_f32: n_groups=%d out of range", n_groups);
  VI_CHECK_ARG(n_groups == 1 || group_row_end, "vi_gemm_f32: grouped call without group_row_end");
  SimtParams p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = ldx; p.w = w; p.bias = bias; p.residual = residual; p.ldr = ldr; p.y = y; p.ldy = ldy;
  p.M = M; p.N = N; p.K = K; p.epilogue = epilogue; p.n_groups = n_groups;
  for (int g = 0; g < n_groups; ++g) {
    if (n_groups == 1) { p.group_row_end[0] = M; break; }
    const int e = group_row_end[g];
    VI_CHECK_ARG(e > 0 && e <= M && (g == 0 || e > group_row_end[g - 1]), "vi_gemm_f32: bad group_row_end[%d]=%d", g, e);
    VI_CHECK_ARG(g == n_groups - 1 || e % 128 == 0, "vi_gemm_f32: group %d must end on a multiple of 128 rows", g);
    p.group_row_end[g] = e;
  }
  dim3 grid((N + TN - 1) / TN, (M + TM - 1) / TM);
  VI_CUDA(vi_launch(gemm_f32_simt_kernel, dim3(grid), dim3(256), (size_t)(0), reinterpret_cast<cudaStream_t>(stream), p));
  VI_LAUNCH_CHECK();
  return VI_OK;
}
