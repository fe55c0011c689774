// vi_common.cuh - shared helpers for the libvlnimagine kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

#include "../../include/vlnimagine.h"

// ----------------------------------------------------------------------------------------------
// host-side error plumbing (never throws / exits across the C ABI)
// ----------------------------------------------------------------------------------------------
void vi_set_error(const char* fmt, ...);

#define VI_CHECK_ARG(cond, ...)                                   \
  do {                                                            \
    if (!(cond)) {                                                \
      vi_set_error(__VA_ARGS__);                                  \
      return VI_ERR_ARG;                                          \
    }                                                             \
  } while (0)

#define VI_CUDA(call)                                                                     \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      vi_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return VI_ERR_CUDA;                                                                 \
    }                                                                                     \
  } while (0)

#define VI_LAUNCH_CHECK()                                                                 \
  do {                                                                                    \
    cudaError_t e_ = cudaGetLastError();                                                  \
    if (e_ != cudaSuccess) {                                                              \
      vi_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
      return VI_ERR_CUDA;                                                                 \
    }                                                                                     \
  } while (0)

int vi_num_sms();
// 2-D row-major TMA tensor map over bf16 / fp16 elements, 128-byte swizzle, boxes of 64 columns x box_rows rows (vi_api.cu)
int vi_make_tmap_h16(CUtensorMap* map, const void* ptr, int f16, uint64_t cols, uint64_t rows, uint64_t ld_elems, uint32_t box_rows);
bool vi_pdl_enabled();      // programmatic dependent launch on every kernel of the library (VI_PDL=0 disables)
void vi_count_launch();     // one more kernel launched by the library (vi_launch_count)

// Launch with the programmatic-stream-serialization attribute: the kernel may start (and run its prologue) while
// its predecessor in the stream is still draining; it calls pdl_wait() before touching global memory.  cluster > 1
// groups that many consecutive CTAs into a cluster (the CTA-pair kernels).  Every kernel of the library is launched here.
#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline cudaError_t vi_launch_cluster(void (*kern)(KArgs...), unsigned cluster, dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  unsigned nattr = 0;
  if (vi_pdl_enabled()) {
    attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[nattr].val.programmaticStreamSerializationAllowed = 1;
    ++nattr;
  }
  if (cluster > 1) {
    attr[nattr].id = cudaLaunchAttributeClusterDimension;
    attr[nattr].val.clusterDim.x = cluster;
    attr[nattr].val.clusterDim.y = 1;
    attr[nattr].val.clusterDim.z = 1;
    ++nattr;
  }
  cfg.attrs = attr;
  cfg.numAttrs = nattr;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
  if (e == cudaSuccess) vi_count_launch();
  return e;
}
template <typename... KArgs, typename... Args>
inline cudaError_t vi_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  return vi_launch_cluster(kern, 1, grid, block, smem, st, args...);
}
#endif

typedef __nv_bfloat16 bf16;

// ----------------------------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// Programmatic dependent launch: let the next kernel of the stream begin its prologue now; wait for the previous
// kernel's memory before reading (or overwriting) anything it may touch.  Both are no-ops without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() { pdl_launch_dependents(); pdl_wait(); }
// NOTE on loads: a kernel launched this way is RESIDENT before its predecessor has finished writing, so data produced by
// earlier kernels must never be read through the non-coherent path (ld.global.nc: __ldg, or loads the compiler proves
// read-only from `const T* __restrict__`): such a load may hit a stale L1 line of the SM.  The kernels of this library
// therefore take plain `const T*` inputs (coherent ld.global), cp.async.cg or TMA.

// Counter-based dropout mask: element `idx` of dropout site `site` is kept iff hash(idx, seed + site) >= threshold, with
// threshold = p * 2^32.  `seed` lives in device memory (it advances once per optimiser step, also inside replayed CUDA
// graphs); the same (seed, site, idx) regenerates the mask in the backward pass, so no mask is ever stored.
__device__ __forceinline__ uint32_t vi_hash32(uint32_t idx, uint32_t key) {
  uint32_t h = idx * 0x9E3779B1u + key;
  h ^= h >> 16; h *= 0x7FEB352Du;
  h ^= h >> 15; h *= 0x846CA68Bu;
  h ^= h >> 16;
  return h;
}
__device__ __forceinline__ uint32_t vi_drop_key(const uint32_t* seed, uint32_t site) {
  return vi_hash32(site, *seed ^ 0xA511E9B3u);
}
__host__ __device__ __forceinline__ uint32_t vi_drop_threshold(float p) {
  const double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float gelu_erf(float x) { return x * 0.5f * (1.0f + erff(x * 0.70710678118654752440f)); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

// 16-bit operand formats of the forward kernels: bf16, or fp16 with saturation (+-65504 instead of inf) - see vi_gemm16
__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ uint32_t pack_h16x2(float lo, float hi, bool f16) { return f16 ? pack_f16x2_sat(lo, hi) : pack_bf16x2(lo, hi); }

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol bug becomes a trap (an error the host sees) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  long long t0 = 0;
  uint32_t spins = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!done) {
      if (++spins == 1024u) t0 = clock64();
      if (spins > 1024u && (spins & 1023u) == 0 && clock64() - t0 > 4000000000LL) __trap();
    }
  } while (!done);
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMA --------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i owns lane i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

#endif  // __CUDACC__
