// vi_api.cu - library-level entry points: init, version, thread-local error string, launch counter.
#include "vi_common.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <atomic>

static thread_local char g_err[512] = "";
static int g_num_sms = 0;

void vi_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int vi_num_sms() {
  if (g_num_sms == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      g_num_sms = n;
    else
      g_num_sms = 148;
  }
  return g_num_sms;
}

bool vi_pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("VI_PDL");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on != 0;
}

int vi_attn_init();
int vi_attn_bwd_init();       // vi_attn_bwd.cu
int vi_attn_bwd_f32_init();   // vi_bwd.cu

// ---- TMA tensor maps (driver entry point resolved once per process) -------------------------------------------------
#include <mutex>
typedef CUresult (*ViEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static ViEncodeTiledFn g_vi_encode = nullptr;
static std::once_flag g_vi_encode_once;

// 2-D row-major tensor map over 16-bit elements with the 128-byte swizzle: boxes of 64 columns x box_rows rows
int vi_make_tmap_h16(CUtensorMap* map, const void* ptr, int f16, uint64_t cols, uint64_t rows, uint64_t ld_elems, uint32_t box_rows) {
  std::call_once(g_vi_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      g_vi_encode = reinterpret_cast<ViEncodeTiledFn>(fn);
  });
  if (!g_vi_encode) {
    vi_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return VI_ERR_CUDA;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld_elems * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_vi_encode(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr),
                           gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vi_set_error("cuTensorMapEncodeTiled failed with CUresult %d (ptr=%p cols=%llu rows=%llu ld=%llu box=64x%u)", (int)r, ptr,
                 (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)ld_elems, box_rows);
    return VI_ERR_CUDA;
  }
  return VI_OK;
}

static std::atomic<int64_t> g_launches{0};

void vi_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

extern "C" int64_t vi_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int vi_version(void) { return 106; }   // 0.1.6

extern "C" const char* vi_last_error(void) { return g_err; }

extern "C" int vi_init(int device) {
  VI_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  VI_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    vi_set_error("libvlnimagine is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    return VI_ERR_UNSUPPORTED;
  }
  g_num_sms = prop.multiProcessorCount;
  if (int rc = vi_attn_init()) return rc;
  if (int rc = vi_attn_bwd_init()) return rc;
  if (int rc = vi_attn_bwd_f32_init()) return rc;
  return VI_OK;
}
