// vi_gemm_tc.cu - bf16 GEMM on the 5th-gen tensor cores: Y = epi(X W^T + bias) + residual.
//
// Persistent, warp-specialised, one CTA (or one CTA pair) per SM walking output tiles:
//   warp 0      : TMA producer  - cp.async.bulk.tensor loads of the X (128 x 64) and W (BN x 64) k-blocks into
//                 a STAGES-deep shared-memory ring (128B swizzle), completion counted on mbarriers;
//   warp 1      : MMA issuer    - one thread issues tcgen05.mma (K=16 per instruction) accumulating fp32 in
//                 TMEM; tcgen05.commit frees ring slots and publishes finished accumulators;
//   warp 2      : TMEM allocator (2 x BN columns: the accumulator is double buffered, so the epilogue of
//                 tile i overlaps the main loop of tile i+1);
//   warps 4..11 : epilogue      - tcgen05.ld (32 lanes x 32 columns per warp), + bias, GELU / ReLU, + residual,
//                 staged through swizzled shared memory and written with TMA stores; the fp32 residual tile
//                 is fetched by TMA into the same staging buffer, so every global access is a bulk copy.
// PAIR mode (cta_group::2): two CTAs of a cluster work on one 256 x BN tile; each loads its own 128 rows of X
// and half of the W tile, the leader issues M=256 MMAs that read both CTAs' shared memory, and each CTA drains
// its own half of the accumulator.  This halves the W traffic per flop, which is what bounds a 128 x BN tile
// (L2 -> SM bandwidth, B300_MICROARCH.md "TMA chip-throughput").
// The grouped form lets consecutive row ranges of X use different weight blocks of a stacked W (DUET's
// global / local encoders, HAMT's language / vision streams) in a single launch.
//
// Replaces nn.Linear + its following activation / residual in the reference
// (VLN-DUET/map_nav_src/models/vilmodel.py:93-95,147,172,186,315-317; transformer.py:178,181).
#include "vi_common.cuh"

#include <mutex>

namespace {

constexpr int BM = 128;
constexpr int BK = 64;           // 64 bf16 = 128 bytes = one swizzle-128B row
constexpr int UMMA_K = 16;
constexpr int MAX_GROUPS = 4;
constexpr int EPI_WARPS = 8;
constexpr int NUM_THREADS = 128 + EPI_WARPS * 32;
constexpr int MAX_CPW = 4;                             // 32-column chunks per epilogue warp per tile (BN <= 256)
// per epilogue warp: the two per-column vectors of the current chunk (bias | folded constant, LayerNorm vector), 32 floats
// each; the next chunk's slices wait in registers until the current ones have been read
constexpr int VEC_BYTES = EPI_WARPS * 2 * 32 * 4;
// what the epilogue writes: a 16-bit tile (bf16 / fp16), an fp32 tile, or both (fp32 residual stream + 16-bit operand copy)
enum { OUT_H16 = 0, OUT_F32 = 1, OUT_DUAL = 2 };
// staging per epilogue warp: two buffers of 32 rows x 32 columns (fp32: 128-byte rows; 16-bit: 64-byte rows).  OUT_DUAL: the two
// fp32 buffers plus ONE 16-bit buffer behind them - a dual output always has a residual, whose prefetch already waits for every
// outstanding store of the warp at the top of each chunk, so the 16-bit copy needs no second buffer
__host__ __device__ constexpr int epi_buf_bytes(int om) { return om == OUT_H16 ? 2048 : 4096; }
__host__ __device__ constexpr int epi_warp_bytes(int om) { return 2 * epi_buf_bytes(om) + (om == OUT_DUAL ? 2048 : 0); }
__host__ __device__ constexpr int epi_bytes(int om) { return EPI_WARPS * epi_warp_bytes(om); }
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;            // clears the CTA-rank bit of a shared::cluster address (pair leader)

enum { LN_NONE = 0, LN_FOLD = 1, LN_RESIDUAL = 2 };

struct GemmParams {
  const float* bias;               // [n_groups * N]; LN_FOLD: the folded constant c = W beta + b; LN_RESIDUAL: beta + b
  const float* vec_a;              // LN_FOLD: s = row sums of the folded weight; LN_RESIDUAL: gamma   ([n_groups * N])
  const float2* stats_in;          // [stats_chunks][stats_ld] (mean, M2) of every 32-column chunk of the rows to normalise
  float2* stats_out;               // [N / 32][stats_ld] (mean, M2) of every 32-column chunk of the output rows, or NULL
  long long stats_ld;
  int stats_chunks;
  int ln_mode;
  float ln_eps;
  int fmt_f16;                     // 16-bit operands / outputs are fp16 (else bf16)
  int has_residual;
  int y_f32;
  int M, N, K;
  int epilogue;
  int n_groups;
  int group_tile_end[MAX_GROUPS];      // in units of 128-row tiles
  int num_m_tiles, num_n_tiles;        // m tiles in units of the launch's tile height (128, or 256 in PAIR mode)
};

__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t saddr) {
  // UMMA shared-memory descriptor, K-major operand, 128-byte swizzle:
  //   bits [0,14) start address >> 4; [16,30) leading byte offset >> 4 (unused for swizzled K-major, 1);
  //   [32,46) stride byte offset >> 4 = 1024 B between 8-row groups; [46,48) descriptor version 1 (sm_100);
  //   [61,64) layout type 2 = SWIZZLE_128B.
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__host__ __device__ constexpr uint32_t make_idesc(int mma_m, int mma_n, bool f16) {
  // kind::f16 instruction descriptor: D=f32 (bits 4-5 = 1), A / B format at bits 7-9 / 10-12 (0 = fp16, 1 = bf16),
  // both operands K-major (bits 15,16 = 0), N>>3 at bits 17-22, M>>4 at bits 24-28.
  return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | ((uint32_t)(mma_n >> 3) << 17) | ((uint32_t)(mma_m >> 4) << 24);
}

// Packed fp32 pair arithmetic (FFMA2 on sm_100): one instruction for two elements.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 bcast2(float v) { return make_float2(v, v); }

// erf-form GELU (D/models/vilmodel.py:32-38) of two elements without any MUFU op: erf(x / sqrt 2) is an odd degree-19
// polynomial in t = clamp(x, +-4.5) / 4.5 (least-squares fit on Chebyshev nodes; |erf error| < 8e-6 on the interval,
// erfc(4.5 / sqrt 2) = 6.8e-6 beyond it), evaluated with packed FFMA2: 13 packed + 4 scalar instructions per PAIR.
// Measured against the exact form over x ~ N(0, 1): RMS error = 0.3 % of the bf16 rounding error of the result.
// The A&S 7.1.26 form it replaces cost two MUFU ops and ~14 FMAs per ELEMENT and was the exposed part of the FFN1 epilogue.
__device__ __forceinline__ void gelu_pair(float& x0, float& x1) {
  const float2 x = make_float2(x0, x1);
  const float2 xc = make_float2(fminf(fmaxf(x0, -4.5f), 4.5f), fminf(fmaxf(x1, -4.5f), 4.5f));
  const float2 t = ffma2(xc, bcast2(1.0f / 4.5f), bcast2(0.f));
  const float2 u = ffma2(t, t, bcast2(0.f));
  float2 p = bcast2(-8.882999948e+00f);
  p = ffma2(p, u, bcast2(5.144924412e+01f));
  p = ffma2(p, u, bcast2(-1.328671530e+02f));
  p = ffma2(p, u, bcast2(2.037066147e+02f));
  p = ffma2(p, u, bcast2(-2.090744719e+02f));
  p = ffma2(p, u, bcast2(1.541237008e+02f));
  p = ffma2(p, u, bcast2(-8.545582162e+01f));
  p = ffma2(p, u, bcast2(3.651658807e+01f));
  p = ffma2(p, u, bcast2(-1.210606152e+01f));
  p = ffma2(p, u, bcast2(3.590346739e+00f));
  const float2 e = ffma2(p, t, bcast2(0.f));                 // erf(x / sqrt 2)
  const float2 hx = ffma2(x, bcast2(0.5f), bcast2(0.f));
  const float2 r = ffma2(hx, e, hx);
  x0 = r.x; x1 = r.y;
}
// ---- PTX helpers that exist only for this kernel ---------------------------------------------------------------
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(tmap), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {          // one lane of a converged warp
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred px;\n\telect.sync _|px, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, px;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// pair mode: this CTA's TMA load completes on the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(tmap), "r"(bar & PEER_MASK), "r"(c0), "r"(c1), "l"(0x1000000000000000ull)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_MASK) : "memory");
}
template <bool PAIR> __device__ __forceinline__ void tc_commit_t(uint32_t bar) {
  if constexpr (PAIR) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
  } else {
    tc_commit(bar);
  }
}
template <bool PAIR>
__device__ __forceinline__ void tc_mma_t(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  if constexpr (PAIR) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
  } else {
    tc_mma_bf16(d_tmem, adesc, bdesc, idesc, acc);
  }
}
template <bool PAIR> __device__ __forceinline__ void tmem_alloc_t(uint32_t dst_smem, uint32_t ncols) {
  if constexpr (PAIR) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  } else {
    tmem_alloc(dst_smem, ncols);
    tmem_relinquish();
  }
}
template <bool PAIR> __device__ __forceinline__ void tmem_dealloc_t(uint32_t taddr, uint32_t ncols) {
  if constexpr (PAIR) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  } else {
    tmem_dealloc(taddr, ncols);
  }
}

__host__ __device__ constexpr uint32_t tmem_cols_for(int bn) { return 2 * bn <= 128 ? 128u : (2 * bn <= 256 ? 256u : 512u); }

template <int BN, int STAGES, bool PAIR, int OUTMODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmR,
                    const __grid_constant__ CUtensorMap tmY2, const GemmParams p) {
  constexpr int BN_CTA = PAIR ? BN / 2 : BN;         // rows of the W tile this CTA stages
  constexpr int A_BYTES = BM * BK * 2;
  constexpr int B_BYTES = BN_CTA * BK * 2;
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = tmem_cols_for(BN);
  constexpr int NCHUNK = BN / 32;                    // 32-column epilogue chunks per tile
  constexpr int EPI_BUF = epi_buf_bytes(OUTMODE);
  constexpr bool HAS_F32 = OUTMODE != OUT_H16;       // fp32 tile staged at offset 0 of a buffer
  constexpr bool HAS_H16 = OUTMODE != OUT_F32;       // 16-bit tile staged at offset 0 (OUT_H16) or 4096 (OUT_DUAL)
  constexpr int EPI_WARP = epi_warp_bytes(OUTMODE);
  constexpr int TILES_PER_M = PAIR ? 2 : 1;          // 128-row tiles per m index
  static_assert(BN % 32 == 0 && BN >= 64 && BN <= 256, "tile N");
  static_assert(A_BYTES % 1024 == 0 && B_BYTES % 1024 == 0, "operand tiles must keep the 1024-byte swizzle alignment");

  // The kernel has no static shared memory, so the dynamic window starts at offset 0 of the CTA's shared memory
  // and is 1024-byte aligned, which the 128B-swizzled tiles need (checked below: a misaligned base traps).
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* epi_smem = smem + STAGES * STAGE_BYTES;
  float* vec_smem = reinterpret_cast<float*>(epi_smem + epi_bytes(OUTMODE));
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem + epi_bytes(OUTMODE) + VEC_BYTES);
  // barrier slots: full[S], empty[S], tfull[2], tempty[2], rbar[EPI_WARPS][2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + 2 * EPI_WARPS);

  const uint32_t smem_base = smem_u32(smem);
  if (smem_base & 1023u) __trap();
  const uint32_t epi_base = smem_u32(epi_smem);
  const uint32_t bar_base = smem_u32(bars);
  auto a_addr = [&](int s) { return smem_base + (uint32_t)(s * STAGE_BYTES); };
  auto b_addr = [&](int s) { return smem_base + (uint32_t)(s * STAGE_BYTES + A_BYTES); };
  auto full_bar = [&](int s) { return bar_base + 8u * (uint32_t)s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (uint32_t)(STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (uint32_t)(2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (uint32_t)(2 * STAGES + 2 + a); };
  auto res_bar = [&](int w, int b) { return bar_base + 8u * (uint32_t)(2 * STAGES + 4 + 2 * w + b); };

  pdl_launch_dependents();                            // the next kernel may begin its own prologue
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;          // tile walker id (CTA or pair)
  const int n_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmY);
    if (p.has_residual) tma_prefetch_desc(&tmR);
    if (OUTMODE == OUT_DUAL) tma_prefetch_desc(&tmY2);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), PAIR ? 2 * EPI_WARPS : EPI_WARPS);      // one arrive per epilogue warp (of both CTAs)
    }
    for (int w = 0; w < EPI_WARPS; ++w) {
      mbar_init(res_bar(w, 0), 1);
      mbar_init(res_bar(w, 1), 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc_t<PAIR>(smem_u32(tmem_slot), TMEM_COLS);
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                         // everything above overlapped the previous kernel's tail

  const int total_tiles = p.num_m_tiles * p.num_n_tiles;
  const int num_kb = p.K / BK;

  auto group_of = [&](int mt128) {                     // group ends ascend: count the ends at or below the tile (static indices)
    int g = 0;
#pragma unroll
    for (int i = 0; i < MAX_GROUPS - 1; ++i) g += (i < p.n_groups - 1 && mt128 >= p.group_tile_end[i]) ? 1 : 0;
    return g;
  };

  if (warp == 0) {
    // ------------------------------- TMA producer (whole warp converged, one elected lane issues) -----------
    int s = 0;
    uint32_t ph = 0;
    for (int t = worker; t < total_tiles; t += n_workers) {
      const int mt = t / p.num_n_tiles, nt = t - mt * p.num_n_tiles;
      const int arow = (mt * TILES_PER_M + (int)rank) * BM;
      const int wrow = group_of(mt * TILES_PER_M) * p.N + nt * BN + (int)rank * BN_CTA;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(empty_bar(s), ph ^ 1u);
        if (elect_one()) {
          if constexpr (PAIR) {
            if (rank == 0) mbar_expect_tx(full_bar(s), 2 * STAGE_BYTES);       // both CTAs' bytes land on the leader
            tma_load_2d_pair(a_addr(s), &tmA, full_bar(s), kb * BK, arow);
            tma_load_2d_pair(b_addr(s), &tmB, full_bar(s), kb * BK, wrow);
          } else {
            mbar_expect_tx(full_bar(s), STAGE_BYTES);
            tma_load_2d(a_addr(s), &tmA, full_bar(s), kb * BK, arow);
            tma_load_2d(b_addr(s), &tmB, full_bar(s), kb * BK, wrow);
          }
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer (pair: leader only; warp converged, elected lane issues) ----
    if (rank == 0) {
      const uint32_t idesc = make_idesc(PAIR ? 256 : 128, BN, p.fmt_f16 != 0);
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int t = worker; t < total_tiles; t += n_workers, ++it) {
        const int acc = it & 1;
        const uint32_t acc_ph = (uint32_t)(it >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_ph ^ 1u);      // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(s), ph);                 // TMA bytes have landed (in both CTAs)
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = make_sw128_kmajor_desc(a_addr(s));
            const uint64_t bdesc = make_sw128_kmajor_desc(b_addr(s));
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              // advance 16 elements (32 bytes) along K inside the swizzle span: +2 in 16-byte units
              tc_mma_t<PAIR>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (uint32_t)((kb | k) != 0));
            }
            tc_commit_t<PAIR>(empty_bar(s));          // frees the ring slot (of both CTAs) when the MMAs retire
            if (kb == num_kb - 1) tc_commit_t<PAIR>(tfull_bar(acc));   // accumulator complete -> epilogue (both CTAs)
          }
          __syncwarp();
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------- epilogue -----------------------------------------------
    const int ew = warp - 4;                          // 0..7
    const int quarter = warp & 3;                     // TMEM lane quarter this warp may read
    const int half = ew >> 2;                         // which interleaved half of the column chunks
    constexpr int CPW0 = (NCHUNK + 1) / 2, CPW1 = NCHUNK / 2;
    const int cpw = half ? CPW1 : CPW0;               // chunks per tile for this warp: half, half+2, ...
    const uint32_t my_buf = epi_base + (uint32_t)(ew * EPI_WARP);
    const uint32_t my_h16 = my_buf + (uint32_t)(2 * EPI_BUF);      // OUT_DUAL: the single 16-bit staging buffer
    float* my_vec = vec_smem + ew * 64;               // [2][32]: per-column vectors of the current chunk
    const uint32_t my_vec_u = smem_u32(my_vec);
    const bool res = p.has_residual != 0;
    const int ln_mode = p.ln_mode;
    const int row_in_tile = (int)rank * BM + quarter * 32;
    const bool has_v0 = p.bias != nullptr, has_v1 = p.vec_a != nullptr;

    auto issue_residual = [&](int n, int row0, int col0) {          // lane 0 only
      const uint32_t bar = res_bar(ew, n & 1);
      mbar_expect_tx(bar, 4096);
      tma_load_2d(my_buf + (uint32_t)((n & 1) * EPI_BUF), &tmR, bar, col0, row0);
    };
    // this lane's elements of the per-column vectors for (group g, column c)
    auto load_vecs = [&](int g, int c, float& a0, float& a1) {
      const long long o = (long long)g * p.N + c + lane;
      a0 = has_v0 ? *(p.bias + o) : 0.f;
      a1 = has_v1 ? *(p.vec_a + o) : 0.f;
    };
    auto park_vecs = [&](float a0, float a1) {
      float* d = my_vec + lane;
      if (has_v0) d[0] = a0;
      if (has_v1) d[32] = a1;
    };

    int n = 0, it = 0;
    if (worker < total_tiles) {
      const int mt = worker / p.num_n_tiles, nt = worker - mt * p.num_n_tiles;
      if (res && lane == 0) issue_residual(0, mt * TILES_PER_M * BM + row_in_tile, nt * BN + half * 32);
      float a0, a1;
      load_vecs(group_of(mt * TILES_PER_M), nt * BN + half * 32, a0, a1);
      park_vecs(a0, a1);
      __syncwarp();
    }
    for (int t = worker; t < total_tiles; t += n_workers, ++it) {
      const int mt = t / p.num_n_tiles, nt = t - mt * p.num_n_tiles;
      const int g = group_of(mt * TILES_PER_M);
      const int row0 = mt * TILES_PER_M * BM + row_in_tile;
      const int tcol0 = nt * BN + half * 32;          // first column chunk of this warp; the next ones are +64 apart
      // first chunk of the NEXT tile (for the residual prefetch that crosses the tile boundary)
      const int tn = t + n_workers;
      const int mtn = tn / p.num_n_tiles, ntn = tn - mtn * p.num_n_tiles;
      const int row0n = mtn * TILES_PER_M * BM + row_in_tile, tcol0n = ntn * BN + half * 32;
      const int gn = tn < total_tiles ? group_of(mtn * TILES_PER_M) : g;
      const int acc = it & 1;
      const uint32_t acc_ph = (uint32_t)(it >> 1) & 1u;
      const long long grow = (long long)row0 + lane;  // this thread's output row
      const bool row_ok = grow < p.M;

      // LayerNorm statistics of this thread's row from the producer's per-chunk (mean, M2) partials (Chan's combination
      // of equal-sized groups), fetched while the main loop of the tile is still running
      float rstd = 1.f, rm = 0.f;                     // 1 / sigma and mu / sigma
      if (ln_mode != LN_NONE) {
        float sm = 0.f, sq = 0.f, m2 = 0.f;
        if (row_ok) {
          const float2* sp = p.stats_in + grow;
          for (int c0 = 0; c0 < p.stats_chunks; c0 += 24) {       // 24 chunks = one 768-wide LayerNorm: ONE round trip to L2
            float2 pr[24];
#pragma unroll
            for (int c = 0; c < 24; ++c) pr[c] = (c0 + c < p.stats_chunks) ? *(sp + (long long)(c0 + c) * p.stats_ld) : make_float2(0.f, 0.f);
#pragma unroll
            for (int c = 0; c < 24; ++c) { sm += pr[c].x; sq = fmaf(pr[c].x, pr[c].x, sq); m2 += pr[c].y; }
          }
        }
        const float inv_c = 1.0f / (float)p.stats_chunks;
        const float mean = sm * inv_c;
        const float var = fmaxf((m2 + 32.0f * (sq - sm * mean)) * inv_c * (1.0f / 32.0f), 0.f);
        rstd = rsqrtf(var + p.ln_eps);
        rm = rstd * mean;
      }

      mbar_wait(tfull_bar(acc), acc_ph);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + half * 32);
      uint32_t r[2][32];
      tmem_ld_32x32(tbase, r[0]);
#pragma unroll
      for (int k = 0; k < MAX_CPW; ++k) {
        if (k < cpw) {
          const uint32_t buf = my_buf + (uint32_t)((n & 1) * EPI_BUF);
          const uint32_t vec_u = my_vec_u;
          const int col0 = tcol0 + k * 64;
          const bool last = k == cpw - 1;
          if (lane == 0) {
            if (res) {
              if (!last || tn < total_tiles) {
                bulk_wait_read<0>();                  // the store that last used the other buffer has read it
                issue_residual(n + 1, last ? row0n : row0, last ? tcol0n : col0 + 64);
              } else if (OUTMODE == OUT_DUAL) {
                bulk_wait_read<0>();                  // the single 16-bit staging buffer: the previous chunk's copy has been read
              }
            } else if (OUTMODE == OUT_DUAL) {
              bulk_wait_read<0>();                    // single 16-bit staging buffer: wait for the previous chunk's stores
            } else {
              bulk_wait_read<1>();                    // the store issued two chunks ago has read this buffer
            }
          }
          // per-column vectors of the NEXT chunk (possibly the first one of the next tile): loaded now, parked at the end
          float nv0 = 0.f, nv1 = 0.f;
          if (!last) load_vecs(g, col0 + 64, nv0, nv1);
          else if (tn < total_tiles) load_vecs(gn, tcol0n, nv0, nv1);
          tmem_ld_wait();
          if (!last) {
            tmem_ld_32x32(tbase + (uint32_t)((k + 1) * 64), r[(k + 1) & 1]);   // next chunk in flight during the math
          } else {                                    // accumulator fully read by this warp: hand it back early
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (PAIR) mbar_arrive_leader(tempty_bar(acc)); else mbar_arrive(tempty_bar(acc));
            }
          }
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[k & 1][j]);
          if (ln_mode == LN_FOLD) {
            // LayerNorm folded into the weights: y = (acc - mu * s_n) / sigma + c_n   (W gamma in the operand, s = its row sums)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 c4, s4;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(c4.x), "=f"(c4.y), "=f"(c4.z), "=f"(c4.w) : "r"(vec_u + (uint32_t)(j * 16)));
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(s4.x), "=f"(s4.y), "=f"(s4.z), "=f"(s4.w) : "r"(vec_u + (uint32_t)(128 + j * 16)));
              const float2 nrm = bcast2(-rm), rs = bcast2(rstd);
              const float2 t0 = ffma2(nrm, make_float2(s4.x, s4.y), make_float2(c4.x, c4.y));
              const float2 t1 = ffma2(nrm, make_float2(s4.z, s4.w), make_float2(c4.z, c4.w));
              const float2 y0 = ffma2(rs, make_float2(v[4 * j], v[4 * j + 1]), t0);
              const float2 y1 = ffma2(rs, make_float2(v[4 * j + 2], v[4 * j + 3]), t1);
              v[4 * j] = y0.x; v[4 * j + 1] = y0.y; v[4 * j + 2] = y1.x; v[4 * j + 3] = y1.y;
            }
          } else if (has_v0 && ln_mode != LN_RESIDUAL) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 b;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                           : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(vec_u + (uint32_t)(j * 16)));
              v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
          }
          if (p.epilogue == VI_EPI_GELU) {
#pragma unroll
            for (int j = 0; j < 16; ++j) gelu_pair(v[2 * j], v[2 * j + 1]);
          } else if (p.epilogue == VI_EPI_RELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
          }
          __syncwarp();                               // lane 0's wait on the staging buffer covers the whole warp
          if (res) {
            mbar_wait(res_bar(ew, n & 1), (uint32_t)(n >> 1) & 1u);
            // residual tile: 32 rows x 128 B, 128B-swizzled: 16-byte chunk j of row r sits at j ^ (r & 7)
            const uint32_t rowb = buf + (uint32_t)(lane * 128);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 q;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                           : "=f"(q.x), "=f"(q.y), "=f"(q.z), "=f"(q.w) : "r"(rowb + (uint32_t)((j ^ (lane & 7)) << 4)));
              if (ln_mode == LN_RESIDUAL) {
                // the residual is LayerNorm(raw) of the producer: (raw - mu) / sigma * gamma + beta, from the raw fp32 rows
                // (the vector in slot 0 is beta + this layer's bias)
                float4 g4, b4;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(g4.x), "=f"(g4.y), "=f"(g4.z), "=f"(g4.w) : "r"(vec_u + (uint32_t)(128 + j * 16)));
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(vec_u + (uint32_t)(j * 16)));
                const float2 nrm = bcast2(-rm), rs = bcast2(rstd);
                const float2 n0 = ffma2(make_float2(q.x, q.y), rs, nrm), n1 = ffma2(make_float2(q.z, q.w), rs, nrm);
                const float2 r0 = ffma2(n0, make_float2(g4.x, g4.y), make_float2(b4.x, b4.y));
                const float2 r1 = ffma2(n1, make_float2(g4.z, g4.w), make_float2(b4.z, b4.w));
                q.x = r0.x; q.y = r0.y; q.z = r1.x; q.w = r1.y;
              }
              v[4 * j] += q.x; v[4 * j + 1] += q.y; v[4 * j + 2] += q.z; v[4 * j + 3] += q.w;
            }
          }
          if (p.stats_out) {
            // (mean, M2) of this row's 32 columns: the consumer of the LayerNorm that follows combines the chunks
            float sm = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) sm += v[j];
            const float mean = sm * (1.0f / 32.0f);
            float m2 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) { const float d = v[j] - mean; m2 = fmaf(d, d, m2); }
            if (row_ok) *(p.stats_out + (long long)(col0 >> 5) * p.stats_ld + grow) = make_float2(mean, m2);
          }
          if constexpr (HAS_F32) {
            const uint32_t rowb = buf + (uint32_t)(lane * 128);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};"
                           ::"r"(rowb + (uint32_t)((j ^ (lane & 7)) << 4)), "f"(v[4 * j]), "f"(v[4 * j + 1]), "f"(v[4 * j + 2]),
                           "f"(v[4 * j + 3]) : "memory");
          }
          if constexpr (HAS_H16) {
            // 16-bit rows are 64 B, 64B-swizzled: chunk j of row r sits at j ^ ((r >> 1) & 3)
            const uint32_t rowb = (OUTMODE == OUT_DUAL ? my_h16 : buf) + (uint32_t)(lane * 64);
            uint32_t h[16];
            if (p.fmt_f16) {
#pragma unroll
              for (int j = 0; j < 16; ++j) h[j] = pack_f16x2_sat(v[2 * j], v[2 * j + 1]);
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) h[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
              asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};"
                           ::"r"(rowb + (uint32_t)((j ^ ((lane >> 1) & 3)) << 4)), "r"(h[4 * j]), "r"(h[4 * j + 1]),
                           "r"(h[4 * j + 2]), "r"(h[4 * j + 3]) : "memory");
          }
          __syncwarp();                               // every lane has read the current vectors
          park_vecs(nv0, nv1);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmY, buf, col0, row0);      // rows beyond M are clipped by the tensor map
            if constexpr (OUTMODE == OUT_DUAL) tma_store_2d(&tmY2, my_h16, col0, row0);
            bulk_commit();
          }
          ++n;
        }
      }
    }
    if (lane == 0) bulk_wait_all();
  }

  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_t<PAIR>(tmem_base, TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
std::once_flag g_encode_once;

int resolve_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  if (!g_encode) {
    vi_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return VI_ERR_CUDA;
  }
  return VI_OK;
}

// 2D row-major tensor map: inner dim contiguous, `box_inner x box_rows` boxes
int make_map(CUtensorMap* map, const void* ptr, CUtensorMapDataType dt, int elem_bytes, uint64_t inner, uint64_t rows,
             uint64_t ld_elems, uint32_t box_inner, uint32_t box_rows, CUtensorMapSwizzle sw) {
  cuuint64_t gdim[2] = {inner, rows};
  cuuint64_t gstride[1] = {ld_elems * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vi_set_error("cuTensorMapEncodeTiled failed with CUresult %d (ptr=%p inner=%llu rows=%llu ld=%llu box=%ux%u)",
                 (int)r, ptr, (unsigned long long)inner, (unsigned long long)rows, (unsigned long long)ld_elems, box_inner,
                 box_rows);
    return VI_ERR_CUDA;
  }
  return VI_OK;
}

template <int BN, int STAGES, bool PAIR, int OUTMODE>
constexpr int smem_bytes() {
  return STAGES * (BM * BK * 2 + (PAIR ? BN / 2 : BN) * BK * 2) + epi_bytes(OUTMODE) + VEC_BYTES +
         (2 * STAGES + 4 + 2 * EPI_WARPS) * 8 + 16;
}

struct Maps { CUtensorMap a, b, y, r, y2; };

template <int BN, int STAGES, bool PAIR, int OUTMODE>
int launch(const Maps& m, const GemmParams& p, int grid, cudaStream_t st) {
  static_assert(smem_bytes<BN, STAGES, PAIR, OUTMODE>() <= 232448, "shared memory budget");
  static bool attr_set = false;          // idempotent; races only repeat the same call
  auto kern = gemm_bf16_tc_kernel<BN, STAGES, PAIR, OUTMODE>;
  if (!attr_set) {
    VI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes<BN, STAGES, PAIR, OUTMODE>()));
    attr_set = true;
  }
  VI_CUDA(vi_launch_cluster(kern, PAIR ? 2 : 1, dim3((unsigned)grid), dim3(NUM_THREADS),
                            (size_t)smem_bytes<BN, STAGES, PAIR, OUTMODE>(), st, m.a, m.b, m.y, m.r, m.y2, p));
  return VI_OK;
}

struct Choice { int bn; bool pair; };

// Tile choice by a two-term cost model (cycles): the tensor pipe (waves x MMA time of a tile) against the
// L2 -> SM operand traffic of the whole problem (about 6300 B/cycle chip-wide), plus one exposed epilogue.
Choice pick_tile(int M, int N, int K, int nsm, bool pair_ok) {
  Choice best = {64, false};
  double best_cost = 1e30;
  const int cands[5] = {256, 192, 128, 96, 64};
  for (int pr = 1; pr >= 0; --pr) {
    if (pr && !pair_ok) continue;
    for (int i = 0; i < 5; ++i) {
      const int bn = cands[i];
      if (N % bn) continue;
      if (pr && bn < 128) continue;
      const int tm = pr ? 256 : 128;
      const long long m_tiles = (M + tm - 1) / tm;
      const long long tiles = m_tiles * (N / bn);
      const long long workers = pr ? nsm / 2 : nsm;
      const long long waves = (tiles + workers - 1) / workers;
      const double kb = K / 64.0;
      const double mma = (double)waves * kb * 4.0 * (bn / 2.0);                 // cycles: K=16 MMA = bn/2 (M=128 per SM)
      const double bytes = (double)tiles * kb * (tm * 128.0 + bn * 128.0);
      const double l2 = bytes / 6300.0;
      const double epi = 1500.0 + 10.0 * bn;
      const double cost = (mma > l2 ? mma : l2) + epi + (double)waves * 300.0;
      if (cost < best_cost - 1e-9) { best_cost = cost; best = Choice{bn, pr != 0}; }
    }
  }
  return best;
}

}  // namespace

extern "C" int vi_gemm16(const vi_gemm_args* args, vi_stream_t stream) {
  VI_CHECK_ARG(args, "vi_gemm16: null args");
  const vi_gemm_args& a = *args;
  const int M = a.M, N = a.N, K = a.K, n_groups = a.n_groups;
  VI_CHECK_ARG(a.x && a.w && a.y, "vi_gemm16: null operand");
  VI_CHECK_ARG(M > 0 && N > 0 && K > 0, "vi_gemm16: empty problem M=%d N=%d K=%d", M, N, K);
  VI_CHECK_ARG(K % BK == 0, "vi_gemm16: K=%d must be a multiple of %d", K, BK);
  VI_CHECK_ARG(N % 64 == 0, "vi_gemm16: N=%d must be a multiple of 64", N);
  VI_CHECK_ARG(a.in_dtype == VI_DT_BF16 || a.in_dtype == VI_DT_F16, "vi_gemm16: operands must be bf16 or fp16 (in_dtype %d)", a.in_dtype);
  VI_CHECK_ARG(a.ldx % 8 == 0 && a.ldx >= K, "vi_gemm16: ldx=%lld must be >= K and a multiple of 8", (long long)a.ldx);
  VI_CHECK_ARG(((uintptr_t)a.x & 15) == 0 && ((uintptr_t)a.w & 15) == 0 && ((uintptr_t)a.y & 15) == 0,
               "vi_gemm16: operands must be 16-byte aligned");
  VI_CHECK_ARG(a.ldy >= N && a.ldy % 8 == 0, "vi_gemm16: ldy=%lld must be >= N and a multiple of 8", (long long)a.ldy);
  VI_CHECK_ARG(!a.residual || (a.ldr >= N && a.ldr % 4 == 0 && ((uintptr_t)a.residual & 15) == 0),
               "vi_gemm16: residual must be 16-byte aligned with ldr >= N, ldr %% 4 == 0");
  VI_CHECK_ARG(!a.bias || ((uintptr_t)a.bias & 15) == 0, "vi_gemm16: bias must be 16-byte aligned");
  VI_CHECK_ARG(a.y_dtype == a.in_dtype || a.y_dtype == VI_DT_F32, "vi_gemm16: y_dtype %d must be fp32 or the operand type", a.y_dtype);
  VI_CHECK_ARG(!a.residual || a.y_dtype == VI_DT_F32,
               "vi_gemm16: a residual needs an fp32 output (the residual stream of the model is fp32)");
  VI_CHECK_ARG(!a.y16 || (a.y_dtype == VI_DT_F32 && a.ldy16 >= N && a.ldy16 % 8 == 0 && ((uintptr_t)a.y16 & 15) == 0),
               "vi_gemm16: the 16-bit copy needs an fp32 primary output, ldy16 >= N, ldy16 %% 8 == 0, 16-byte alignment");
  VI_CHECK_ARG(a.epilogue >= VI_EPI_NONE && a.epilogue <= VI_EPI_RELU, "vi_gemm16: bad epilogue %d", a.epilogue);
  VI_CHECK_ARG(n_groups >= 1 && n_groups <= MAX_GROUPS, "vi_gemm16: n_groups=%d out of range", n_groups);
  VI_CHECK_ARG(n_groups == 1 || a.group_row_end, "vi_gemm16: grouped call without group_row_end");
  VI_CHECK_ARG(a.ln_mode >= VI_LN_NONE && a.ln_mode <= VI_LN_RESIDUAL, "vi_gemm16: bad ln_mode %d", a.ln_mode);
  if (a.ln_mode != VI_LN_NONE) {
    VI_CHECK_ARG(a.ln_stats && a.ln_chunks > 0 && a.ln_chunks <= 256 && a.stats_ld >= M,
                 "vi_gemm16: LayerNorm modes need ln_stats, ln_chunks and stats_ld >= M");
    VI_CHECK_ARG(a.ln_mode != VI_LN_FOLD || (a.bias && a.ln_vec_a), "vi_gemm16: VI_LN_FOLD needs bias (= W beta + b) and ln_vec_a (row sums)");
    VI_CHECK_ARG(a.ln_mode != VI_LN_RESIDUAL || (a.residual && a.bias && a.ln_vec_a && a.ln_chunks * 32 == N && a.epilogue == VI_EPI_NONE),
                 "vi_gemm16: VI_LN_RESIDUAL needs residual, bias (= beta + b), gamma, N == 32 * ln_chunks and no activation");
  }
  VI_CHECK_ARG(!a.stats_out || a.stats_ld >= M, "vi_gemm16: stats_out needs stats_ld >= M");
  VI_CHECK_ARG(((uintptr_t)a.ln_stats & 7) == 0 && ((uintptr_t)a.stats_out & 7) == 0, "vi_gemm16: statistics must be 8-byte aligned");
  if (int rc = resolve_encode()) return rc;

  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.bias = a.bias; p.has_residual = a.residual != nullptr; p.y_f32 = (a.y_dtype == VI_DT_F32);
  p.M = M; p.N = N; p.K = K; p.epilogue = a.epilogue; p.n_groups = n_groups;
  p.vec_a = a.ln_mode != VI_LN_NONE ? a.ln_vec_a : nullptr;
  p.stats_in = reinterpret_cast<const float2*>(a.ln_stats);
  p.stats_out = reinterpret_cast<float2*>(a.stats_out);
  p.stats_ld = a.stats_ld; p.stats_chunks = a.ln_chunks; p.ln_mode = a.ln_mode; p.ln_eps = a.ln_eps;
  p.fmt_f16 = a.in_dtype == VI_DT_F16;
  bool pair_ok = true;                   // a 256-row pair tile must not straddle two weight groups
  const int m_tiles128 = (M + BM - 1) / BM;
  for (int g = 0; g < n_groups; ++g) {
    if (n_groups == 1) { p.group_tile_end[g] = m_tiles128; break; }
    const int e = a.group_row_end[g];
    VI_CHECK_ARG(e > 0 && e <= M && (g == 0 || e > a.group_row_end[g - 1]), "vi_gemm16: bad group_row_end[%d]=%d", g, e);
    VI_CHECK_ARG(g == n_groups - 1 || e % BM == 0, "vi_gemm16: group %d must end on a multiple of %d rows (got %d)", g, BM, e);
    if (g < n_groups - 1 && e % (2 * BM) != 0) pair_ok = false;
    p.group_tile_end[g] = (e + BM - 1) / BM;
  }
  VI_CHECK_ARG(n_groups == 1 || a.group_row_end[n_groups - 1] == M, "vi_gemm16: last group must end at M");

  const int nsm = vi_num_sms();
  Choice c;
  if (a.tile != 0) {                     // caller-selected tile (the Python host keeps a measured table per shape)
    const int bn = a.tile & 0xFFF;
    const bool pr = (a.tile & VI_TILE_PAIR) != 0;
    VI_CHECK_ARG((bn == 64 || bn == 96 || bn == 128 || bn == 192 || bn == 256) && N % bn == 0,
                 "vi_gemm16: tile width %d does not divide N=%d", bn, N);
    VI_CHECK_ARG(!pr || (pair_ok && bn >= 128), "vi_gemm16: CTA-pair tiles need width >= 128 and 256-row group ends");
    c = Choice{bn, pr};
  } else {
    c = pick_tile(M, N, K, nsm, pair_ok);
  }
  const int tm = c.pair ? 2 * BM : BM;
  p.num_m_tiles = (M + tm - 1) / tm;
  p.num_n_tiles = N / c.bn;
  const long long tiles = (long long)p.num_m_tiles * p.num_n_tiles;
  int grid;
  if (c.pair) {
    const long long workers = tiles < nsm / 2 ? tiles : nsm / 2;
    grid = (int)(2 * workers);
  } else {
    grid = (int)(tiles < nsm ? tiles : nsm);
  }

  const CUtensorMapDataType dt16 = p.fmt_f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  Maps m;
  memset(&m, 0, sizeof(m));
  if (int rc = make_map(&m.a, a.x, dt16, 2, (uint64_t)K, (uint64_t)M, (uint64_t)a.ldx, BK, BM, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = make_map(&m.b, a.w, dt16, 2, (uint64_t)K, (uint64_t)n_groups * N, (uint64_t)K, BK,
                        (uint32_t)(c.pair ? c.bn / 2 : c.bn), CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (p.y_f32) {
    if (int rc = make_map(&m.y, a.y, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (uint64_t)N, (uint64_t)M, (uint64_t)a.ldy, 32, 32,
                          CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  } else {
    if (int rc = make_map(&m.y, a.y, dt16, 2, (uint64_t)N, (uint64_t)M, (uint64_t)a.ldy, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  }
  if (a.residual) {
    if (int rc = make_map(&m.r, a.residual, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (uint64_t)N, (uint64_t)M, (uint64_t)a.ldr, 32, 32,
                          CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  } else {
    m.r = m.y;
  }
  if (a.y16) {
    if (int rc = make_map(&m.y2, a.y16, dt16, 2, (uint64_t)N, (uint64_t)M, (uint64_t)a.ldy16, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  } else {
    m.y2 = m.y;
  }

  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int om = a.y16 ? OUT_DUAL : (p.y_f32 ? OUT_F32 : OUT_H16);
  // ring depth = what fits beside the epilogue staging (16-bit out: 32 KB, fp32 out: 64 KB, both: 80 KB) in 227 KB
#define VI_LAUNCH(BN_, SH_, SF_, SD_, PAIR_)                                                     \
  (om == OUT_DUAL ? launch<BN_, SD_, PAIR_, OUT_DUAL>(m, p, grid, st)                            \
   : om == OUT_F32 ? launch<BN_, SF_, PAIR_, OUT_F32>(m, p, grid, st)                            \
                   : launch<BN_, SH_, PAIR_, OUT_H16>(m, p, grid, st))
  if (c.pair) {
    switch (c.bn) {
      case 256: return VI_LAUNCH(256, 6, 5, 4, true);
      case 192: return VI_LAUNCH(192, 6, 5, 5, true);
      default:  return VI_LAUNCH(128, 8, 6, 5, true);
    }
  }
  switch (c.bn) {
    case 256: return VI_LAUNCH(256, 4, 3, 2, false);
    case 192: return VI_LAUNCH(192, 4, 4, 3, false);
    case 128: return VI_LAUNCH(128, 6, 5, 4, false);
    case 96:  return VI_LAUNCH(96, 6, 5, 5, false);
    default:  return VI_LAUNCH(64, 8, 6, 6, false);
  }
#undef VI_LAUNCH
}
