// vi_wgrad.cu - weight and bias gradients of a dense layer on the 5th-gen tensor cores, without transposes:
//
//     dW[g] = dY[g]^T X[g]   ([N x K] fp32),      db[g] = column sums of dY[g]   ([N] fp32)          per row group g
//
// dY [rows x N] and X [rows x K] are the row-major 16-bit tensors the backward pass already holds; the contraction runs over
// their ROWS.  Both operands are therefore MN-major for tcgen05.mma: a k-block is 64 rows of dY / X, loaded by TMA as boxes
// of 64 rows x 64 columns (128B swizzle) exactly as they lie in memory - the canonical MN-major layout
// ((8,8,m),(8,k)):((1,8,LBO),(64,SBO)) with SBO = 1024 B between 8-row groups and LBO = 8192 B between 64-column blocks -
// and the instruction descriptor marks A and B as MN-major.  Rows past the end of a group are zero-filled by TMA (every
// group has its own tensor maps), so no padding copies exist either.
//
// The output has few tiles (768 x 768 = 18 tiles of 128 x 256) and a long contraction (2304 - 4608 rows), so the rows are
// split over `splits` work units per tile; with splits > 1 every unit writes its fp32 partial tile to a workspace and a
// second kernel adds the partials in a fixed order (deterministic: no floating-point atomics).  The bias gradient rides
// on the tensor cores as well: the units of the first column tile issue one extra N = 16 MMA per k-step against a tile of
// ones, which leaves the column sums of their dY tile in 16 spare TMEM columns.
//
// Replaces what loss.backward() does for nn.Linear (grad_weight = grad_output^T input, grad_bias = grad_output.sum(0)) in
// VLN-DUET/map_nav_src/models/vilmodel.py:93-95,147,172,186,315-317 and transformer.py:178,181.
#include "vi_common.cuh"

namespace {

constexpr int BM = 128;                 // dW rows per tile (columns of dY)
constexpr int BK = 64;                  // contraction rows per k-block
constexpr int MAXG = 4;
constexpr int NUM_THREADS = 256;        // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warps 4-7 epilogue
constexpr int ONES_BYTES = 2048;
constexpr int STAGE_EPI = 4 * 2 * 4096; // four epilogue warps x two 32 x 32 fp32 staging buffers

struct WgradParams {
  float* db_part;                       // [G][S][N] column sums (or the final db when splits == 1); NULL: no bias gradient
  int N, K;                             // columns of dY / of X
  int n_groups, splits;
  int kb_total[MAXG];                   // k-blocks (64 rows) per group
  int m_tiles, n_tiles;                 // N / 128, K / BN
  int fmt_f16;
  int accumulate;                       // splits == 1 only: add the tile to what `out` / db hold (TMA reduce-add, one writer per element)
};
struct WgradMaps { CUtensorMap dy[MAXG], x[MAXG], out; };

__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t saddr) {
  // MN-major operand, 128-byte swizzle: LBO (bits 16-29) = 8192 B between 64-element MN blocks, SBO (bits 32-45) = 1024 B
  // between 8-row K groups, descriptor version 1 (bit 46), layout type SWIZZLE_128B (bits 61-63 = 2)
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(8192 >> 4) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__host__ __device__ constexpr uint32_t idesc_mn(int n, bool f16) {
  // kind::f16, D = f32, A / B 16-bit formats, A and B MN-major (bits 15, 16), N >> 3 at 17-22, M = 128 >> 4 at 24-28
  return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(BM >> 4) << 24);
}
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(tmap), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const void* tmap, uint32_t src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(tmap), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred px;\n\telect.sync _|px, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, px;\n\t}" : "=r"(pred));
  return pred != 0;
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ WgradMaps maps, const WgradParams p) {
  constexpr int A_BYTES = BK * BM * 2;               // two boxes of 64 rows x 64 columns
  constexpr int B_BYTES = BK * BN * 2;               // BN / 64 boxes
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = BN + 32 <= 128 ? 128u : (BN + 32 <= 256 ? 256u : 512u);
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ones_smem = smem + STAGES * STAGE_BYTES;
  uint8_t* epi_smem = ones_smem + ONES_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem + STAGE_EPI);      // full[S], empty[S], tfull, tempty
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 2);

  const uint32_t smem_base = smem_u32(smem);
  if (smem_base & 1023u) __trap();
  const uint32_t bar_base = smem_u32(bars);
  auto a_addr = [&](int s) { return smem_base + (uint32_t)(s * STAGE_BYTES); };
  auto b_addr = [&](int s) { return smem_base + (uint32_t)(s * STAGE_BYTES + A_BYTES); };
  auto full_bar = [&](int s) { return bar_base + 8u * (uint32_t)s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (uint32_t)(STAGES + s); };
  const uint32_t tfull_bar = bar_base + 8u * (uint32_t)(2 * STAGES), tempty_bar = tfull_bar + 8u;

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int g = 0; g < p.n_groups; ++g) { tma_prefetch_desc(&maps.dy[g]); tma_prefetch_desc(&maps.x[g]); }
    tma_prefetch_desc(&maps.out);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, 4);                         // one arrive per epilogue warp
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_slot), TMEM_COLS); tmem_relinquish(); }
  if (warp == 3) {                                    // the tile of ones behind the bias gradient (any layout reads as ones)
    const uint32_t one2 = p.fmt_f16 ? 0x3C003C00u : 0x3F803F80u;
    for (int i = lane; i < ONES_BYTES / 4; i += 32) reinterpret_cast<uint32_t*>(ones_smem)[i] = one2;
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  const int tiles_per_group = p.m_tiles * p.n_tiles;
  const int total_units = p.n_groups * tiles_per_group * p.splits;
  auto decode = [&](int u, int& g, int& mt, int& nt, int& s, int& kb0, int& kb1) {
    s = u % p.splits; u /= p.splits;
    nt = u % p.n_tiles; u /= p.n_tiles;
    mt = u % p.m_tiles; g = u / p.m_tiles;
    const int kt = p.kb_total[g];
    kb0 = (int)((long long)s * kt / p.splits);
    kb1 = (int)((long long)(s + 1) * kt / p.splits);
  };
  const bool want_db = p.db_part != nullptr;

  if (warp == 0) {
    // ------------------------------- TMA producer ----------------------------------------------------------------
    int st = 0;
    uint32_t ph = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
      int g, mt, nt, s, kb0, kb1;
      decode(u, g, mt, nt, s, kb0, kb1);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar(st), ph ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(full_bar(st), STAGE_BYTES);
#pragma unroll
          for (int j = 0; j < BM / 64; ++j)
            tma_load_2d(a_addr(st) + (uint32_t)(j * 8192), &maps.dy[g], full_bar(st), mt * BM + j * 64, kb * BK);
#pragma unroll
          for (int j = 0; j < BN / 64; ++j)
            tma_load_2d(b_addr(st) + (uint32_t)(j * 8192), &maps.x[g], full_bar(st), nt * BN + j * 64, kb * BK);
        }
        __syncwarp();
        if (++st == STAGES) { st = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -------------------------------------------------------------------
    const uint32_t idesc = idesc_mn(BN, p.fmt_f16 != 0), idesc1 = idesc_mn(16, p.fmt_f16 != 0);
    const uint64_t ones_desc = desc_mn_sw128(smem_u32(ones_smem));
    int st = 0, it = 0;
    uint32_t ph = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++it) {
      int g, mt, nt, s, kb0, kb1;
      decode(u, g, mt, nt, s, kb0, kb1);
      mbar_wait(tempty_bar, ((uint32_t)it & 1u) ^ 1u);                   // the epilogue has drained the accumulator
      tc_fence_after();
      const bool db_unit = want_db && nt == 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(full_bar(st), ph);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t adesc = desc_mn_sw128(a_addr(st)), bdesc = desc_mn_sw128(b_addr(st));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // 16 contraction rows = two 8-row groups = 2048 bytes further into every 64-column block
            const uint32_t acc = (uint32_t)((kb != kb0) || k != 0);
            tc_mma_bf16(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, acc);
            if (db_unit) tc_mma_bf16(tmem_base + (uint32_t)BN, adesc + (uint64_t)(128 * k), ones_desc, idesc1, acc);
          }
          tc_commit(empty_bar(st));
          if (kb == kb1 - 1) tc_commit(tfull_bar);
        }
        __syncwarp();
        if (++st == STAGES) { st = 0; ph ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------- epilogue: TMEM -> swizzled shared memory -> TMA store --------------------------
    const int ew = warp - 4;                          // == warp & 3: the TMEM lane quarter this warp may read
    const uint32_t my_buf = smem_u32(epi_smem) + (uint32_t)(ew * 8192);
    int it = 0, n = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++it) {
      int g, mt, nt, s, kb0, kb1;
      decode(u, g, mt, nt, s, kb0, kb1);
      const int orow0 = (g * p.splits + s) * p.N + mt * BM + ew * 32;    // first output row of this warp
      mbar_wait(tfull_bar, (uint32_t)it & 1u);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(ew * 32) << 16);
      uint32_t r[32];
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c, ++n) {
        tmem_ld_32x32(tbase + (uint32_t)(c * 32), r);
        const uint32_t buf = my_buf + (uint32_t)((n & 1) * 4096);
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the store two chunks ago has read this buffer
        __syncwarp();
        tmem_ld_wait();
        const uint32_t rowb = buf + (uint32_t)(lane * 128);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};"
                       ::"r"(rowb + (uint32_t)((j ^ (lane & 7)) << 4)), "r"(r[4 * j]), "r"(r[4 * j + 1]), "r"(r[4 * j + 2]), "r"(r[4 * j + 3])
                       : "memory");
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (p.accumulate) tma_reduce_add_2d(&maps.out, buf, nt * BN + c * 32, orow0);
          else tma_store_2d(&maps.out, buf, nt * BN + c * 32, orow0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
      if (want_db && nt == 0) {
        tmem_ld_32x32(tbase + (uint32_t)BN, r);       // 16 identical columns of sums (+ 16 unused ones)
        tmem_ld_wait();
        float* dst = p.db_part + (long long)(g * p.splits + s) * p.N + mt * BM + ew * 32 + lane;
        *dst = p.accumulate ? *dst + __uint_as_float(r[0]) : __uint_as_float(r[0]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar);
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------------------------------
// CTA-pair form (cta_group::2), the default when N % 256 == 0: two CTAs of a cluster work on one 256 x BN tile of dW.  Each CTA
// loads ITS 128 columns of dY (its half of the M = 256 operand) and HALF of the X columns (its half of the N operand), the leader
// issues M = 256 MMAs that read both CTAs' shared memory, every CTA drains its own 128 TMEM lanes.  A 128 x 256 single-CTA tile
// pulls 48 KB per k-block = 94 B/clk/SM from L2 (bound: cuBLAS was 15 - 75 % faster on these shapes); the pair pulls 32 KB per
// CTA for the same 512 cycles of MMA.  Barrier protocol as in the forward kernel's PAIR mode (vi_gemm_tc.cu): both CTAs' TMA
// bytes land on the LEADER's full barrier, tcgen05.commit is multicast to both CTAs' empty / accumulator-full barriers, the
// epilogue warps of both CTAs arrive on the leader's accumulator-empty barrier.
// ---------------------------------------------------------------------------------------------------------------------------
constexpr uint32_t PEER_MASK_W = 0xFEFFFFFFu;          // clears the CTA-rank bit of a shared::cluster address (pair leader)
__device__ __forceinline__ uint32_t cluster_ctarank_w() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_w() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_w(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar & PEER_MASK_W), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader_w(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_MASK_W) : "memory");
}
__device__ __forceinline__ void tc_commit_pair_w(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma_pair_w(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__host__ __device__ constexpr uint32_t idesc_mn_m256(int n, bool f16) {
  return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(256 >> 4) << 24);
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_pair_kernel(const __grid_constant__ WgradMaps maps, const WgradParams p) {
  constexpr int A_BYTES = BK * BM * 2;               // this CTA's 128 columns of dY: two boxes of 64 rows x 64 columns
  constexpr int BN_CTA = BN / 2;                     // this CTA's half of the X columns
  constexpr int B_BYTES = BK * BN_CTA * 2;
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = BN + 32 <= 128 ? 128u : (BN + 32 <= 256 ? 256u : 512u);
  static_assert(BN_CTA % 64 == 0, "a CTA stages whole 64-column blocks of X");
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ones_smem = smem + STAGES * STAGE_BYTES;
  uint8_t* epi_smem = ones_smem + ONES_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem + STAGE_EPI);      // full[S], empty[S], tfull, tempty
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 2);

  const uint32_t smem_base = smem_u32(smem);
  if (smem_base & 1023u) __trap();
  const uint32_t bar_base = smem_u32(bars);
  auto a_addr = [&](int s) { return smem_base + (uint32_t)(s * STAGE_BYTES); };
  auto b_addr = [&](int s) { return smem_base + (uint32_t)(s * STAGE_BYTES + A_BYTES); };
  auto full_bar = [&](int s) { return bar_base + 8u * (uint32_t)s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (uint32_t)(STAGES + s); };
  const uint32_t tfull_bar = bar_base + 8u * (uint32_t)(2 * STAGES), tempty_bar = tfull_bar + 8u;

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank_w();
  const int worker = (int)(blockIdx.x >> 1), n_workers = (int)(gridDim.x >> 1);
  if (warp == 0 && lane == 0) {
    for (int g = 0; g < p.n_groups; ++g) { tma_prefetch_desc(&maps.dy[g]); tma_prefetch_desc(&maps.x[g]); }
    tma_prefetch_desc(&maps.out);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, 8);                         // one arrive per epilogue warp of BOTH CTAs (on the leader's barrier)
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (warp == 3) {
    const uint32_t one2 = p.fmt_f16 ? 0x3C003C00u : 0x3F803F80u;
    for (int i = lane; i < ONES_BYTES / 4; i += 32) reinterpret_cast<uint32_t*>(ones_smem)[i] = one2;
    fence_proxy_async();
  }
  tc_fence_before();
  cluster_sync_w();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  const int tiles_per_group = p.m_tiles * p.n_tiles;                       // m tiles of 256 rows here
  const int total_units = p.n_groups * tiles_per_group * p.splits;
  auto decode = [&](int u, int& g, int& mt, int& nt, int& s, int& kb0, int& kb1) {
    s = u % p.splits; u /= p.splits;
    nt = u % p.n_tiles; u /= p.n_tiles;
    mt = u % p.m_tiles; g = u / p.m_tiles;
    const int kt = p.kb_total[g];
    kb0 = (int)((long long)s * kt / p.splits);
    kb1 = (int)((long long)(s + 1) * kt / p.splits);
  };
  const bool want_db = p.db_part != nullptr;

  if (warp == 0) {
    // ------------------------------- TMA producer (both CTAs; bytes are counted on the leader's barrier) -----------
    int st = 0;
    uint32_t ph = 0;
    for (int u = worker; u < total_units; u += n_workers) {
      int g, mt, nt, s, kb0, kb1;
      decode(u, g, mt, nt, s, kb0, kb1);
      const int acol = mt * 256 + (int)rank * BM;                          // this CTA's 128 columns of dY
      const int bcol = nt * BN + (int)rank * BN_CTA;                       // this CTA's half of the X columns
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar(st), ph ^ 1u);
        if (elect_one()) {
          if (rank == 0) mbar_expect_tx(full_bar(st), 2 * STAGE_BYTES);
#pragma unroll
          for (int j = 0; j < BM / 64; ++j)
            tma_load_2d_pair_w(a_addr(st) + (uint32_t)(j * 8192), &maps.dy[g], full_bar(st), acol + j * 64, kb * BK);
#pragma unroll
          for (int j = 0; j < BN_CTA / 64; ++j)
            tma_load_2d_pair_w(b_addr(st) + (uint32_t)(j * 8192), &maps.x[g], full_bar(st), bcol + j * 64, kb * BK);
        }
        __syncwarp();
        if (++st == STAGES) { st = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer (leader only) -----------------------------------------------------
    if (rank == 0) {
      const uint32_t idesc = idesc_mn_m256(BN, p.fmt_f16 != 0), idesc1 = idesc_mn_m256(16, p.fmt_f16 != 0);
      const uint64_t ones_desc = desc_mn_sw128(smem_u32(ones_smem));
      int st = 0, it = 0;
      uint32_t ph = 0;
      for (int u = worker; u < total_units; u += n_workers, ++it) {
        int g, mt, nt, s, kb0, kb1;
        decode(u, g, mt, nt, s, kb0, kb1);
        mbar_wait(tempty_bar, ((uint32_t)it & 1u) ^ 1u);                 // both CTAs' epilogues have drained the accumulator
        tc_fence_after();
        const bool db_unit = want_db && nt == 0;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(st), ph);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = desc_mn_sw128(a_addr(st)), bdesc = desc_mn_sw128(b_addr(st));
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint32_t acc = (uint32_t)((kb != kb0) || k != 0);
              tc_mma_pair_w(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, acc);
              if (db_unit) tc_mma_pair_w(tmem_base + (uint32_t)BN, adesc + (uint64_t)(128 * k), ones_desc, idesc1, acc);
            }
            tc_commit_pair_w(empty_bar(st));
            if (kb == kb1 - 1) tc_commit_pair_w(tfull_bar);
          }
          __syncwarp();
          if (++st == STAGES) { st = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------- epilogue (both CTAs, each its own 128 rows of the tile) ------------------------
    const int ew = warp - 4;
    const uint32_t my_buf = smem_u32(epi_smem) + (uint32_t)(ew * 8192);
    int it = 0, n = 0;
    for (int u = worker; u < total_units; u += n_workers, ++it) {
      int g, mt, nt, s, kb0, kb1;
      decode(u, g, mt, nt, s, kb0, kb1);
      const int mrow0 = mt * 256 + (int)rank * BM + ew * 32;             // row of dW inside the group
      const int orow0 = (g * p.splits + s) * p.N + mrow0;
      mbar_wait(tfull_bar, (uint32_t)it & 1u);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(ew * 32) << 16);
      uint32_t r[32];
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c, ++n) {
        tmem_ld_32x32(tbase + (uint32_t)(c * 32), r);
        const uint32_t buf = my_buf + (uint32_t)((n & 1) * 4096);
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        tmem_ld_wait();
        const uint32_t rowb = buf + (uint32_t)(lane * 128);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};"
                       ::"r"(rowb + (uint32_t)((j ^ (lane & 7)) << 4)), "r"(r[4 * j]), "r"(r[4 * j + 1]), "r"(r[4 * j + 2]), "r"(r[4 * j + 3])
                       : "memory");
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (p.accumulate) tma_reduce_add_2d(&maps.out, buf, nt * BN + c * 32, orow0);
          else tma_store_2d(&maps.out, buf, nt * BN + c * 32, orow0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
      if (want_db && nt == 0) {
        tmem_ld_32x32(tbase + (uint32_t)BN, r);
        tmem_ld_wait();
        float* dst = p.db_part + (long long)(g * p.splits + s) * p.N + mrow0 + lane;
        *dst = p.accumulate ? *dst + __uint_as_float(r[0]) : __uint_as_float(r[0]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader_w(tempty_bar);
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  cluster_sync_w();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// out[g][i] = sum over s (fixed order) of part[g][s][i]   for two segments (weight and bias gradients)
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* part_w, float* out_w, long long per_group_w4,
                                                           const float* part_b, float* out_b, long long per_group_b4, int G, int S,
                                                           int accumulate) {
  pdl_enter();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nw = (long long)G * per_group_w4, nb = (long long)G * per_group_b4;
  const float* part; float* out; long long per, j;
  if (i < nw) { part = part_w; out = out_w; per = per_group_w4; j = i; }
  else if (i < nw + nb) { part = part_b; out = out_b; per = per_group_b4; j = i - nw; }
  else return;
  const long long g = j / per, e = j - g * per;
  const float4* src = reinterpret_cast<const float4*>(part) + (g * S) * per + e;
  float4 acc = *src;
  for (int s = 1; s < S; ++s) {
    const float4 v = *(src + (long long)s * per);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  if (accumulate) {
    const float4 o = reinterpret_cast<const float4*>(out)[j];
    acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
  }
  reinterpret_cast<float4*>(out)[j] = acc;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_f32_out_map(CUtensorMap* map, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld) {
  static EncodeTiledFn enc = nullptr;
  if (!enc) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      vi_set_error("cuTensorMapEncodeTiled is not available from the driver");
      return VI_ERR_CUDA;
    }
    enc = reinterpret_cast<EncodeTiledFn>(fn);
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vi_set_error("vi_wgrad16: cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return VI_ERR_CUDA;
  }
  return VI_OK;
}

template <int BN, int STAGES> constexpr int wgrad_smem() {
  return STAGES * (BK * BM * 2 + BK * BN * 2) + ONES_BYTES + STAGE_EPI + (2 * STAGES + 2) * 8 + 16;
}
template <int BN, int STAGES>
int launch_wgrad(const WgradMaps& m, const WgradParams& p, int grid, cudaStream_t st) {
  static_assert(wgrad_smem<BN, STAGES>() <= 232448, "shared memory budget");
  static bool attr_set = false;
  auto kern = wgrad_tc_kernel<BN, STAGES>;
  if (!attr_set) {
    VI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, wgrad_smem<BN, STAGES>()));
    attr_set = true;
  }
  VI_CUDA(vi_launch(kern, dim3((unsigned)grid), dim3(NUM_THREADS), (size_t)wgrad_smem<BN, STAGES>(), st, m, p));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

template <int BN, int STAGES> constexpr int wgrad_pair_smem() {
  return STAGES * (BK * BM * 2 + BK * (BN / 2) * 2) + ONES_BYTES + STAGE_EPI + (2 * STAGES + 2) * 8 + 16;
}
template <int BN, int STAGES>
int launch_wgrad_pair(const WgradMaps& m, const WgradParams& p, int pairs, cudaStream_t st) {
  static_assert(wgrad_pair_smem<BN, STAGES>() <= 232448, "shared memory budget");
  static bool attr_set = false;
  auto kern = wgrad_pair_kernel<BN, STAGES>;
  if (!attr_set) {
    VI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, wgrad_pair_smem<BN, STAGES>()));
    attr_set = true;
  }
  VI_CUDA(vi_launch_cluster(kern, 2, dim3((unsigned)(2 * pairs)), dim3(NUM_THREADS), (size_t)wgrad_pair_smem<BN, STAGES>(), st, m, p));
  VI_LAUNCH_CHECK();
  return VI_OK;
}

// the CTA-pair form serves shapes whose N is a multiple of 256 and whose K is a multiple of 128
bool wgrad_pair_ok(int N, int K) { return N % 256 == 0 && K % 128 == 0; }

}  // namespace

extern "C" int64_t vi_wgrad16_workspace(int N, int K, int n_groups, const int32_t* group_rows, int splits) {
  // floats the caller must provide for the split partials (0 when one unit per tile suffices); splits <= 0: the library's choice
  if (n_groups < 1 || n_groups > MAXG || !group_rows || N <= 0 || K <= 0) return -1;
  int s = splits > 0 ? splits : vi_wgrad16_splits(N, K, n_groups, group_rows);
  if (s <= 1) return 0;
  return (int64_t)n_groups * s * ((int64_t)N * K + N);
}

extern "C" int vi_wgrad16_splits(int N, int K, int n_groups, const int32_t* group_rows) {
  if (n_groups < 1 || n_groups > MAXG || !group_rows || N <= 0 || K <= 0) return 1;
  const int bn = K % 256 == 0 ? 256 : (K % 128 == 0 ? 128 : 64);
  const bool pair = wgrad_pair_ok(N, K);
  // work units: 128-row tiles on one SM each, or 256-row tiles on a pair of SMs
  const long long tiles = pair ? (long long)n_groups * (N / 256) * (K / bn) * 2 : (long long)n_groups * (N / BM) * (K / bn);
  int min_kb = 1 << 30;
  for (int g = 0; g < n_groups; ++g) {
    const int kb = (group_rows[g] + BK - 1) / BK;
    min_kb = kb < min_kb ? kb : min_kb;
  }
  const int nsm = vi_num_sms();
  int s = (int)((nsm + tiles / 2) / (tiles > 0 ? tiles : 1));           // units ~ one wave of the SMs
  if (s > min_kb / 2) s = min_kb / 2;                                     // at least two k-blocks per unit
  if (s > 16) s = 16;
  return s < 1 ? 1 : s;
}

extern "C" int vi_wgrad16(const void* dy, int64_t lddy, const void* x, int64_t ldx, int dtype, int N, int K, int n_groups,
                          const int32_t* group_row_end, float* dw, float* db, float* workspace, int64_t workspace_floats,
                          int splits, int accumulate, vi_stream_t stream) {
  VI_CHECK_ARG(dy && x && dw, "vi_wgrad16: null operand");
  VI_CHECK_ARG(dtype == VI_DT_BF16 || dtype == VI_DT_F16, "vi_wgrad16: operands must be bf16 or fp16");
  VI_CHECK_ARG(N > 0 && N % BM == 0, "vi_wgrad16: N=%d (columns of dY) must be a multiple of %d", N, BM);
  VI_CHECK_ARG(K > 0 && K % 64 == 0, "vi_wgrad16: K=%d (columns of X) must be a multiple of 64", K);
  VI_CHECK_ARG(lddy >= N && lddy % 8 == 0 && ldx >= K && ldx % 8 == 0, "vi_wgrad16: leading dimensions must cover the rows and be multiples of 8");
  VI_CHECK_ARG((((uintptr_t)dy | (uintptr_t)x | (uintptr_t)dw) & 15) == 0 && ((uintptr_t)db & 3) == 0, "vi_wgrad16: operands must be 16-byte aligned");
  VI_CHECK_ARG(n_groups >= 1 && n_groups <= MAXG && group_row_end, "vi_wgrad16: 1..%d groups with group_row_end", MAXG);
  int32_t rows[MAXG];
  for (int g = 0; g < n_groups; ++g) {
    rows[g] = group_row_end[g] - (g ? group_row_end[g - 1] : 0);
    VI_CHECK_ARG(rows[g] > 0, "vi_wgrad16: group %d is empty", g);
  }
  const int S = splits > 0 ? splits : vi_wgrad16_splits(N, K, n_groups, rows);
  const int bn = K % 256 == 0 ? 256 : (K % 128 == 0 ? 128 : 64);
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.N = N; p.K = K; p.n_groups = n_groups; p.splits = S; p.m_tiles = N / BM; p.n_tiles = K / bn; p.fmt_f16 = dtype == VI_DT_F16;
  p.accumulate = (accumulate != 0 && S == 1) ? 1 : 0;
  for (int g = 0; g < n_groups; ++g) {
    p.kb_total[g] = (rows[g] + BK - 1) / BK;
    VI_CHECK_ARG(S <= p.kb_total[g], "vi_wgrad16: %d splits exceed the %d k-blocks of group %d", S, p.kb_total[g], g);
  }
  const int64_t need = S > 1 ? (int64_t)n_groups * S * ((int64_t)N * K + N) : 0;
  VI_CHECK_ARG(S == 1 || (workspace && workspace_floats >= need && ((uintptr_t)workspace & 15) == 0),
               "vi_wgrad16: %d splits need a 16-byte aligned workspace of %lld floats", S, (long long)need);
  float* part_w = S > 1 ? workspace : dw;
  float* part_b = S > 1 ? workspace + (int64_t)n_groups * S * N * K : db;
  p.db_part = db ? part_b : nullptr;

  WgradMaps m;
  memset(&m, 0, sizeof(m));
  for (int g = 0; g < n_groups; ++g) {
    const int64_t r0 = g ? group_row_end[g - 1] : 0;
    const uint8_t* dyg = reinterpret_cast<const uint8_t*>(dy) + r0 * lddy * 2;
    const uint8_t* xg = reinterpret_cast<const uint8_t*>(x) + r0 * ldx * 2;
    if (int rc = vi_make_tmap_h16(&m.dy[g], dyg, p.fmt_f16, (uint64_t)N, (uint64_t)rows[g], (uint64_t)lddy, BK)) return rc;
    if (int rc = vi_make_tmap_h16(&m.x[g], xg, p.fmt_f16, (uint64_t)K, (uint64_t)rows[g], (uint64_t)ldx, BK)) return rc;
  }
  if (int rc = make_f32_out_map(&m.out, part_w, (uint64_t)K, (uint64_t)n_groups * S * N, (uint64_t)K)) return rc;

  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int nsm = vi_num_sms();
  int rc;
  if (wgrad_pair_ok(N, K)) {
    p.m_tiles = N / 256;
    const long long units = (long long)n_groups * p.m_tiles * p.n_tiles * S;
    const int pairs = (int)(units < nsm / 2 ? units : nsm / 2);
    rc = bn == 256 ? launch_wgrad_pair<256, 6>(m, p, pairs, st) : launch_wgrad_pair<128, 8>(m, p, pairs, st);
  } else {
    const long long units = (long long)n_groups * p.m_tiles * p.n_tiles * S;
    const int grid = (int)(units < nsm ? units : nsm);
    if (bn == 256) rc = launch_wgrad<256, 4>(m, p, grid, st);
    else if (bn == 128) rc = launch_wgrad<128, 6>(m, p, grid, st);
    else rc = launch_wgrad<64, 8>(m, p, grid, st);
  }
  if (rc) return rc;
  if (S > 1) {
    const long long w4 = (long long)N * K / 4, b4 = db ? N / 4 : 0;
    const long long total = (long long)n_groups * (w4 + b4);
    VI_CUDA(vi_launch(wgrad_reduce_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), (size_t)0, st, (const float*)part_w, dw, w4,
                      (const float*)part_b, db, b4, n_groups, S, (int)(accumulate != 0)));
    VI_LAUNCH_CHECK();
  }
  return VI_OK;
}
