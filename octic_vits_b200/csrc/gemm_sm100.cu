// Grouped bf16 GEMM for sm_100a: TMA -> shared memory -> tcgen05.mma (fp32 accumulators in TMEM)
// -> fused epilogue.  One persistent CTA per SM, warp-specialised:
//   warp 0     TMA producer (one lane)
//   warp 1     MMA issuer (one lane) + TMEM allocation (whole warp)
//   warps 2-17 epilogue: tcgen05.ld -> registers -> per-warp smem transpose -> coalesced global I/O
// gemm_tn_kernel<MODE, 2> runs as CTA pairs (cluster of 2, tcgen05 cta_group::2, M = 256): each CTA loads its own
// 128 A rows and HALF of the B tile, so the operand traffic out of L2 per flop drops by a third -- at 128 x 256
// single-CTA tiles the kernel is bound by L2 -> SM bandwidth, not by the tensor pipe.
//
// Two kernels live here:
//   gemm_tn_kernel     C[m, n] = sum_k A[m, k] * B[n, k]   (both operands K-major).  A "problem" is a list of
//                      up to 8 groups that share the token (M) dimension but have their own K-range inside
//                      the packed activation row, their own weight rows, and their own output columns.  This
//                      is exactly the irrep-block-diagonal LinearD8 of the reference
//                      (octic_vits/d8_layers.py:104-127): 4 groups for A1/A2/B1/B2 and 2 groups (the two rows
//                      of the 2-D irrep E) that share W_E.  groups = 1 is the dense nn.Linear of the
//                      non-octic half (deit/vit.py:29-33).  dgrad reuses it with transposed weights.
//   gemm_wgrad_kernel  dW[n_out, k_in] += sum_t dY[t, n_out] * X[t, k_in]   (both operands MN-major, the
//                      contraction runs over tokens), split over token ranges, reduced with red.add.f32.
#include "octic_capi_internal.h"
#include "sm100_ptx.cuh"
#include "gelu_math.cuh"
#include <stdlib.h>

namespace octic {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;           // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int kUmmaK = 16;
constexpr int kEpiWarps = 16;              // TN kernel: four epilogue warps per TMEM lane quarter
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;
constexpr int kWgradThreads = 192;
constexpr int kMaxStages = 8;
constexpr int kAStageBytes = kBlockM * kBlockK * 2;   // 16 KiB
constexpr int kStagingWords = 32 * 36;                // per epilogue warp: 32 rows x (32+1) words, or x 36 (16-byte rows)
constexpr int kTmemCols = 512;
constexpr int kAccStride = 256;                       // columns between the two accumulator stages

struct SmemLayout {
  uint32_t a_off, b_off, stg_off, bar_off, total;
};
// b_slots: B k-block buffers -- one per ring stage, or (weight-stationary mode) the k-blocks of one whole-K weight tile
__host__ __device__ inline SmemLayout smem_layout(int stages, int b_stage_bytes, int epi_warps, int b_slots = -1) {
  SmemLayout L;
  L.a_off = 0;
  L.b_off = stages * kAStageBytes;
  L.stg_off = L.b_off + (b_slots < 0 ? stages : b_slots) * b_stage_bytes;
  L.bar_off = L.stg_off + epi_warps * kStagingWords * 4;
  L.total = L.bar_off + (2 * kMaxStages + 4) * 8 + 16 + 2 * 8;     // ring + accumulator barriers, TMEM pointer, wfull / wempty
  return L;
}

// erf via Abramowitz-Stegun 7.1.26 (|abs err| <= 1.5e-7): one MUFU.RCP + one MUFU.EX2 + 6 FMA instead of erff's ~30
__device__ __forceinline__ float erf_fast(float x) {
  const float z = fabsf(x);
  const float t = __frcp_rn(fmaf(0.3275911f, z, 1.0f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float e = 1.0f - poly * t * __expf(-z * z);
  return copysignf(e, x);
}
__device__ __forceinline__ float gelu_fast(float x) { return 0.5f * x * (1.0f + erf_fast(x * 0.70710678118654752f)); }
// d/dx gelu(x) = Phi(x) + x phi(x) with the same erf approximation: one MUFU.EX2 + one MUFU.RCP (reference
// octic_vits/d8_gelu.py:16-26 states the derivative; the dense fc1 activation is nn.GELU, deit/vit.py:126-129)
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  const float e = __expf(-0.5f * x * x);
  const float t = __frcp_rn(fmaf(0.3275911f, z, 1.0f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erfv = copysignf(1.0f - poly * t * e, x);
  return fmaf(x, 0.3989422804014327f * e, 0.5f * (1.0f + erfv));
}
// two elements per instruction (FFMA2): the GELU epilogues are instruction-issue bound (ncu: 58-62 % issue slots)
__device__ __forceinline__ void gelu_pair(float a, float b, float& ga, float& gb) {
  un2(mul2(gelu_x2_2(mk2(a, b)), sp2(0.5f)), ga, gb);
}
__device__ __forceinline__ void gelu_grad_pair(float a, float b, float& ga, float& gb) {
  un2(gelu_grad_2(mk2(a, b)), ga, gb);
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 b = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&b);
}

// ------------------------------------------------------------------------------------------------------------
//  TN kernel
// ------------------------------------------------------------------------------------------------------------
template <int MODE, int NCTA>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB0,
               const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment; the dynamic smem base is only guaranteed 16.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // Warp roles: producer 0 / MMA 1 / epilogue 2-17 (p.roles_low, the default) or producer 16 / MMA 17 / epilogue 0-15
  // (experiment switch, see roles_low_env).
  const int prod_warp = p.roles_low ? 0 : kEpiWarps, mma_warp = p.roles_low ? 1 : kEpiWarps + 1;
  const int stages = p.num_stages;
  const int b_rows = p.block_n / NCTA;                    // B rows held by this CTA
  const int b_stage_bytes = b_rows * kBlockK * 2;
  // Weight-stationary mode (p.ws, CTA pairs only; the small-K irrep groups of LinearD8, K <= 320): a CTA pair walks a
  // CONTIGUOUS range of the tile list in (group, n block)-major order, so consecutive tiles share their weight tile.
  // The whole-K weight tile is loaded once into its own buffer and only the A k-blocks stream through the ring: the
  // L2 -> shared-memory traffic per tile drops from A + B (144 KB for a 128 x 256 x 192 tile) to A (48 KB).  In tile
  // order the kernel was bound by exactly that traffic (1.06 GB per fc1 launch at ~10 TB/s of L2 bandwidth = 105 of its
  // 144 us; the epilogue alone drains the same output in 65 us, profiles/r02_epilogue_probe.txt).
  const bool ws = NCTA == 2 && p.ws != 0;
  const SmemLayout L = smem_layout(stages, b_stage_bytes, kEpiWarps, ws ? p.ws_kb_max : -1);
  const int rank = NCTA == 2 ? static_cast<int>(cluster_ctarank()) : 0;
  const int cid = blockIdx.x / NCTA, ncl = gridDim.x / NCTA;   // this CTA (pair) and the number of them

  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tfull_bar = empty_bar + kMaxStages;   // [2]
  uint64_t* tempty_bar = tfull_bar + 2;           // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  uint64_t* wfull_bar = reinterpret_cast<uint64_t*>(tmem_ptr + 4);   // weight tile landed (leader's barrier)
  uint64_t* wempty_bar = wfull_bar + 1;                              // every MMA that reads the weight tile has completed

  if (warp == prod_warp && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB0);
    tma_prefetch_desc(&tmB1);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], kEpiWarps * NCTA);   // one arrive per epilogue warp of the pair (leader's barrier)
    }
    mbar_init(wfull_bar, 1);
    mbar_init(wempty_bar, 1);
    fence_mbar_init();
  }
  if (warp == mma_warp) {
    if (NCTA == 2) tmem_alloc_pair(tmem_ptr, kTmemCols);
    else tmem_alloc(tmem_ptr, kTmemCols);
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int total_tiles = p.num_m_blocks * p.tiles_per_m;     // num_m_blocks counts 128 * NCTA-row blocks
  // tile sequence of this CTA (pair): tile_first, tile_first + tile_step, ... < tile_last
  //   tile order      : tile = m_pair * tiles_per_m + j, CTAs take every ncl-th tile
  //   weight stationary: tile = j * num_m_blocks + m_pair, CTAs take contiguous ranges (same j => same weight tile)
  const int tile_first = ws ? static_cast<int>(static_cast<long>(total_tiles) * cid / ncl) : cid;
  const int tile_last = ws ? static_cast<int>(static_cast<long>(total_tiles) * (cid + 1) / ncl) : total_tiles;
  const int tile_step = ws ? 1 : ncl;

  auto decode = [&](int tile, int& m_blk, int& g, int& n_blk) {
    const int mp = ws ? tile % p.num_m_blocks : tile / p.tiles_per_m;
    m_blk = mp * NCTA + rank;                                  // this CTA's own 128-row block
    int j = ws ? tile / p.num_m_blocks : tile - mp * p.tiles_per_m;
    g = 0;
#pragma unroll 1
    for (int i = 1; i < p.num_groups; ++i)
      if (j >= p.g[i].tile_begin) g = i;
    n_blk = j - p.g[g].tile_begin;
  };

  if (warp == prod_warp) {
    // ------------------------------------------ TMA producer ------------------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int cur_j = -1;
      uint32_t wphase = 0;
      for (int tile = tile_first; tile < tile_last; tile += tile_step) {
        int m_blk, g, n_blk;
        decode(tile, m_blk, g, n_blk);
        const GemmGroup& G = p.g[g];
        const CUtensorMap* tmB = G.b_map ? &tmB1 : &tmB0;
        if (NCTA == 2 && ws) {
          const int j = tile / p.num_m_blocks;
          if (j != cur_j) {
            // new (group, n block): replace the stationary weight tile once every MMA that reads the old one is done
            if (cur_j >= 0) { mbar_wait(wempty_bar, wphase); wphase ^= 1; }
            cur_j = j;
            if (rank == 0) mbar_arrive_expect_tx(wfull_bar, 2 * G.k_blocks * b_stage_bytes);
            for (int kb = 0; kb < G.k_blocks; ++kb)
              tma_load_2d_pair(smem + L.b_off + kb * b_stage_bytes, tmB, wfull_bar, kb * kBlockK,
                               G.b_row + n_blk * p.block_n + rank * b_rows);
          }
        }
        for (int kb = 0; kb < G.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = smem + L.a_off + stage * kAStageBytes;
          uint8_t* b_dst = smem + L.b_off + stage * b_stage_bytes;
          if (NCTA == 2 && ws) {
            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kAStageBytes);
            tma_load_2d_pair(a_dst, &tmA, &full_bar[stage], G.a_col + kb * kBlockK, m_blk * kBlockM);
          } else if (NCTA == 2) {
            // both CTAs' loads complete on the leader's barrier, which expects the bytes of the pair
            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * (kAStageBytes + b_stage_bytes));
            tma_load_2d_pair(a_dst, &tmA, &full_bar[stage], G.a_col + kb * kBlockK, m_blk * kBlockM);
            tma_load_2d_pair(b_dst, tmB, &full_bar[stage], kb * kBlockK, G.b_row + n_blk * p.block_n + rank * b_rows);
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], kAStageBytes + b_stage_bytes);
            tma_load_2d(a_dst, &tmA, &full_bar[stage], G.a_col + kb * kBlockK, m_blk * kBlockM);
            tma_load_2d(b_dst, tmB, &full_bar[stage], kb * kBlockK, G.b_row + n_blk * p.block_n);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == mma_warp) {
    // -------------------------------------------- MMA issuer --------------------------------------------
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc_bf16(kBlockM * NCTA, p.block_n, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      int cur_j = -1;
      uint32_t wphase = 0;
      for (int tile = tile_first; tile < tile_last; tile += tile_step, ++it) {
        int m_blk, g, n_blk;
        decode(tile, m_blk, g, n_blk);
        const int k_blocks = p.g[g].k_blocks;
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        const int j = ws ? tile / p.num_m_blocks : 0;
        if (ws && j != cur_j) {
          mbar_wait(wfull_bar, wphase);      // the stationary weight tile of this (group, n block) has landed
          wphase ^= 1;
          cur_j = j;
        }
        mbar_wait(&tempty_bar[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * kAccStride;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          // K-major, SWIZZLE_128B: rows are 128 B, 8-row groups are 1024 B apart (SBO); LBO unused.
          const uint64_t da = make_smem_desc(smem_u32(smem + L.a_off + stage * kAStageBytes), 0, 1024);
          const uint64_t db = make_smem_desc(smem_u32(smem + L.b_off + (ws ? kb : stage) * b_stage_bytes), 0, 1024);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            // advancing 16 bf16 (32 B) inside the swizzle atom = +2 in the (addr >> 4) field
            if (NCTA == 2) umma_bf16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            else umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          if (NCTA == 2) {
            umma_commit_pair(&empty_bar[stage]);
            if (kb == k_blocks - 1) umma_commit_pair(&tfull_bar[as]);
          } else {
            umma_commit(&empty_bar[stage]);
            if (kb == k_blocks - 1) umma_commit(&tfull_bar[as]);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        if (NCTA == 2 && ws) {
          // last tile of this weight tile: tell both producers when its MMAs have completed
          const int nxt = tile + tile_step;
          if (nxt < tile_last && nxt / p.num_m_blocks != j) umma_commit_pair(wempty_bar);
        }
      }
    }
  } else {
    // --------------------------------------------- epilogue ---------------------------------------------
    // 16 warps: warp w may touch TMEM lanes 32*(w%4)..+31; the four warps of a lane quarter take every fourth
    // 32-column chunk (the epilogue is latency bound per warp: more warps, not more work per warp, keep it ahead of
    // the tensor pipe).
    // A chunk goes TMEM -> registers (thread = row) -> per-warp smem transpose -> coalesced global I/O (lane = column).
    const int ew = p.roles_low ? warp - 2 : warp;
    const int q = warp & 3;
    const int half = ew >> 2;                  // 0..3: first chunk of this warp
    constexpr int kChunkStep = 32 * (kEpiWarps / 4);
    const uint32_t stg = smem_u32(smem + L.stg_off) + ew * kStagingWords * 4;
    // EPI_RESID: the fp32 residual rows of the warp's NEXT 32 x 32 chunk are fetched while the current chunk is
    // processed (and, across tiles, while the MMAs of the next tile run): the epilogue is otherwise paced by one
    // DRAM round trip per 8 rows.  res_ok is warp-uniform.
    //
    // Direct path (every full 32-column chunk of an aligned, un-remapped output): the thread keeps its row -- 32
    // consecutive columns -- in registers and reads / writes global memory with 16-byte accesses straight from there.
    // No shared-memory transpose: the operand reads of tcgen05.mma plus the TMA fills already use most of the
    // 128 B/clk of shared-memory bandwidth, which is what bounds this kernel.  The staged path below remains for
    // head-remapped outputs, column tails and unaligned shapes.
    const bool direct_ptrs =
        p.direct != 0 && p.head_H == 0 && p.remap_group == 0 &&
        (MODE == EPI_RESID
             ? ((reinterpret_cast<uintptr_t>(p.resid_out) | reinterpret_cast<uintptr_t>(p.resid_in) |
                 reinterpret_cast<uintptr_t>(p.gamma) | reinterpret_cast<uintptr_t>(p.branch_out)) & 15) == 0 &&
                   (p.ldr & 3) == 0 && (p.ldb & 7) == 0
             : MODE == EPI_F32
                   ? (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 && (p.ldo & 3) == 0
                   : ((reinterpret_cast<uintptr_t>(p.out) | reinterpret_cast<uintptr_t>(p.branch_out) |
                       reinterpret_cast<uintptr_t>(p.gelu_pre)) & 15) == 0 && (p.ldo & 7) == 0) &&
        (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
    auto direct_ok = [&](const GemmGroup& G_, int n0_, int c0_) {
      return direct_ptrs && c0_ + 32 <= min(p.block_n, G_.n - n0_) && ((G_.c_col + n0_ + c0_) & 7) == 0 &&
             (G_.bias_off < 0 || ((G_.bias_off + n0_ + c0_) & 3) == 0);
    };
    // EPI_RESID: the fp32 residual values of the warp's NEXT 32 x 32 chunk are fetched while the current chunk is
    // processed (and, across tiles, while the MMAs of the next tile run): the epilogue is otherwise paced by one DRAM
    // round trip per 8 rows (ncu: 22 % of the stall samples on the FFMAs that consume the loads).  Staged path:
    // lane = column, res[rr] = row rr (res_ok is warp-uniform); direct path: thread = row, res[] = its 32 columns.
    float res[32];
    bool res_ok = false, res_packed = false;
    // Packed epilogue (every full, aligned 32 x 32 chunk of the bf16-valued modes; see process_packed): the chunk is
    // converted to bf16 BEFORE the shared-memory transpose.  ptrs_packed = the launch-wide part of the condition.
    const bool ptrs_packed =
        p.packed != 0 && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0 &&
        (MODE == EPI_BF16 ? p.head_H == 0 && (p.ldo & 7) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0
         : MODE == EPI_GELU_BF16
             ? (p.ldo & 7) == 0 && ((reinterpret_cast<uintptr_t>(p.out) | reinterpret_cast<uintptr_t>(p.branch_out)) & 15) == 0
             : MODE == EPI_RESID
                   ? p.remap_group == 0 && (p.ldr & 3) == 0 &&
                         ((reinterpret_cast<uintptr_t>(p.resid_out) | reinterpret_cast<uintptr_t>(p.resid_in) |
                           reinterpret_cast<uintptr_t>(p.gamma) | reinterpret_cast<uintptr_t>(p.branch_out)) & 15) == 0 &&
                         (p.branch_out == nullptr || (p.ldb & 7) == 0)
                   : false);
    auto packed_ok = [&](const GemmGroup& G_, int n0_, int c0_, int row0_) {
      return ptrs_packed && row0_ + 32 <= p.M && c0_ + 32 <= min(p.block_n, G_.n - n0_) && ((G_.c_col + n0_ + c0_) & 7) == 0 &&
             (G_.bias_off < 0 || ((G_.bias_off + n0_ + c0_) & 3) == 0);
    };
    auto prefetch_resid = [&](int tile_, int c0_) {
      res_ok = false;
      res_packed = false;
      if (MODE != EPI_RESID || p.resid_in == nullptr || tile_ >= tile_last) return;
      int mb_, g_, nb_;
      decode(tile_, mb_, g_, nb_);
      const GemmGroup& G_ = p.g[g_];
      const int n0_ = nb_ * p.block_n, row_ = mb_ * kBlockM + q * 32 + lane;
      if (packed_ok(G_, n0_, c0_, mb_ * kBlockM + q * 32)) {
        // packed layout: lane = (row lane >> 2 of each 8-row pass, 8 columns (lane & 3) * 8 ..): 32 bytes per pass
        const float* rin_ = p.resid_in + static_cast<long>(mb_ * kBlockM + q * 32 + (lane >> 2)) * p.ldr + G_.c_col + n0_ + c0_ +
                            (lane & 3) * 8;
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          const float4 t0 = *reinterpret_cast<const float4*>(rin_ + static_cast<long>(h) * 8 * p.ldr);
          const float4 t1 = *reinterpret_cast<const float4*>(rin_ + static_cast<long>(h) * 8 * p.ldr + 4);
          res[8 * h] = t0.x; res[8 * h + 1] = t0.y; res[8 * h + 2] = t0.z; res[8 * h + 3] = t0.w;
          res[8 * h + 4] = t1.x; res[8 * h + 5] = t1.y; res[8 * h + 6] = t1.z; res[8 * h + 7] = t1.w;
        }
        res_ok = true;
        res_packed = true;
        return;
      }
      if (!direct_ok(G_, n0_, c0_)) {
        const int row0_ = mb_ * kBlockM + q * 32;
        if (p.remap_group != 0 || c0_ + 32 > min(p.block_n, G_.n - n0_) || row0_ + 32 > p.M) return;
        const float* rin_ = p.resid_in + static_cast<long>(row0_) * p.ldr + G_.c_col + n0_ + c0_ + lane;
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) res[rr] = rin_[rr * p.ldr];
        res_ok = true;
        return;
      }
      if (row_ >= p.M) return;
      const float4* rin_ = reinterpret_cast<const float4*>(p.resid_in + static_cast<long>(row_) * p.ldr + G_.c_col + n0_ + c0_);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 t = rin_[j];
        res[4 * j] = t.x; res[4 * j + 1] = t.y; res[4 * j + 2] = t.z; res[4 * j + 3] = t.w;
      }
    };
    int it = 0;
    prefetch_resid(tile_first, half * 32);
    for (int tile = tile_first; tile < tile_last; tile += tile_step, ++it) {
      int m_blk, g, n_blk;
      decode(tile, m_blk, g, n_blk);
      const GemmGroup& G = p.g[g];
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const int n0 = n_blk * p.block_n;                 // first column of the tile inside the group
      const int n_valid = min(p.block_n, G.n - n0);     // columns of this tile that exist
      const int row0 = m_blk * kBlockM + q * 32;        // first row handled by this warp
      const int rmax = min(32, p.M - row0);
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kAccStride;
      const bool has_bias = p.bias != nullptr && G.bias_off >= 0;

      // Packed path.  ncu (profiles/r02_ncu_summary.md): the small-K launches are bound by SHARED-MEMORY bandwidth, and
      // half of the traffic is this epilogue's fp32 transpose (8 STS.128 + 8 LDS.128 per lane and chunk, 24 % of the
      // wavefronts bank-conflict replays).  Everything that is per element and needs no neighbour -- bias, the bf16
      // rounding of the Linear output, the GELU -- is therefore done while the thread still holds its ROW, and only
      // the bf16 result (64 B per row) goes through shared memory: 4 STS.128 + 4 LDS.128, conflict free with the
      // 16-byte pieces of row r stored at piece ^ (r >> 1).  After the transpose a lane owns 8 columns of 4 rows and
      // does the global I/O (bf16 stores; fp32 residual read-modify-write with gamma and the DropPath factor).
      auto process_packed = [&](const uint32_t (&r)[32], int c0) {
        const int ocol0 = G.c_col + n0 + c0;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (has_bias) {
          const float4* bp = reinterpret_cast<const float4*>(p.bias + G.bias_off + n0 + c0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 t = __ldg(bp + j);
            v[4 * j] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w;
          }
        }
        uint32_t w[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) w[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
        const uint32_t wr = stg + lane * 64, sw = static_cast<uint32_t>(lane >> 1);
        const int rsub = lane >> 2, cq = lane & 3;
        const uint32_t rd = stg + rsub * 64 + (((cq ^ (rsub >> 1)) & 3) << 4);      // + pass * 512: (row >> 1) & 3 = (rsub >> 1) & 3
        const long orow = row0 + rsub;
#pragma unroll
        for (int j = 0; j < 4; ++j) sts_v4(wr + (((j ^ sw) & 3) << 4), w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
        __syncwarp();
        if (MODE == EPI_GELU_BF16) {
          // the staged tile is the bf16 pre-activation (what the reference's Linear emits under autocast): write it out
          // for backward, then stage gelu(pre) the same way
          if (p.branch_out != nullptr) {
            __nv_bfloat16* pre = reinterpret_cast<__nv_bfloat16*>(p.branch_out) + orow * p.ldo + ocol0 + cq * 8;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const float4 t = lds_v4(rd + h * 512);
              *reinterpret_cast<float4*>(pre + static_cast<long>(h) * 8 * p.ldo) = t;
            }
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float2 hf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
            float g0, g1;
            gelu_pair(hf.x, hf.y, g0, g1);
            w[j] = pack_bf16x2(g0, g1);
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) sts_v4(wr + (((j ^ sw) & 3) << 4), w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
          __syncwarp();
        }
        if (MODE == EPI_BF16 || MODE == EPI_GELU_BF16) {
          __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(p.out) + orow * p.ldo + ocol0 + cq * 8;
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            const float4 t = lds_v4(rd + h * 512);
            *reinterpret_cast<float4*>(outp + static_cast<long>(h) * 8 * p.ldo) = t;
          }
        } else {
          // EPI_RESID: out = resid + DropPath factor * gamma * bf16(acc + bias)
          const int ocol = ocol0 + cq * 8;
          float gm[8];
          if (p.gamma != nullptr) {
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(p.gamma + ocol));
            const float4 g1 = __ldg(reinterpret_cast<const float4*>(p.gamma + ocol + 4));
            gm[0] = g0.x; gm[1] = g0.y; gm[2] = g0.z; gm[3] = g0.w; gm[4] = g1.x; gm[5] = g1.y; gm[6] = g1.z; gm[7] = g1.w;
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) gm[i] = 1.f;
          }
          const bool have_res = res_ok && res_packed;
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            const long grow = orow + h * 8;
            const float4 t = lds_v4(rd + h * 512);
            if (p.branch_out != nullptr)
              *reinterpret_cast<float4*>(reinterpret_cast<__nv_bfloat16*>(p.branch_out) + grow * p.ldb + ocol) = t;
            const float sc = p.row_scale != nullptr ? __ldg(p.row_scale + grow / p.rows_per_sample) : 1.f;
            float base[8];
            if (have_res) {
#pragma unroll
              for (int i = 0; i < 8; ++i) base[i] = res[8 * h + i];
            } else if (p.resid_in != nullptr) {
              const float4 b0 = *reinterpret_cast<const float4*>(p.resid_in + grow * p.ldr + ocol);
              const float4 b1 = *reinterpret_cast<const float4*>(p.resid_in + grow * p.ldr + ocol + 4);
              base[0] = b0.x; base[1] = b0.y; base[2] = b0.z; base[3] = b0.w; base[4] = b1.x; base[5] = b1.y; base[6] = b1.z; base[7] = b1.w;
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) base[i] = 0.f;
            }
            const uint32_t tw[4] = {__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w)};
            float o[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&tw[i]));
              o[2 * i] = fmaf(sc * gm[2 * i], f.x, base[2 * i]);
              o[2 * i + 1] = fmaf(sc * gm[2 * i + 1], f.y, base[2 * i + 1]);
            }
            float* ro = p.resid_out + grow * p.ldr + ocol;
            *reinterpret_cast<float4*>(ro) = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<float4*>(ro + 4) = make_float4(o[4], o[5], o[6], o[7]);
          }
        }
        __syncwarp();
      };
      // Direct path: one 32-column chunk, thread = row, global I/O from registers (see above).
      auto process_direct = [&](const uint32_t (&r)[32], int c0) {
        const int row = row0 + lane;
        const bool rv = lane < rmax;
        const int ocol0 = G.c_col + n0 + c0;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (has_bias) {
          const float4* bp = reinterpret_cast<const float4*>(p.bias + G.bias_off + n0 + c0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 t = __ldg(bp + j);
            v[4 * j] += t.x; v[4 * j + 1] += t.y; v[4 * j + 2] += t.z; v[4 * j + 3] += t.w;
          }
        }
        if (MODE == EPI_F32) {
          if (rv) {
            float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + static_cast<long>(row) * p.ldo + ocol0);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
        } else if (MODE == EPI_RESID) {
          uint32_t hb[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) hb[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);   // the Linear emits bf16 under autocast
          if (rv) {
            if (p.branch_out != nullptr) {
              uint4* br = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.branch_out) + static_cast<long>(row) * p.ldb + ocol0);
#pragma unroll
              for (int j = 0; j < 4; ++j) br[j] = make_uint4(hb[4 * j], hb[4 * j + 1], hb[4 * j + 2], hb[4 * j + 3]);
            }
            const float sc = p.row_scale != nullptr ? __ldg(p.row_scale + row / p.rows_per_sample) : 1.f;
            float4* ro = reinterpret_cast<float4*>(p.resid_out + static_cast<long>(row) * p.ldr + ocol0);
            const float4* gp = reinterpret_cast<const float4*>(p.gamma + ocol0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 gm = make_float4(1.f, 1.f, 1.f, 1.f);
              if (p.gamma != nullptr) gm = __ldg(gp + j);
              const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hb[2 * j]));
              const float2 c = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hb[2 * j + 1]));
              float4 o;
              o.x = (p.resid_in != nullptr ? res[4 * j] : 0.f) + sc * gm.x * a.x;
              o.y = (p.resid_in != nullptr ? res[4 * j + 1] : 0.f) + sc * gm.y * a.y;
              o.z = (p.resid_in != nullptr ? res[4 * j + 2] : 0.f) + sc * gm.z * c.x;
              o.w = (p.resid_in != nullptr ? res[4 * j + 3] : 0.f) + sc * gm.w * c.y;
              ro[j] = o;
            }
          }
        } else {
          // bf16 outputs, one 8-column piece (16 bytes) at a time so that only one piece of GELU math is live
          uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + static_cast<long>(row) * p.ldo + ocol0);
          uint4* pr = (MODE == EPI_GELU_BF16 && p.branch_out != nullptr)
                          ? reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.branch_out) + static_cast<long>(row) * p.ldo + ocol0)
                          : nullptr;
          uint4 pv[4];
          if (MODE == EPI_GELU_BWD) {
            const uint4* pp = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.gelu_pre) + static_cast<long>(row) * p.ldo + ocol0);
#pragma unroll
            for (int j = 0; j < 4; ++j) pv[j] = rv ? __ldg(pp + j) : make_uint4(0u, 0u, 0u, 0u);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float* t = v + 8 * j;
            if (MODE == EPI_GELU_BF16) {
              // the reference rounds the pre-activation to bf16 before nn.GELU under autocast
              const uint4 h = make_uint4(pack_bf16x2(t[0], t[1]), pack_bf16x2(t[2], t[3]), pack_bf16x2(t[4], t[5]), pack_bf16x2(t[6], t[7]));
              if (rv && pr != nullptr) pr[j] = h;
              const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float2 hf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hw[i]));
                t[2 * i] = gelu_fast(hf.x);
                t[2 * i + 1] = gelu_fast(hf.y);
              }
            } else if (MODE == EPI_GELU_BWD) {
              const uint32_t pw[4] = {pv[j].x, pv[j].y, pv[j].z, pv[j].w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float2 pf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pw[i]));
                t[2 * i] *= gelu_grad_fast(pf.x);
                t[2 * i + 1] *= gelu_grad_fast(pf.y);
              }
            }
            if (rv) o[j] = make_uint4(pack_bf16x2(t[0], t[1]), pack_bf16x2(t[2], t[3]), pack_bf16x2(t[4], t[5]), pack_bf16x2(t[6], t[7]));
            if (MODE != EPI_BF16) asm volatile("" ::: "memory");
          }
          if (MODE == EPI_GELU_BWD && p.colsum != nullptr) {
            // column sums over the warp's 32 rows: recursive halving (31 shuffles); lane c ends up with column c
            if (!rv) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = 0.f;
            }
#pragma unroll
            for (int w = 16; w >= 1; w >>= 1) {
              const bool up = (lane & w) != 0;
#pragma unroll
              for (int j = 0; j < w; ++j) {
                const float mine = up ? v[j + w] : v[j];
                const float send = up ? v[j] : v[j + w];
                v[j] = mine + __shfl_xor_sync(0xffffffffu, send, w);
              }
            }
            // after the halving steps lane l holds column bitrev-free index: bit b of the lane selected the upper half
            atomicAdd(p.colsum + ocol0 + lane, v[0]);
          }
        }
      };
      // One 32-column chunk: registers (thread = row) -> per-warp smem transpose -> coalesced global I/O.
      auto process_chunk = [&](const uint32_t (&r)[32], int c0) {
        const bool full = (rmax == 32) && (c0 + 32 <= n_valid);
        if (MODE == EPI_BF16 || MODE == EPI_GELU_BF16 || MODE == EPI_GELU_BWD) {
          // Vector path (full chunk, 16-byte aligned bf16 rows, no head remap): rows are staged 36 words apart so both
          // the 16-byte writes (thread = row) and the 16-byte reads (4 lanes per row, 8 columns each) are conflict
          // free; every store instruction then writes 8 rows x 64 B.  ~3x fewer instructions than the 4-byte path.
          const int ocol0 = G.c_col + n0 + c0;
          const bool vec = full && p.head_H == 0 && ((ocol0 | static_cast<int>(p.ldo)) & 7) == 0 &&
                           (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 &&
                           (MODE != EPI_GELU_BF16 || p.branch_out == nullptr || (reinterpret_cast<uintptr_t>(p.branch_out) & 15) == 0) &&
                           (MODE != EPI_GELU_BWD || (reinterpret_cast<uintptr_t>(p.gelu_pre) & 15) == 0);
          if (vec) {
            const int cq = lane & 3, rsub = lane >> 2;
            // EPI_GELU_BWD: the pre-activation rows of this chunk are requested before the accumulators are staged
            uint4 prv[4];
            if (MODE == EPI_GELU_BWD) {
              const __nv_bfloat16* prep = reinterpret_cast<const __nv_bfloat16*>(p.gelu_pre) +
                                          static_cast<long>(row0 + rsub) * p.ldo + ocol0 + cq * 8;
#pragma unroll
              for (int h = 0; h < 4; ++h) prv[h] = __ldg(reinterpret_cast<const uint4*>(prep + static_cast<long>(h) * 8 * p.ldo));
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) sts_v4(stg + lane * 144 + j * 16, r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
            __syncwarp();
            float cs[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) cs[i] = 0.f;
            float bias8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) bias8[i] = has_bias ? __ldg(p.bias + G.bias_off + n0 + c0 + cq * 8 + i) : 0.f;
            const long obase = static_cast<long>(row0 + rsub) * p.ldo + ocol0 + cq * 8;
            __nv_bfloat16* outv = reinterpret_cast<__nv_bfloat16*>(p.out) + obase;
            __nv_bfloat16* prev = (MODE == EPI_GELU_BF16 && p.branch_out != nullptr)
                                      ? reinterpret_cast<__nv_bfloat16*>(p.branch_out) + obase : nullptr;
#pragma unroll
            for (int h2 = 0; h2 < 4; h2 += 2) {        // two 8-row passes at a time (register budget)
              float v[2][8];
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                const uint32_t a = stg + ((h2 + u) * 8 + rsub) * 144 + cq * 32;
                const float4 x0 = lds_v4(a), x1 = lds_v4(a + 16);
                v[u][0] = x0.x + bias8[0]; v[u][1] = x0.y + bias8[1]; v[u][2] = x0.z + bias8[2]; v[u][3] = x0.w + bias8[3];
                v[u][4] = x1.x + bias8[4]; v[u][5] = x1.y + bias8[5]; v[u][6] = x1.z + bias8[6]; v[u][7] = x1.w + bias8[7];
              }
              if (MODE == EPI_GELU_BF16) {
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                  uint4 h;
                  h.x = pack_bf16x2(v[u][0], v[u][1]); h.y = pack_bf16x2(v[u][2], v[u][3]);
                  h.z = pack_bf16x2(v[u][4], v[u][5]); h.w = pack_bf16x2(v[u][6], v[u][7]);
                  if (prev != nullptr) *reinterpret_cast<uint4*>(prev + static_cast<long>(h2 + u) * 8 * p.ldo) = h;
                  // the reference rounds the pre-activation to bf16 before nn.GELU under autocast
                  const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const float2 hf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hw[i]));
                    gelu_pair(hf.x, hf.y, v[u][2 * i], v[u][2 * i + 1]);
                  }
                }
              }
              if (MODE == EPI_GELU_BWD) {
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                  const uint32_t pw[4] = {prv[h2 + u].x, prv[h2 + u].y, prv[h2 + u].z, prv[h2 + u].w};
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const float2 pf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pw[i]));
                    float g0, g1;
                    gelu_grad_pair(pf.x, pf.y, g0, g1);
                    v[u][2 * i] *= g0;
                    v[u][2 * i + 1] *= g1;
                  }
#pragma unroll
                  for (int i = 0; i < 8; ++i) cs[i] += v[u][i];
                }
              }
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                uint4 o;
                o.x = pack_bf16x2(v[u][0], v[u][1]); o.y = pack_bf16x2(v[u][2], v[u][3]);
                o.z = pack_bf16x2(v[u][4], v[u][5]); o.w = pack_bf16x2(v[u][6], v[u][7]);
                *reinterpret_cast<uint4*>(outv + static_cast<long>(h2 + u) * 8 * p.ldo) = o;
              }
            }
            if (MODE == EPI_GELU_BWD && p.colsum != nullptr) {
              // column sums of the 32 rows: fold the 8 row lanes (lane = rsub * 4 + cq), one red.add per column
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 4);
                cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 8);
                cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 16);
              }
              if (rsub == 0) {
#pragma unroll
                for (int i = 0; i < 8; ++i) atomicAdd(p.colsum + ocol0 + cq * 8 + i, cs[i]);
              }
            }
            __syncwarp();
            return;
          }
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) sts_u32(stg + (lane * 33 + j) * 4, r[j]);
        __syncwarp();

        if (MODE == EPI_BF16 || MODE == EPI_GELU_BF16 || MODE == EPI_GELU_BWD) {
          // lane -> (row parity, column pair): each store instruction writes 2 rows x 64 B
          const int cp = (lane & 15) * 2;
          const int rsel = lane >> 4;
          const int col = c0 + cp;                       // column inside the tile
          const bool cv0 = col < n_valid, cv1 = col + 1 < n_valid;
          float b0 = 0.f, b1 = 0.f;
          if (has_bias) {
            if (cv0) b0 = __ldg(p.bias + G.bias_off + n0 + col);
            if (cv1) b1 = __ldg(p.bias + G.bias_off + n0 + col + 1);
          }
          const uint32_t rd = stg + (rsel * 33 + cp) * 4;
          int ocol = G.c_col + n0 + col;
          if (MODE == EPI_BF16 && p.head_H > 0) {
            // feature n = [s][h][j] of this group -> head-major column (pairs never straddle: c_g is even)
            const int cg_all = G.n / p.head_S, cg = cg_all / p.head_H, n = n0 + col;
            const int s_ = n / cg_all, rem = n - s_ * cg_all, h_ = rem / cg, j_ = rem - h_ * cg;
            ocol = s_ * p.head_D + h_ * (p.head_D / p.head_H) + G.head_off + j_;
          }
          const long o0 = static_cast<long>(row0 + rsel) * p.ldo + ocol;
          __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(p.out) + o0;
          __nv_bfloat16* pre = (MODE == EPI_GELU_BF16 && p.branch_out != nullptr)
                                   ? reinterpret_cast<__nv_bfloat16*>(p.branch_out) + o0 : nullptr;
          const long step = 2 * p.ldo;
          if (MODE == EPI_GELU_BWD) {
            // tails and unaligned shapes only (the vector path above takes every full chunk)
            const __nv_bfloat16* prep = reinterpret_cast<const __nv_bfloat16*>(p.gelu_pre) + o0;
            float s0 = 0.f, s1 = 0.f;
            if (cv0) {
              for (int rr = 0; rr < 16; ++rr) {
                if (rr * 2 + rsel < rmax) {
                  const float v0 = lds_f32(rd + rr * 264) * gelu_grad_fast(__bfloat162float(prep[rr * step]));
                  outp[rr * step] = __float2bfloat16(v0);
                  s0 += v0;
                  if (cv1) {
                    const float v1 = lds_f32(rd + rr * 264 + 4) * gelu_grad_fast(__bfloat162float(prep[rr * step + 1]));
                    outp[rr * step + 1] = __float2bfloat16(v1);
                    s1 += v1;
                  }
                }
              }
            }
            if (p.colsum != nullptr) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, 16);
              s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
              if (rsel == 0 && cv0) {
                atomicAdd(p.colsum + ocol, s0);
                if (cv1) atomicAdd(p.colsum + ocol + 1, s1);
              }
            }
          } else if (full) {
            // eight row pairs at a time: all shared-memory reads first, then the (independent) math, then the stores,
            // so the GELU chains of different rows overlap instead of running one after the other
#pragma unroll
            for (int h8 = 0; h8 < 16; h8 += 8) {
              float v0[8], v1[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                v0[i] = lds_f32(rd + (h8 + i) * 264) + b0;
                v1[i] = lds_f32(rd + (h8 + i) * 264 + 4) + b1;
              }
              if (MODE == EPI_GELU_BF16) {
                __nv_bfloat162 hb[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) hb[i] = __floats2bfloat162_rn(v0[i], v1[i]);
                if (pre != nullptr) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) *reinterpret_cast<__nv_bfloat162*>(pre + (h8 + i) * step) = hb[i];
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  // the reference rounds the pre-activation to bf16 before nn.GELU under autocast
                  const float2 hf = __bfloat1622float2(hb[i]);
                  v0[i] = gelu_fast(hf.x);
                  v1[i] = gelu_fast(hf.y);
                }
              }
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<__nv_bfloat162*>(outp + (h8 + i) * step) = __floats2bfloat162_rn(v0[i], v1[i]);
            }
          } else if (cv0) {
            for (int rr = 0; rr < 16; ++rr) {
              if (rr * 2 + rsel < rmax) {
                float v0 = lds_f32(rd + rr * 264) + b0;
                float v1 = lds_f32(rd + rr * 264 + 4) + b1;
                if (MODE == EPI_GELU_BF16) {
                  const __nv_bfloat16 h0 = __float2bfloat16(v0), h1 = __float2bfloat16(v1);
                  if (pre != nullptr) { pre[rr * step] = h0; if (cv1) pre[rr * step + 1] = h1; }
                  v0 = gelu_fast(__bfloat162float(h0));
                  v1 = gelu_fast(__bfloat162float(h1));
                }
                outp[rr * step] = __float2bfloat16(v0);
                if (cv1) outp[rr * step + 1] = __float2bfloat16(v1);
              }
            }
          }
        } else {
          // lane -> column: 128 B of fp32 per row per instruction
          const int col = c0 + lane;
          const bool cv = col < n_valid;
          float bv = 0.f, gv = 1.f;
          if (cv) {
            if (has_bias) bv = __ldg(p.bias + G.bias_off + n0 + col);
            if (MODE == EPI_RESID && p.gamma != nullptr) gv = __ldg(p.gamma + G.c_col + n0 + col);
          }
          const long ocol = G.c_col + n0 + col;
          const uint32_t rd = stg + lane * 4;
          const bool fast = full && p.remap_group == 0 && (p.row_scale == nullptr || p.rows_per_sample >= 32);
          if (fast) {
            if (MODE == EPI_F32) {
              float* outp = reinterpret_cast<float*>(p.out) + static_cast<long>(row0) * p.ldo + ocol;
#pragma unroll
              for (int rr = 0; rr < 32; ++rr) outp[rr * p.ldo] = lds_f32(rd + rr * 132) + bv;
            } else {
              // DropPath factor: a 32-row block spans at most two samples when rows_per_sample >= 32
              float s_a = 1.f, s_b = 1.f;
              int boundary = 32;
              if (p.row_scale != nullptr) {
                const int smp = row0 / p.rows_per_sample;
                boundary = (smp + 1) * p.rows_per_sample - row0;
                s_a = __ldg(p.row_scale + smp);
                s_b = boundary < 32 ? __ldg(p.row_scale + smp + 1) : s_a;
              }
              const float* rin = p.resid_in != nullptr ? p.resid_in + static_cast<long>(row0) * p.ldr + ocol : nullptr;
              float* rout = p.resid_out + static_cast<long>(row0) * p.ldr + ocol;
              __nv_bfloat16* br = p.branch_out != nullptr
                                      ? reinterpret_cast<__nv_bfloat16*>(p.branch_out) + static_cast<long>(row0) * p.ldb + ocol
                                      : nullptr;
#pragma unroll
              for (int r8 = 0; r8 < 32; r8 += 8) {
                float base[8];
                // all loads of a batch before its stores (resid_in may alias resid_out)
                if (res_ok && !res_packed) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) base[i] = res[r8 + i];
                } else {
#pragma unroll
                  for (int i = 0; i < 8; ++i) base[i] = rin != nullptr ? rin[(r8 + i) * p.ldr] : 0.f;
                }
                float acc[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = lds_f32(rd + (r8 + i) * 132) + bv;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const int rr = r8 + i;
                  const __nv_bfloat16 vb = __float2bfloat16(acc[i]);
                  if (br != nullptr) br[rr * p.ldb] = vb;
                  // the reference's Linear emits bf16 under autocast; keep that rounding point
                  rout[rr * p.ldr] = base[i] + (rr < boundary ? s_a : s_b) * gv * __bfloat162float(vb);
                }
              }
            }
          } else if (cv) {
#pragma unroll 1
            for (int r8 = 0; r8 < rmax; r8 += 8) {
              long mo[8];
              float base[8], sc[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const long m = row0 + r8 + i;
                mo[i] = (p.remap_group > 0) ? m + (m / p.remap_group) * p.remap_extra + p.remap_off : m;
                const bool rv = r8 + i < rmax;
                base[i] = (MODE == EPI_RESID && rv && p.resid_in != nullptr) ? p.resid_in[mo[i] * p.ldr + ocol] : 0.f;
                sc[i] = (MODE == EPI_RESID && rv && p.row_scale != nullptr) ? __ldg(p.row_scale + mo[i] / p.rows_per_sample) : 1.f;
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (r8 + i < rmax) {
                  float v = lds_f32(rd + (r8 + i) * 132) + bv;
                  if (MODE == EPI_F32) {
                    reinterpret_cast<float*>(p.out)[mo[i] * p.ldo + ocol] = v;
                  } else {
                    if (p.branch_out != nullptr)
                      reinterpret_cast<__nv_bfloat16*>(p.branch_out)[mo[i] * p.ldb + ocol] = __float2bfloat16(v);
                    v = __bfloat162float(__float2bfloat16(v));
                    p.resid_out[mo[i] * p.ldr + ocol] = base[i] + sc[i] * gv * v;
                  }
                }
              }
            }
          }
        }
        __syncwarp();
      };
      // The TMEM load of the warp's next chunk is in flight while the current one is transposed and stored
      // (tcgen05.ld latency is a few hundred cycles; with K = 160 / 320 the epilogue paces the octic GEMMs).
      if constexpr (MODE == EPI_RESID) {
        uint32_t ra[32];
        for (int c0 = half * 32; c0 < n_valid; c0 += kChunkStep) {
          tmem_ld_32x32(t_addr + c0, ra);
          tmem_ld_wait();
          // (res[] is consumed inside) then fetch the residual rows of the next chunk
          if (packed_ok(G, n0, c0, row0)) process_packed(ra, c0);
          else if (direct_ok(G, n0, c0)) process_direct(ra, c0);
          else process_chunk(ra, c0);
          if (c0 + kChunkStep < n_valid) prefetch_resid(tile, c0 + kChunkStep);
          else prefetch_resid(tile + tile_step, half * 32);
        }
        if (half * 32 >= n_valid) prefetch_resid(tile + tile_step, half * 32);
      } else {
        uint32_t ra[32];
        for (int c0 = half * 32; c0 < n_valid; c0 += kChunkStep) {
          tmem_ld_32x32(t_addr + c0, ra);
          tmem_ld_wait();
          if ((MODE == EPI_BF16 || MODE == EPI_GELU_BF16) && packed_ok(G, n0, c0, row0)) process_packed(ra, c0);
          else if (direct_ok(G, n0, c0)) process_direct(ra, c0);
          else process_chunk(ra, c0);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (NCTA == 2) mbar_arrive_cluster(&tempty_bar[as], 0);
        else mbar_arrive(&tempty_bar[as]);
      }
    }
  }

  tc_fence_before();
  if (NCTA == 2) cluster_sync_all();
  else __syncthreads();
  if (warp == mma_warp) {
    tc_fence_after();
    if (NCTA == 2) tmem_dealloc_pair(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------------------
//  wgrad kernel (MN-major operands, contraction over tokens, split-K with fp32 red.add)
// ------------------------------------------------------------------------------------------------------------
template <int NCTA>
__global__ void __launch_bounds__(kWgradThreads, 1)
gemm_wgrad_kernel(const __grid_constant__ CUtensorMap tmDY, const __grid_constant__ CUtensorMap tmX,
                  const __grid_constant__ WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // warp roles as in gemm_tn_kernel: epilogue warps 0-3, TMA producer 4, MMA issuer 5 (roles_low: producer 0, MMA 1, epilogue 2-5)
  const int prod_warp = p.roles_low ? 0 : 4, mma_warp = p.roles_low ? 1 : 5;
  const int stages = p.num_stages;
  const int b_cols = p.block_n / NCTA;                    // X columns (N extent) held by this CTA: whole 64-wide atoms
  const int b_stage_bytes = b_cols * kBlockK * 2;
  const SmemLayout L = smem_layout(stages, b_stage_bytes, 8);
  const int rank = NCTA == 2 ? static_cast<int>(cluster_ctarank()) : 0;
  const int cid = blockIdx.x / NCTA, ncl = gridDim.x / NCTA;

  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tfull_bar = empty_bar + kMaxStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  if (warp == prod_warp && lane == 0) {
    tma_prefetch_desc(&tmDY);
    tma_prefetch_desc(&tmX);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 4 * NCTA);
    }
    fence_mbar_init();
  }
  if (warp == mma_warp) {
    if (NCTA == 2) tmem_alloc_pair(tmem_ptr, kTmemCols);
    else tmem_alloc(tmem_ptr, kTmemCols);
  }
  tc_fence_before();
  if (NCTA == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // Work distribution (per CTA, or per CTA pair whose tile has 256 dY features): "data-parallel + stream-K".
  //   * whole tiles first: in round r CTA c takes tile r * ncl + c over the FULL token range.  All CTAs then sweep the
  //     tokens in lock step, so every dY / X column block is fetched from DRAM once and shared through L2 (a pure
  //     stream-K line made every CTA stream its own token range: 2.4 GB of DRAM reads for 0.42 GB of operands).
  //   * the remaining total_tiles mod ncl tiles: either p.rem_splits > 0 -- every tile is cut into rem_splits equal token
  //     ranges, one (tile, range) item per CTA, CTAs of one range neighbours (again lock step: used when the items fill
  //     >= 3/4 of the CTAs, the case of the irrep groups whose few tiles would otherwise each stream the operands from
  //     DRAM on their own) -- or their (tile, k-block) pairs, k-block fastest, form one line that is cut into ncl
  //     equal contiguous ranges, so no CTA runs a mostly empty last wave.
  // Every segment (one tile, k-blocks [kb0, kb1)) ends in a red.add epilogue.
  const int kb_total = (p.T + kBlockK - 1) / kBlockK;
  const int full_rounds = p.total_tiles / ncl;
  const int rem_tiles = p.total_tiles - full_rounds * ncl;
  const long rem_units = static_cast<long>(rem_tiles) * kb_total;
  const long r_begin = rem_units * cid / ncl;
  const long r_end = rem_units * (cid + 1) / ncl;
  auto next_seg = [&](int& round, long& u, int& g, int& m_t, int& n_t, int& kb0, int& kb1) -> bool {
    int j;
    if (round < full_rounds) {
      j = round * ncl + cid;
      kb0 = 0;
      kb1 = kb_total;
      ++round;
    } else if (p.rem_splits > 0) {
      if (u != r_begin || cid >= rem_tiles * p.rem_splits) return false;     // one item per CTA
      u = r_begin + 1;
      const int part = cid / rem_tiles, len = (kb_total + p.rem_splits - 1) / p.rem_splits;
      j = full_rounds * ncl + (cid - part * rem_tiles);
      kb0 = part * len;
      kb1 = min(kb_total, kb0 + len);
      if (kb1 <= kb0) return false;
    } else if (u < r_end) {
      const int jr = static_cast<int>(u / kb_total);
      j = full_rounds * ncl + jr;
      kb0 = static_cast<int>(u - static_cast<long>(jr) * kb_total);
      kb1 = static_cast<int>(min(static_cast<long>(kb_total), kb0 + (r_end - u)));
      u += kb1 - kb0;
    } else {
      return false;
    }
    g = 0;
#pragma unroll 1
    for (int i = 1; i < p.num_groups; ++i)
      if (j >= p.g[i].tile_begin) g = i;
    j -= p.g[g].tile_begin;
    m_t = j / p.g[g].n_tiles;
    n_t = j - m_t * p.g[g].n_tiles;
    return true;
  };
  const int n_atoms = b_cols / 64;

  if (warp == prod_warp) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int round = 0, g, m_t, n_t, kb0, kb1;
      long u = r_begin;
      while (next_seg(round, u, g, m_t, n_t, kb0, kb1)) {
        const WgradGroup& G = p.g[g];
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = smem + L.a_off + stage * kAStageBytes;
          uint8_t* b_dst = smem + L.b_off + stage * b_stage_bytes;
          const int a_col0 = G.dy_col + (m_t * NCTA + rank) * kBlockM;
          const int b_col0 = G.x_col + n_t * p.block_n + rank * b_cols;
          // each box: 64 features (128 B, swizzled) x 64 tokens = 8 KiB; consecutive boxes = consecutive MN atoms
          if (NCTA == 2) {
            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * (kAStageBytes + b_stage_bytes));
            for (int i = 0; i < 2; ++i) tma_load_2d_pair(a_dst + i * 8192, &tmDY, &full_bar[stage], a_col0 + i * 64, kb * kBlockK);
            for (int i = 0; i < n_atoms; ++i) tma_load_2d_pair(b_dst + i * 8192, &tmX, &full_bar[stage], b_col0 + i * 64, kb * kBlockK);
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], kAStageBytes + b_stage_bytes);
            for (int i = 0; i < 2; ++i) tma_load_2d(a_dst + i * 8192, &tmDY, &full_bar[stage], a_col0 + i * 64, kb * kBlockK);
            for (int i = 0; i < n_atoms; ++i) tma_load_2d(b_dst + i * 8192, &tmX, &full_bar[stage], b_col0 + i * 64, kb * kBlockK);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == mma_warp) {
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc_bf16(kBlockM * NCTA, p.block_n, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      int round = 0, g, m_t, n_t, kb0, kb1;
      long u = r_begin;
      for (; next_seg(round, u, g, m_t, n_t, kb0, kb1); ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tempty_bar[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * kAccStride;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          // MN-major, SWIZZLE_128B: an atom is 64 MN-elements (128 B) x 8 K-rows (1024 B).
          // SBO = stride between 8-row groups along K (1024 B), LBO = stride between MN atoms (64 K-rows x 128 B).
          const uint64_t da = make_smem_desc(smem_u32(smem + L.a_off + stage * kAStageBytes), 8192, 1024);
          const uint64_t db = make_smem_desc(smem_u32(smem + L.b_off + stage * b_stage_bytes), 8192, 1024);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            // 16 K-rows x 128 B = 2048 B -> +128 in the (addr >> 4) field
            if (NCTA == 2) umma_bf16_pair(d_tmem, da + 128 * k, db + 128 * k, idesc, (kb > kb0) || (k != 0));
            else umma_bf16(d_tmem, da + 128 * k, db + 128 * k, idesc, (kb > kb0) || (k != 0));
          }
          if (NCTA == 2) {
            umma_commit_pair(&empty_bar[stage]);
            if (kb == kb1 - 1) umma_commit_pair(&tfull_bar[as]);
          } else {
            umma_commit(&empty_bar[stage]);
            if (kb == kb1 - 1) umma_commit(&tfull_bar[as]);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    const int q = warp & 3;
    float* stg = reinterpret_cast<float*>(smem + L.stg_off) + (p.roles_low ? warp - 2 : warp) * kStagingWords;
    int it = 0;
    int round = 0, g, m_t, n_t, kb0, kb1;
    long u = r_begin;
    for (; next_seg(round, u, g, m_t, n_t, kb0, kb1); ++it) {
      const WgradGroup& G = p.g[g];
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const int n0 = n_t * p.block_n;
      const int n_valid = min(p.block_n, G.k_in - n0);
      const int row0 = (m_t * NCTA + rank) * kBlockM + q * 32;   // out-feature row inside the group
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kAccStride;
      {
        const int rmax = min(32, G.n_out - row0);
        const bool vec_ok = (G.ldw & 3) == 0 && (reinterpret_cast<uintptr_t>(G.dw) & 15) == 0 && (n0 & 3) == 0;
        for (int c0 = 0; c0 < n_valid; c0 += 32) {
          uint32_t r[32];
          tmem_ld_32x32(t_addr + c0, r);
          tmem_ld_wait();
          if (vec_ok && c0 + 32 <= n_valid) {
            // thread = dW row: eight 16-byte vector reductions straight from registers (scalar RED.F32 at one float per
            // lane is bound by the L2 atomic rate: 4x fewer operations this way)
            if (lane < rmax) {
              float* dst = G.dw + static_cast<long>(row0 + lane) * G.ldw + n0 + c0;
#pragma unroll
              for (int j = 0; j < 8; ++j)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * j), "f"(__uint_as_float(r[4 * j])),
                             "f"(__uint_as_float(r[4 * j + 1])), "f"(__uint_as_float(r[4 * j + 2])),
                             "f"(__uint_as_float(r[4 * j + 3]))
                             : "memory");
            }
            continue;
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = __uint_as_float(r[j]);
          __syncwarp();
          const int col = c0 + lane;
          if (col < n_valid) {
            for (int rr = 0; rr < rmax; ++rr) {
              float* dst = G.dw + static_cast<long>(row0 + rr) * G.ldw + n0 + col;
              atomicAdd(dst, stg[rr * 33 + lane]);   // compiles to RED.ADD.F32 (result unused)
            }
          }
          __syncwarp();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (NCTA == 2) mbar_arrive_cluster(&tempty_bar[as], 0);
        else mbar_arrive(&tempty_bar[as]);
      }
    }
  }

  tc_fence_before();
  if (NCTA == 2) cluster_sync_all();
  else __syncthreads();
  if (warp == mma_warp) {
    tc_fence_after();
    if (NCTA == 2) tmem_dealloc_pair(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------------------
//  host side
// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || ptr == nullptr) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// 2-D bf16 row-major tensor [rows, cols] with row stride `ld` elements; box = (64 cols, box_rows), 128B swizzle.
static int make_map_bf16(CUtensorMap* m, const void* base, long rows, long cols, long ld, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) return OCTIC_ERR_DRIVER;
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld * 2) % 16 != 0) return OCTIC_ERR_ALIGN;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? OCTIC_OK : OCTIC_ERR_TMAP;
}

static int g_num_sms = 0;
static int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return g_num_sms;
}

// Plan of the last launch on this host thread (octic_gemm_last_plan): written right before the kernel launch from the
// variables the launch uses.
static thread_local octic_gemm_plan t_last_plan;
static thread_local bool t_have_plan = false;

int gemm_last_plan(octic_gemm_plan* out) {
  if (out == nullptr || !t_have_plan) return OCTIC_ERR_ARG;
  *out = t_last_plan;
  return OCTIC_OK;
}

constexpr int kMaxDynSmem = 232448;   // 227 KiB
// Warp-role order.  Default: TMA producer / MMA issuer on warps 0 / 1.  OCTIC_GEMM_ROLES_HIGH=1 moves them to the two
// highest warp ids (the issue arbiter is said to prefer high warp ids); measured on B200 it is neutral to worse
// (profiles/r02_gemm_warp_roles.txt: fc2-dgrad + GELU' 420 vs 394 us, dense fc1 dgrad 333 vs 313), so it stays a switch.
static int roles_low_env() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("OCTIC_GEMM_ROLES_HIGH");
    v = (e != nullptr && e[0] == '1') ? 0 : 1;
  }
  return v;
}
// Measured on B200 (tools/gpu/r1_s5_e.sh, profiles/r01_gemm_epilogue_policy_s5.txt): the register-direct epilogue issues
// one 16-byte access per lane to 32 different lines and is bound by L1 line transactions; the staged (coalesced) path
// wins for every mode, so direct is off by default and kept only as an experiment switch.
constexpr int kDefaultDirectMask = 0;

template <int MODE, int NCTA>
static int launch_tn_one(const GemmParams& p, const CUtensorMap& tmA, const CUtensorMap& tmB0, const CUtensorMap& tmB1,
                         int grid, int smem_bytes, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(gemm_tn_kernel<MODE, NCTA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem) != cudaSuccess)
      return OCTIC_ERR_CUDA;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, gemm_tn_kernel<MODE, NCTA>, tmA, tmB0, tmB1, p) == cudaSuccess ? OCTIC_OK : OCTIC_ERR_CUDA;
}
template <int NCTA>
static int launch_tn_mode(const GemmParams& p, const CUtensorMap& tmA, const CUtensorMap& tmB0, const CUtensorMap& tmB1,
                          int grid, int smem_bytes, cudaStream_t stream) {
  switch (p.mode) {
    case EPI_BF16: return launch_tn_one<EPI_BF16, NCTA>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream);
    case EPI_RESID: return launch_tn_one<EPI_RESID, NCTA>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream);
    case EPI_F32: return launch_tn_one<EPI_F32, NCTA>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream);
    case EPI_GELU_BF16: return launch_tn_one<EPI_GELU_BF16, NCTA>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream);
    case EPI_GELU_BWD: return launch_tn_one<EPI_GELU_BWD, NCTA>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream);
    default: return OCTIC_ERR_ARG;
  }
}

int launch_gemm_tn(const octic_gemm_desc* d, cudaStream_t stream) {
  if (d->num_groups < 1 || d->num_groups > OCTIC_MAX_GROUPS) return OCTIC_ERR_ARG;
  if (d->block_n < 16 || d->block_n > 256 || (d->block_n % 16) != 0) return OCTIC_ERR_ARG;
  if (d->M <= 0) return OCTIC_OK;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = d->M;
  p.num_groups = d->num_groups;
  p.block_n = d->block_n;
  // CTA pairs (cta_group::2, M = 256) whenever the B tile splits into two halves of whole 8-row swizzle groups;
  // OCTIC_GEMM_NCTA=1 forces single CTAs (A/B measurements).
  static int forced_ncta = -1;
  if (forced_ncta < 0) {
    const char* e = getenv("OCTIC_GEMM_NCTA");
    forced_ncta = (e != nullptr && e[0] == '1') ? 1 : (e != nullptr && e[0] == '2') ? 2 : 0;
  }
  static int direct_mask = -1;     // bit MODE set: that epilogue takes the register-direct path (OCTIC_GEMM_DIRECT=mask)
  if (direct_mask < 0) {
    const char* e = getenv("OCTIC_GEMM_DIRECT");
    direct_mask = e != nullptr ? atoi(e) : kDefaultDirectMask;
  }
  p.direct = (direct_mask >> d->mode) & 1;
  p.roles_low = roles_low_env();
  {
    static int packed_env = -1;     // OCTIC_GEMM_PACKED=0: fp32-staged epilogue everywhere (A/B measurements)
    if (packed_env < 0) {
      const char* e = getenv("OCTIC_GEMM_PACKED");
      packed_env = (e != nullptr && e[0] == '0') ? 0 : 1;
    }
    p.packed = packed_env;
  }
  // Pairs pay off when the tile's MMA time dominates (dense layers, K >= 512) or the epilogue is the slow head-major
  // scatter; the irrep groups with K = 160 / 320 (3-5 k-blocks per tile) run faster as single CTAs (same measurement).
  int kmax = 0;
  for (int i = 0; i < d->num_groups; ++i) kmax = d->groups[i].k > kmax ? d->groups[i].k : kmax;
  // Weight-stationary tile order (see gemm_tn_kernel) for the grouped small-K launches: every group's whole-K weight
  // tile must fit next to a >= 3-stage A ring (K <= 320 -> 5 k-blocks).  OFF by default: measured SLOWER on B200 at the
  // headline shapes (tools/gpu/r2_f.sh, profiles/r02_gemm_weight_stationary.txt: fc1 172 vs 136 us, proj + residual
  // 166 vs 129, qkv head-major 455 vs 232) -- the L2 -> SM operand traffic it removes was not the limiter, and walking
  // the output in (n block)-major order writes every row in 20-30 separate visits instead of one.  OCTIC_GEMM_WS=1
  // enables it for experiments.
  static int ws_env = -1;
  if (ws_env < 0) {
    const char* e = getenv("OCTIC_GEMM_WS");
    ws_env = (e != nullptr && e[0] == '1') ? 1 : 0;
  }
  const bool pairs_possible = d->block_n % 16 == 0 && d->block_n >= 32 && d->M > kBlockM && num_sms() >= 2;
  const bool want_ws = ws_env == 1 && forced_ncta != 1 && d->num_groups > 1 && kmax <= 320 && pairs_possible &&
                       d->remap_group == 0;
  // round-2 re-measurement with the 256 / 128-column tile rule of pick_block_n_d8 (tools/gpu/r2_v.sh): wide bf16 outputs
  // with K <= 320 and 256-column tiles gain 5-6 % as pairs (fc1 115 -> 109 us, fc2 dgrad 116 -> 109, qkv 89 -> 84); the
  // head-major scatter epilogue stays on pairs and takes a 3-stage ring (176 -> 160 us; single CTAs 164, single CTAs with
  // 3 stages 180).
  const bool wide_small_k = d->num_groups > 1 && kmax <= 320 && d->block_n == 256 && d->head_H == 0 && d->mode == EPI_BF16;
  const bool want_pairs = want_ws || forced_ncta == 2 ||
                          (forced_ncta != 1 && (d->num_groups == 1 || kmax >= 512 || d->head_H > 0 || wide_small_k));
  const int ncta = (want_pairs && pairs_possible) ? 2 : 1;
  p.num_m_blocks = (d->M + kBlockM * ncta - 1) / (kBlockM * ncta);
  int tiles = 0;
  for (int i = 0; i < d->num_groups; ++i) {
    const octic_gemm_group& s = d->groups[i];
    GemmGroup& G = p.g[i];
    if (s.k <= 0 || s.n <= 0) return OCTIC_ERR_ARG;
    // the A box of a group starts at column a_col: the TMA load needs it on a 16-byte boundary (a misaligned start never
    // completes its transaction count and the pipeline's barrier wait times out)
    if (s.a_col % 8 != 0) return OCTIC_ERR_ALIGN;
    G.a_col = s.a_col;
    G.k_blocks = (s.k + kBlockK - 1) / kBlockK;
    G.b_map = s.b_map;
    G.b_row = s.b_row;
    G.n = s.n;
    G.n_tiles = (s.n + d->block_n - 1) / d->block_n;
    G.c_col = s.c_col;
    G.bias_off = s.bias_off;
    G.tile_begin = tiles;
    tiles += G.n_tiles;
    G.head_off = d->head_off[i];
    if (d->head_H > 0) {
      if (d->mode != EPI_BF16 || d->head_S < 1 || d->head_D % d->head_H || s.n % (d->head_S * d->head_H) ||
          ((s.n / (d->head_S * d->head_H)) & 1) || (G.head_off & 1))
        return OCTIC_ERR_ARG;
    }
  }
  p.head_H = d->head_H;
  p.head_S = d->head_S;
  p.head_D = d->head_D;
  p.tiles_per_m = tiles;
  const int b_stage_bytes = (d->block_n / ncta) * kBlockK * 2;
  const int fixed_bytes = 1024 + kEpiWarps * kStagingWords * 4 + (2 * kMaxStages + 4) * 8 + 16 + 2 * 8;
  int stages = (kMaxDynSmem - fixed_bytes) / (kAStageBytes + b_stage_bytes);
  if (want_ws) {
    int kb_max = 0;
    for (int i = 0; i < d->num_groups; ++i) kb_max = p.g[i].k_blocks > kb_max ? p.g[i].k_blocks : kb_max;
    const int ring = (kMaxDynSmem - fixed_bytes - kb_max * b_stage_bytes) / kAStageBytes;
    if (ring >= 3) {
      p.ws = 1;
      p.ws_kb_max = kb_max;
      stages = ring;
    }
  }
  if (stages > kMaxStages) stages = kMaxStages;
  static int stage_cap = -1;      // OCTIC_GEMM_STAGES=n caps the TMA ring depth (pipeline-depth experiments)
  if (stage_cap < 0) {
    const char* e = getenv("OCTIC_GEMM_STAGES");
    stage_cap = e != nullptr ? atoi(e) : 0;
  }
  if (stage_cap >= 2 && stages > stage_cap) stages = stage_cap;
  // Epilogue-paced small-K launches (head-major scatter; irrep groups with the fp32 residual epilogue) run FASTER with a
  // shallow ring: a producer that runs far ahead only competes with the epilogue's own global traffic (measured,
  // tools/gpu/r1_s5_st.sh: qkv head-major 269 -> 214 us, octic proj + residual 152 -> 127 us at 2 stages; K >= 640 and the
  // plain epilogues want the deep ring).
  if (stage_cap == 0 && !p.ws) {
    if (d->mode == EPI_RESID && kmax <= 320 && stages > 2) stages = 2;
    else if (d->head_H > 0 && stages > 3) stages = 3;
    else if (d->mode == EPI_RESID && d->num_groups > 1 && stages > 4) stages = 4;     // fc2 + residual: 168 -> 158 us
  }
  if (stages < 2) return OCTIC_ERR_ARG;
  p.num_stages = stages;
  p.mode = d->mode;
  p.out = d->out;
  p.ldo = d->ldo;
  p.bias = d->bias;
  p.gamma = d->gamma;
  p.resid_in = d->resid_in;
  p.resid_out = d->resid_out;
  p.ldr = d->ldr;
  p.row_scale = d->row_scale;
  p.rows_per_sample = d->rows_per_sample > 0 ? d->rows_per_sample : 1;
  p.branch_out = d->branch_out;
  p.ldb = d->ldb;
  p.remap_group = d->remap_group;
  p.remap_extra = d->remap_extra;
  p.remap_off = d->remap_off;
  p.gelu_pre = d->gelu_pre;
  p.colsum = d->colsum;
  if (p.mode == EPI_GELU_BWD && (p.gelu_pre == nullptr || d->head_H > 0 || d->bias != nullptr)) return OCTIC_ERR_ARG;
  if (p.mode == EPI_RESID && p.resid_out == nullptr) return OCTIC_ERR_ARG;
  // EPI_GELU_BF16 writes its pre-activation copy with the row stride of out: refuse a different ldb instead of ignoring it
  if (p.mode == EPI_GELU_BF16 && p.branch_out != nullptr && d->ldb != 0 && d->ldb != d->ldo) return OCTIC_ERR_ARG;
  if (p.mode != EPI_RESID && p.out == nullptr) return OCTIC_ERR_ARG;

  CUtensorMap tmA, tmB0, tmB1;
  int rc = make_map_bf16(&tmA, d->a, d->M, d->a_cols, d->lda, kBlockM);
  if (rc) return rc;
  rc = make_map_bf16(&tmB0, d->b0, d->b0_rows, d->b0_cols, d->b0_ld, d->block_n / ncta);
  if (rc) return rc;
  if (d->b1 != nullptr) {
    rc = make_map_bf16(&tmB1, d->b1, d->b1_rows, d->b1_cols, d->b1_ld, d->block_n / ncta);
    if (rc) return rc;
  } else {
    tmB1 = tmB0;
  }
  const SmemLayout L = smem_layout(stages, b_stage_bytes, kEpiWarps, p.ws ? p.ws_kb_max : -1);
  const int smem_bytes = L.total + 1024;
  const int total_tiles = p.num_m_blocks * p.tiles_per_m;
  int grid = num_sms() / ncta;                       // CTAs (ncta = 1) or CTA pairs (ncta = 2)
  if (grid > total_tiles) grid = total_tiles;
  grid *= ncta;
  memset(&t_last_plan, 0, sizeof(t_last_plan));
  t_last_plan.kind = OCTIC_GEMM_PLAN_TN;
  t_last_plan.mode = p.mode;
  t_last_plan.ncta = ncta;
  t_last_plan.num_stages = p.num_stages;
  t_last_plan.ws = p.ws;
  t_last_plan.block_n = p.block_n;
  t_last_plan.grid = grid;
  t_last_plan.num_m_blocks = p.num_m_blocks;
  t_last_plan.total_tiles = total_tiles;
  t_last_plan.packed = p.packed;
  t_last_plan.direct = p.direct;
  t_last_plan.roles_low = p.roles_low;
  t_have_plan = true;
  return ncta == 2 ? launch_tn_mode<2>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream)
                   : launch_tn_mode<1>(p, tmA, tmB0, tmB1, grid, smem_bytes, stream);
}

template <int NCTA>
static int launch_wgrad_t(const WgradParams& p, const CUtensorMap& tmDY, const CUtensorMap& tmX, int grid, int smem_bytes,
                          cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(gemm_wgrad_kernel<NCTA>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem) != cudaSuccess)
      return OCTIC_ERR_CUDA;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kWgradThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, gemm_wgrad_kernel<NCTA>, tmDY, tmX, p) == cudaSuccess ? OCTIC_OK : OCTIC_ERR_CUDA;
}

int launch_gemm_wgrad(const octic_wgrad_desc* d, cudaStream_t stream) {
  if (d->num_groups < 1 || d->num_groups > OCTIC_MAX_GROUPS) return OCTIC_ERR_ARG;
  if (d->block_n < 64 || d->block_n > 256 || (d->block_n % 64) != 0) return OCTIC_ERR_ARG;
  if (d->T <= 0) return OCTIC_OK;
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.T = d->T;
  p.num_groups = d->num_groups;
  p.block_n = d->block_n;
  // CTA pairs (M = 256 dY features per tile, each CTA holds half of the X columns) when the halves are whole atoms
  static int forced_ncta = -1;
  if (forced_ncta < 0) {
    const char* e = getenv("OCTIC_GEMM_NCTA");
    forced_ncta = (e != nullptr && e[0] == '1') ? 1 : 0;
  }
  bool wide = false;
  for (int i = 0; i < d->num_groups; ++i) wide = wide || d->groups[i].n_out > kBlockM;
  const int ncta = (forced_ncta != 1 && d->block_n % 128 == 0 && wide && num_sms() >= 2) ? 2 : 1;
  int tiles = 0;
  for (int i = 0; i < d->num_groups; ++i) {
    const octic_wgrad_group& s = d->groups[i];
    WgradGroup& G = p.g[i];
    if (s.n_out <= 0 || s.k_in <= 0 || s.dw == nullptr) return OCTIC_ERR_ARG;
    if (s.dy_col % 8 != 0 || s.x_col % 8 != 0) return OCTIC_ERR_ALIGN;     // TMA box starts on 16-byte boundaries
    G.dy_col = s.dy_col;
    G.x_col = s.x_col;
    G.n_out = s.n_out;
    G.k_in = s.k_in;
    G.dw = s.dw;
    G.ldw = s.ldw;
    G.n_tiles = (s.k_in + d->block_n - 1) / d->block_n;
    G.m_tiles = (s.n_out + kBlockM * ncta - 1) / (kBlockM * ncta);
    G.tile_begin = tiles;
    tiles += G.n_tiles * G.m_tiles;
  }
  p.total_tiles = tiles;
  // stream-K grid: one CTA (pair) per SM (pair); splits > 0: at most tiles * splits of them; each at least 4 k-blocks
  const int kb_total = (d->T + kBlockK - 1) / kBlockK;
  const long total_units = static_cast<long>(tiles) * kb_total;
  long grid_l = num_sms() / ncta;
  if (d->splits > 0 && static_cast<long>(tiles) * d->splits < grid_l) grid_l = static_cast<long>(tiles) * d->splits;
  if (grid_l > (total_units + 3) / 4) grid_l = (total_units + 3) / 4;
  if (grid_l < 1) grid_l = 1;
  p.splits = d->splits;
  p.roles_low = roles_low_env();
  {
    const int ncl = static_cast<int>(grid_l), rem = tiles % ncl;
    const int s_al = rem > 0 ? ncl / rem : 0;
    p.rem_splits = (d->splits <= 0 && s_al >= 2 && 4 * rem * s_al >= 3 * ncl && kb_total >= 8 * s_al) ? s_al : 0;
  }
  const int b_stage_bytes = (d->block_n / ncta) * kBlockK * 2;
  int stages = (kMaxDynSmem - 1024 - (8 * kStagingWords * 4 + (2 * kMaxStages + 4) * 8 + 16)) / (kAStageBytes + b_stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  p.num_stages = stages;

  CUtensorMap tmDY, tmX;
  int rc = make_map_bf16(&tmDY, d->dy, d->T, d->dy_cols, d->ld_dy, kBlockK);
  if (rc) return rc;
  rc = make_map_bf16(&tmX, d->x, d->T, d->x_cols, d->ld_x, kBlockK);
  if (rc) return rc;
  const SmemLayout L = smem_layout(stages, b_stage_bytes, 8);
  const int smem_bytes = L.total + 1024;
  const int grid = static_cast<int>(grid_l) * ncta;
  memset(&t_last_plan, 0, sizeof(t_last_plan));
  t_last_plan.kind = OCTIC_GEMM_PLAN_WGRAD;
  t_last_plan.mode = -1;
  t_last_plan.ncta = ncta;
  t_last_plan.num_stages = p.num_stages;
  t_last_plan.block_n = p.block_n;
  t_last_plan.grid = grid;
  t_last_plan.total_tiles = p.total_tiles;
  t_last_plan.kb_total = kb_total;
  t_last_plan.full_rounds = p.total_tiles / static_cast<int>(grid_l);   // the kernel's ncl = gridDim.x / NCTA
  t_last_plan.rem_tiles = p.total_tiles - t_last_plan.full_rounds * static_cast<int>(grid_l);
  t_last_plan.rem_splits = p.rem_splits;
  t_last_plan.splits = p.splits;
  t_last_plan.roles_low = p.roles_low;
  t_have_plan = true;
  return ncta == 2 ? launch_wgrad_t<2>(p, tmDY, tmX, grid, smem_bytes, stream)
                   : launch_wgrad_t<1>(p, tmDY, tmX, grid, smem_bytes, stream);
}

}  // namespace octic
