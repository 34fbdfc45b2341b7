// Octic / dense multi-head attention on tcgen05 (sm_100a), forward and backward, for ViT-length sequences
// (N = 1..~300 tokens: the whole K, V (and Q, dO in backward) of one (image, head) live in shared memory).
//
// Reference: AttentionD8.forward (octic_vits/d8_layers.py:623-656) = pack 5-tuple -> F.scaled_dot_product_attention ->
// unpack; dense Attention (deit/vit.py:36-50).
//
// Input layout.  q, k, v (and dO in backward) are read HEAD-MAJOR: the head vector of (s, h) is the contiguous column
// range [s*D + h*hd, +hd) of a [B, N, 3D] (dO: [B, N, D]) bf16 tensor.  That is the dense layout of deit/vit.py, and
// for octic layers the qkv LinearD8 GEMM (and the proj dgrad GEMM) write it directly from their epilogues
// (gemm_sm100.cu, "head remap"), so the reference's cat / permute / contiguous copies (d8_layers.py:632-641) never
// exist and the operands arrive by TMA (3-D tensor map [B][N][cols]: rows past N are zero-filled by the hardware).
// Outputs (o; dq, dk, dv) are scattered straight into the packed octic rows of d8_layers.py:650-656 (or the dense row).
//
// Operand tiles.  A row-major [rows][hd] bf16 matrix is kept in the SWIZZLE_32B "atom column" format of sm100_ptx.cuh
// (exactly what a TMA box of 16 columns x rows produces): it feeds tcgen05.mma both K-major (contraction over hd:
// Q K^T, dO V^T) and MN-major (contraction over tokens: P V, P^T dO, dS^T Q, dS K) without a transposed copy, and
// hd = 80 (ViT-H/14) costs no padding.
//
// Warp specialisation.  One control warp (one elected lane) issues every TMA load and every tcgen05.mma; the math
// warps never issue MMAs and never __syncthreads with the control warp: all hand-offs are mbarriers
// (MMA -> math: tcgen05.commit; math -> MMA: one arrive per math thread).
//
// Forward (CTA = (image, head); 8 math warps on 128 TMEM lanes = 128 query rows per tile; two CTAs per SM), ONE pass:
//   S chunk = Q_tile K_chunk^T -> TMEM (two ping-pong buffers) -> p = exp2(s*c - ref*c) -> bf16 P written in place over S
//   -> O += P V_chunk with the A operand read from TMEM (tcgen05.mma .ts form), accumulators in TMEM.
//   ref = the row's reference maximum, fixed by the first chunk and raised LAZILY: only when a later chunk exceeds it by
//   more than 2^8 (in the exponent) are O (TMEM read-modify-write) and the row sum rescaled -- P stays <= 256, exact in
//   bf16's range, and on real score distributions the rescale never runs after the first chunk.  (Round 1 made two
//   passes -- exact row max first: 8 instead of 4 jobs per tile; 182 -> 170 us per launch, profiles/r02_attn_fwd_onepass.txt.)
// Backward (CTA = (image, head); 8 math warps: two warps per TMEM lane quarter split the columns; one CTA per SM):
//   phase 0 (lanes = keys)     S^T = K Q^T, dP^T = V dO^T per query chunk -> P^T, dS^T (bf16, in place) ->
//                              dV += P^T dO, dK += dS^T Q
//   phase 1 (lanes = queries)  S = Q K^T, dP = dO V^T per key chunk -> dS in place -> dQ += dS K
//   The (phase, tile, chunk) jobs form one flat pipeline: the first-level MMAs of job g+2 are issued as soon as the
//   second-level MMAs of job g are, across tile and phase boundaries.
//   delta = rowsum(dO * O) comes from attn_delta_kernel (attention.cu).
#include "attention_common.cuh"
#include "sm100_ptx.cuh"
#include <stdlib.h>

namespace octic {

// Optional in-kernel timeline (tools/attn_trace.cu builds this file with -DOCTIC_ATTN_TRACE): CTA 0 records
// (clock64 << 8 | event id) for the control thread (slot 0) and math thread 0 (slot 1).
#ifdef OCTIC_ATTN_TRACE
__device__ long long g_trace[2 * 2048];
__device__ int g_trace_n[2];
// store-only (the event counter lives in a register of the recording thread): no load latency is added to the timeline
#define OCTIC_TRACE_DECL int tr_i_ = 0
#define OCTIC_TRACE(slot, id)                                                                           \
  do {                                                                                                  \
    if (blockIdx.x == 0 && tr_i_ < 2048) {                                                              \
      g_trace[(slot) * 2048 + tr_i_] = (static_cast<long long>(clock64()) << 8) | (id);                 \
      g_trace_n[slot] = ++tr_i_;                                                                        \
    }                                                                                                   \
  } while (0)
#else
#define OCTIC_TRACE_DECL do { } while (0)
#define OCTIC_TRACE(slot, id) do { } while (0)
#endif

struct ChunkPlan {
  int n;
  int off[8];
  int w[8];
};

__host__ __device__ constexpr int tc_chunk_width(int hd) { return hd <= 96 ? 80 : 64; }

static bool make_plan(ChunkPlan* p, int N, int hd) {
  const int cw = tc_chunk_width(hd);
  const int Rk = (N + 15) / 16 * 16;
  const int units = Rk / 16;
  const int n = (Rk + cw - 1) / cw;
  if (n > 8) return false;
  int off = 0;
  for (int i = 0; i < n; ++i) {
    const int w = 16 * (units / n + (i < units % n ? 1 : 0));
    p->off[i] = off;
    p->w[i] = w;
    off += w;
  }
  for (int i = n; i < 8; ++i) { p->off[i] = off; p->w[i] = 0; }
  p->n = n;
  return true;
}

__device__ __forceinline__ uint32_t pack2_bf16(float lo, float hi) {
  const __nv_bfloat162 b = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&b);
}

__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int x, int y, int z) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z)
      : "memory");
}

// One thread: rows [row0, row0 + R) x columns [col0, col0 + HD) of image b -> an [R][HD] SWIZZLE_32B tile at dst.
// The map's box is 16 columns x box_rows rows (box_rows divides R).  Completion: R * HD * 2 bytes on `bar`.
template <int HD>
__device__ __forceinline__ void tma_load_tile(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int col0, int row0,
                                              int b, int R, int box_rows) {
#pragma unroll
  for (int a = 0; a < HD / 16; ++a)
    for (int r = 0; r < R; r += box_rows)
      tma_load_3d(dst + a * (R * 32) + r * 32, map, bar, col0 + 16 * a, row0 + r, b);
}

// Rows [0, nvalid) of a plain row-major [.][HD] bf16 staging tile -> global rows (scatter through the column map).
// Executed by the `nthreads` math threads (thread index tid).
template <int HD, int GRAN>
__device__ __forceinline__ void store_tile(const uint8_t* stg, __nv_bfloat16* dst, long ld, int nvalid, const int* cb,
                                           const int* sm, int s, int tid, int nthreads) {
  constexpr int EU = GRAN / 2, NU = HD / EU;
  const int rpi = nthreads / NU;
  const int u = tid % NU, r0 = tid / NU;
  if (r0 >= rpi) return;
  const int col = cb[u] + (sm != nullptr ? s * sm[u] : 0);
  // a thread keeps its column unit and walks the rows: shared-memory address and global pointer advance by constants,
  // four rows are loaded before they are stored (the 4-byte scatter of the octic layouts is instruction bound)
  uint32_t sa = smem_u32(stg) + r0 * (HD * 2) + u * GRAN;
  uint8_t* gp = reinterpret_cast<uint8_t*>(dst + static_cast<long>(r0) * ld + col);
  const uint32_t sstep = rpi * (HD * 2);
  const long gstep = static_cast<long>(rpi) * ld * 2;
  int r = r0;
  if (GRAN == 16) {
    for (; r + 3 * rpi < nvalid; r += 4 * rpi) {
      uint4 v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[i].x), "=r"(v[i].y), "=r"(v[i].z), "=r"(v[i].w) : "r"(sa + i * sstep));
#pragma unroll
      for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(gp + i * gstep) = v[i];
      sa += 4 * sstep; gp += 4 * gstep;
    }
    for (; r < nvalid; r += rpi) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sa));
      *reinterpret_cast<uint4*>(gp) = v;
      sa += sstep; gp += gstep;
    }
  } else {
    for (; r + 3 * rpi < nvalid; r += 4 * rpi) {
      uint32_t v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v[i]) : "r"(sa + i * sstep));
#pragma unroll
      for (int i = 0; i < 4; ++i) *reinterpret_cast<uint32_t*>(gp + i * gstep) = v[i];
      sa += 4 * sstep; gp += 4 * gstep;
    }
    for (; r < nvalid; r += rpi) {
      uint32_t v;
      asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(sa));
      *reinterpret_cast<uint32_t*>(gp) = v;
      sa += sstep; gp += gstep;
    }
  }
}

// pieces [P0, P1) (16 fp32 accumulator columns each; compile-time range) of this thread's TMEM lane -> * scale -> bf16
// -> 32 bytes each of its staging row.  All loads are issued before the single wait (TMEM latency paid once).
template <int P0, int P1>
__device__ __forceinline__ void acc_pieces_to_stg(uint32_t taddr, float scale, uint8_t* dst_row) {
  uint32_t r[P1 - P0][16];
#pragma unroll
  for (int i = 0; i < P1 - P0; ++i) tmem_ld_32x16(taddr + (P0 + i) * 16, r[i]);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < P1 - P0; ++i) {
    uint4 v0, v1;
    v0.x = pack2_bf16(__uint_as_float(r[i][0]) * scale, __uint_as_float(r[i][1]) * scale);
    v0.y = pack2_bf16(__uint_as_float(r[i][2]) * scale, __uint_as_float(r[i][3]) * scale);
    v0.z = pack2_bf16(__uint_as_float(r[i][4]) * scale, __uint_as_float(r[i][5]) * scale);
    v0.w = pack2_bf16(__uint_as_float(r[i][6]) * scale, __uint_as_float(r[i][7]) * scale);
    v1.x = pack2_bf16(__uint_as_float(r[i][8]) * scale, __uint_as_float(r[i][9]) * scale);
    v1.y = pack2_bf16(__uint_as_float(r[i][10]) * scale, __uint_as_float(r[i][11]) * scale);
    v1.z = pack2_bf16(__uint_as_float(r[i][12]) * scale, __uint_as_float(r[i][13]) * scale);
    v1.w = pack2_bf16(__uint_as_float(r[i][14]) * scale, __uint_as_float(r[i][15]) * scale);
    *reinterpret_cast<uint4*>(dst_row + (P0 + i) * 32) = v0;
    *reinterpret_cast<uint4*>(dst_row + (P0 + i) * 32 + 16) = v1;
  }
}
// column-half hh of a KS-piece accumulator: pieces [0, (KS+1)/2) or [(KS+1)/2, KS)
template <int KS>
__device__ __forceinline__ void acc_half_to_stg(uint32_t taddr, int hh, float scale, uint8_t* dst_row) {
  if (hh == 0) acc_pieces_to_stg<0, (KS + 1) / 2>(taddr, scale, dst_row);
  else acc_pieces_to_stg<(KS + 1) / 2, KS>(taddr, scale, dst_row);
}

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// Backward math on one 16-column piece, branch-free over the 16 independent elements (the compiler interleaves them):
//   p = exp2(x * scale_log2 - lse), ds = p * (y - delta); columns >= nvalid get p = 0.
// COLS: lse / delta vary along the columns (phase 0: lanes are keys, columns are queries; read from shared memory at
// lse_addr / del_addr); otherwise they are the per-lane constants lse_r / del_r (phase 1).
template <bool COLS>
__device__ __forceinline__ void bwd_piece(const uint32_t (&rx)[16], const uint32_t (&ry)[16], uint32_t (&pkp)[8],
                                          uint32_t (&pkd)[8], float scale_log2, uint32_t lse_addr, uint32_t del_addr,
                                          float lse_r, float del_r, int nvalid) {
  float ls[16], dl[16];
  if (COLS) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 a = lds_f4(lse_addr + q * 16), d = lds_f4(del_addr + q * 16);
      ls[4 * q] = a.x; ls[4 * q + 1] = a.y; ls[4 * q + 2] = a.z; ls[4 * q + 3] = a.w;
      dl[4 * q] = d.x; dl[4 * q + 1] = d.y; dl[4 * q + 2] = d.z; dl[4 * q + 3] = d.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) { ls[i] = lse_r; dl[i] = del_r; }
  }
  float pv[16], dv[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) pv[i] = exp2f(fmaf(__uint_as_float(rx[i]), scale_log2, -ls[i]));
  if (nvalid < 16) {
#pragma unroll
    for (int i = 0; i < 16; ++i) pv[i] = i < nvalid ? pv[i] : 0.f;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) dv[i] = pv[i] * (__uint_as_float(ry[i]) - dl[i]);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    pkp[i] = pack2_bf16(pv[2 * i], pv[2 * i + 1]);
    pkd[i] = pack2_bf16(dv[2 * i], dv[2 * i + 1]);
  }
}

// =====================================================================================================================
//  forward
// =====================================================================================================================
constexpr int kFwdMathThreads = 256;
constexpr int kFwdThreads = kFwdMathThreads + 64;   // + control warp + tail-row warp
constexpr int kTailMax = 8;                         // N mod 128 <= kTailMax: those query rows leave the tensor path
constexpr int kTailKpl = 16;                        // keys per lane of the tail warp (Rk <= 512)
__host__ __device__ inline int attn_tail_rows(int N) { return (N >= 128 && (N & 127) <= kTailMax) ? (N & 127) : 0; }

__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
// 16 consecutive columns (atom column a) of row j of a SWIZZLE_32B tile with R rows -> fp32
__device__ __forceinline__ void lds_row16(uint32_t tile, int R, int a, int j, float (&v)[16]) {
  const uint32_t addr = tile + a * (R * 32) + j * 32;
  const uint32_t sw = ((j >> 2) & 1) << 4;
  const uint4 x = lds_u4(addr + sw), y = lds_u4(addr + (sw ^ 16u));
  v[0] = bf_lo(x.x); v[1] = bf_hi(x.x); v[2] = bf_lo(x.y); v[3] = bf_hi(x.y);
  v[4] = bf_lo(x.z); v[5] = bf_hi(x.z); v[6] = bf_lo(x.w); v[7] = bf_hi(x.w);
  v[8] = bf_lo(y.x); v[9] = bf_hi(y.x); v[10] = bf_lo(y.y); v[11] = bf_hi(y.y);
  v[12] = bf_lo(y.z); v[13] = bf_hi(y.z); v[14] = bf_lo(y.w); v[15] = bf_hi(y.w);
}

template <int HD, int GRAN>
__global__ void __launch_bounds__(kFwdThreads, 2) attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmKV,
                                                                     const __grid_constant__ CUtensorMap tmQ,
                                                                     __nv_bfloat16* __restrict__ o, float* __restrict__ lse,
                                                                     int N, int H, HeadMap m, float scale_log2,
                                                                     const __grid_constant__ ChunkPlan cp,
                                                                     int kv_box_rows,
                                                                     const __nv_bfloat16* __restrict__ qkv, int n_tail) {
  constexpr int KS = HD / 16, CW = tc_chunk_width(HD), OCOL = 2 * CW, NU = HD / (GRAN / 2);
  constexpr int NPW = (CW / 16 + 1) / 2;        // max 16-column pieces per warp in one job
  constexpr int KS0 = (KS + 1) / 2;             // epilogue: accumulator pieces handled by column-half 0
  constexpr uint32_t kTmemCols = 256;
  // BAR_OFULL: one completion per P V job (the lazy rescale waits for the previous job's, the epilogue for the last)
  enum { BAR_K = 0, BAR_V = 1, BAR_Q = 2, BAR_SFULL = 3, BAR_SDONE = 5, BAR_OFULL = 7, BAR_QFREE = 8, NBARS = 9 };
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int Rk = cp.off[cp.n - 1] + cp.w[cp.n - 1];
  const uint32_t kv_bytes = static_cast<uint32_t>(Rk) * HD * 2;
  constexpr uint32_t q_bytes = 128 * HD * 2;
  uint8_t* Ks = smem;
  uint8_t* Vs = Ks + kv_bytes;
  uint8_t* Qs = Vs + kv_bytes;
  float* xch = reinterpret_cast<float*>(Qs + q_bytes);           // [2 job parities][2][128] chunk max exchange between warp pairs
  float* xcl = xch + 512;                                        // [2][128] row sum exchange (own array: the sum of a
                                                                 // fast warp must not overwrite a max its partner has not read)
  int* ocb = reinterpret_cast<int*>(xcl + 256);
  uint64_t* bars = reinterpret_cast<uint64_t*>(ocb + NU + (NU & 1));
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + NBARS);
  // tail warp: q row [HD] + reduction scratch [32][17] (16-byte aligned for vector loads)
  float* tailf = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_ptr + 4) + 15) & ~uintptr_t(15));

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x / H, h = blockIdx.x - b * H;
  __nv_bfloat16* orows = o + static_cast<long>(b) * N * m.D;
  const int Nm = N - n_tail;                                     // query rows handled by the tensor path

  if (tid < NU) ocb[tid] = o_col(m, h, tid * (GRAN / 2));
  if (tid == kFwdMathThreads) {
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmQ);
    mbar_init(&bars[BAR_K], 1); mbar_init(&bars[BAR_V], 1); mbar_init(&bars[BAR_Q], 1);
    mbar_init(&bars[BAR_SFULL], 1); mbar_init(&bars[BAR_SFULL + 1], 1);
    mbar_init(&bars[BAR_SDONE], kFwdMathThreads); mbar_init(&bars[BAR_SDONE + 1], kFwdMathThreads);
    mbar_init(&bars[BAR_OFULL], 1);
    mbar_init(&bars[BAR_QFREE], kFwdMathThreads);
    fence_mbar_init();
    // first operand loads before the TMEM allocation and the block barrier (this thread initialised their barriers)
    mbar_arrive_expect_tx(&bars[BAR_K], kv_bytes);
    tma_load_tile<HD>(smem_u32(Ks), &tmKV, &bars[BAR_K], m.D + h * HD, 0, b, Rk, kv_box_rows);
    mbar_arrive_expect_tx(&bars[BAR_Q], q_bytes);
    tma_load_tile<HD>(smem_u32(Qs), &tmQ, &bars[BAR_Q], h * HD, 0, b, 128, 128);
    mbar_arrive_expect_tx(&bars[BAR_V], kv_bytes);
    tma_load_tile<HD>(smem_u32(Vs), &tmKV, &bars[BAR_V], 2 * m.D + h * HD, 0, b, Rk, kv_box_rows);
  }
  if (warp == 8) tmem_alloc(tmem_ptr, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t q_addr = smem_u32(Qs), k_addr = smem_u32(Ks), v_addr = smem_u32(Vs);
  const int nt = (Nm + 127) >> 7, nc = cp.n, njobs = nc;

  if (warp == 9) {
    // -------------------------------------------------- tail warp --------------------------------------------------
    // N = 128 k + (a few) rows (ViT: 256 patches + cls = 257): a third 128-row tensor tile would be 99 % padding, i.e.
    // a third of all MMA work.  The last n_tail query rows are instead done here on the CUDA cores, from the same K / V
    // tiles in shared memory, while the tensor pipeline runs the full tiles: lane = key (stride 32), exact softmax.
    if (n_tail > 0) {
      float* qf = tailf;
      float* red = tailf + HD;
      const int kpl = (Rk + 31) >> 5;
      mbar_wait(&bars[BAR_K], 0);
      for (int r = Nm; r < N; ++r) {
        const __nv_bfloat16* qrow = qkv + (static_cast<long>(b) * N + r) * (3L * m.D) + h * HD;
        for (int i = lane; i < HD / 2; i += 32) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(qrow + 2 * i));
          qf[2 * i] = f.x * scale_log2;
          qf[2 * i + 1] = f.y * scale_log2;
        }
        __syncwarp();
        float sc[kTailKpl];
#pragma unroll
        for (int i = 0; i < kTailKpl; ++i) sc[i] = 0.f;
#pragma unroll 1
        for (int a = 0; a < KS; ++a) {
          float q16[16];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float4 f = lds_f4(smem_u32(qf) + (a * 16 + u * 4) * 4);
            q16[4 * u] = f.x; q16[4 * u + 1] = f.y; q16[4 * u + 2] = f.z; q16[4 * u + 3] = f.w;
          }
#pragma unroll
          for (int i = 0; i < kTailKpl; ++i) {
            const int j = lane + 32 * i;
            if (i < kpl && j < Rk) {
              float kv[16];
              lds_row16(k_addr, Rk, a, j, kv);
              float acc = sc[i];
#pragma unroll
              for (int c = 0; c < 16; ++c) acc = fmaf(q16[c], kv[c], acc);
              sc[i] = acc;
            }
          }
        }
        float mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < kTailKpl; ++i) {
          if (lane + 32 * i >= N) sc[i] = -INFINITY;
          mx = fmaxf(mx, sc[i]);
        }
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o2));
        float l = 0.f;
#pragma unroll
        for (int i = 0; i < kTailKpl; ++i) {
          sc[i] = exp2f(sc[i] - mx);          // -inf -> 0
          l += sc[i];
        }
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o2);
        if (lane == 0 && lse != nullptr) lse[(static_cast<long>(b) * H + h) * N + r] = (mx + log2f(l)) * kLn2;
        const float inv = 1.0f / l;
        if (r == Nm) mbar_wait(&bars[BAR_V], 0);
#pragma unroll 1
        for (int a = 0; a < KS; ++a) {
          float acc[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) acc[c] = 0.f;
#pragma unroll
          for (int i = 0; i < kTailKpl; ++i) {
            const int j = lane + 32 * i;
            if (i < kpl && j < Rk) {
              // P is rounded to bf16 like the tensor path (the reference's SDPA also multiplies a bf16 P with V)
              const float pj = __bfloat162float(__float2bfloat16(sc[i]));
              float vv[16];
              lds_row16(v_addr, Rk, a, j, vv);
#pragma unroll
              for (int c = 0; c < 16; ++c) acc[c] = fmaf(pj, vv[c], acc[c]);
            }
          }
#pragma unroll
          for (int c = 0; c < 16; ++c) red[lane * 17 + c] = acc[c];
          __syncwarp();
          if (lane < 16) {
            float t0 = 0.f, t1 = 0.f;
#pragma unroll
            for (int u = 0; u < 32; u += 2) { t0 += red[u * 17 + lane]; t1 += red[(u + 1) * 17 + lane]; }
            orows[static_cast<long>(r) * m.D + o_col(m, h, a * 16 + lane)] = __float2bfloat16((t0 + t1) * inv);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 8) {
    // ------------------------------------------------ control warp ------------------------------------------------
    // The whole warp runs the loops (so addresses and descriptors stay warp-uniform); lane 0 issues TMA / MMA / commit.
    const bool leader = lane == 0;
    OCTIC_TRACE_DECL;
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    const int colq = h * HD, colk = m.D + h * HD, colv = 2 * m.D + h * HD;
    // (K, the first Q tile and V were requested by this warp's lane 0 in the prologue)
    const uint32_t q_lo = desc_lo_sw32(q_addr, 0), k_lo = desc_lo_sw32(k_addr, 0), v_lo = desc_lo_sw32(v_addr, Rk * 32);
    const uint32_t q_step = (128 * 32) >> 4, k_step = static_cast<uint32_t>(Rk * 32) >> 4;
    const uint32_t idesc_pv = make_idesc_bf16(128, HD, 0, 1);

    auto issue_s = [&](int c, int buf) {      // S chunk c = Q_tile K_c^T  -> buffer buf
      const uint32_t idesc = make_idesc_bf16(128, cp.w[c], 0, 0);
      const uint32_t d = tb + buf * CW, kb = k_lo + cp.off[c] * 2;
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) umma_ss_lohi(d, q_lo + ks * q_step, kb + ks * k_step, kDescHiSw32, idesc, ks != 0);
        umma_commit(&bars[BAR_SFULL + buf]);
      }
    };
    // P of K-step kk: warp set 0 wrote the first half of the pieces at columns kk * 8, set 1 the second half at the
    // start of its own column range (see the math warps)
    auto issue_pv = [&](int c, int buf, bool first, bool last) {   // O (+)= P_c V_c, P read from TMEM
      const int nk = cp.w[c] >> 4, hsplit = (nk + 1) >> 1;
      const uint32_t a = tb + buf * CW, vb = v_lo + cp.off[c] * 2;
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < CW / 16; ++kk)
          if (kk < nk) {
            const uint32_t ak = kk < hsplit ? kk * 8 : hsplit * 16 + (kk - hsplit) * 8;
            umma_ts_lohi(tb + OCOL, a + ak, vb + kk * 32, kDescHiSw32, idesc_pv, !(first && kk == 0));
          }
        umma_commit(&bars[BAR_OFULL]);
      }
    };

    mbar_wait(&bars[BAR_K], 0);
    bool v_ready = false;
    uint32_t phq = 0, phd0 = 0, phd1 = 0, phf = 0;
    for (int t = 0; t < nt; ++t) {
      if (t > 0) {
        mbar_wait(&bars[BAR_QFREE], phf);      // epilogue of tile t-1 has drained O and the staging copy in Qs
        phf ^= 1u;
        if (leader) {
          mbar_arrive_expect_tx(&bars[BAR_Q], q_bytes);
          tma_load_tile<HD>(q_addr, &tmQ, &bars[BAR_Q], colq, t * 128, b, 128, 128);
        }
      }
      mbar_wait(&bars[BAR_Q], phq);
      phq ^= 1u;
      tc_fence_after();
      issue_s(0, 0);
      if (nc > 1) issue_s(1, 1);
      for (int j = 0; j < njobs; ++j) {
        const int buf = j & 1;
        if (buf == 0) { mbar_wait(&bars[BAR_SDONE], phd0); phd0 ^= 1u; }
        else { mbar_wait(&bars[BAR_SDONE + 1], phd1); phd1 ^= 1u; }
        tc_fence_after();
        if (leader) OCTIC_TRACE(0, 1);
        if (!v_ready) { mbar_wait(&bars[BAR_V], 0); v_ready = true; }
        issue_pv(j, buf, j == 0, j == njobs - 1);
        if (j + 2 < njobs) issue_s(j + 2, buf);
        if (leader) OCTIC_TRACE(0, 2);
      }
    }
  } else {
    // -------------------------------------------------- math warps --------------------------------------------------
    // Warp (q4, bsel) works on TMEM lane quarter q4 of EVERY job: set bsel = 0 takes the first half of the chunk's
    // 16-column pieces, set 1 the second half (half the math latency per job; the other buffer's job keeps the tensor
    // pipe busy): chunk max (combined with the partner set through one pair barrier per job), lazy raise of the row's
    // reference, p = exp2(.), bf16 P written at the start of the set's own column range -- output piece q lands on columns
    // of the set's input piece q/2, already consumed, so the sets need no barrier for that.  The row sums of the two
    // warps are combined once per tile; for the output accumulator the pair splits the columns (hh = bsel).
    const int q4 = warp & 3, bsel = warp >> 2, hh = bsel;
    const int rloc = q4 * 32 + lane;                   // row inside the tile
    OCTIC_TRACE_DECL;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    // largest exponent gap a row tolerates before it is rescaled (raw score units): p <= 2^kLazyExp
    constexpr float kLazyExp = 8.0f;
    const float lazy_gap = kLazyExp / scale_log2;
    int gj = 0;                                        // jobs done so far = P V jobs committed before the current one
    uint32_t phs0 = 0u, phs1 = 0u;                     // phases of the two S buffers (nc may be odd: tiles restart at buffer 0)
    for (int t = 0; t < nt; ++t) {
      const bool warp_valid = t * 128 + q4 * 32 < Nm;
      float mx = -INFINITY, l = 0.f, moff = 0.f;       // mx: the row's reference maximum, moff = mx * scale_log2
      for (int j = 0; j < njobs; ++j, ++gj) {
        const int c = j;
        const int buf = j & 1;
        if (buf == 0) { mbar_wait(&bars[BAR_SFULL], phs0); phs0 ^= 1u; }
        else { mbar_wait(&bars[BAR_SFULL + 1], phs1); phs1 ^= 1u; }
        tc_fence_after();
        if (tid == 0) OCTIC_TRACE(1, 3);
        if (warp_valid) {
          const int w = cp.w[c], k0 = cp.off[c];
          const int np = w >> 4, hsplit = (np + 1) >> 1;
          const int p0 = bsel ? hsplit : 0, cnt = bsel ? np - hsplit : hsplit;     // this set's pieces [p0, p0 + cnt)
          const uint32_t ta = t_lane + buf * CW + p0 * 16;                          // the set's inputs / outputs start here
          constexpr int QMAX = (CW / 16 + 1) / 2;
          // all of the set's pieces are fetched with one TMEM round trip
          uint32_t r[QMAX][16];
#pragma unroll
          for (int q = 0; q < QMAX; ++q)
            if (q < cnt) tmem_ld_32x16(ta + q * 16, r[q]);
          tmem_ld_wait();
          // ---- chunk maximum of the row: this set's columns, then the partner set's (pair barrier) ----
          float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
          for (int q = 0; q < QMAX; ++q)
            if (q < cnt) {
              const int nvalid = N - (k0 + (p0 + q) * 16);
              if (nvalid < 16) {
#pragma unroll
                for (int i = 0; i < 16; ++i) r[q][i] = i < nvalid ? r[q][i] : 0xff800000u;      // -inf
              }
#pragma unroll
              for (int i = 0; i < 16; i += 4) {
                m0 = fmaxf(m0, __uint_as_float(r[q][i])); m1 = fmaxf(m1, __uint_as_float(r[q][i + 1]));
                m2 = fmaxf(m2, __uint_as_float(r[q][i + 2])); m3 = fmaxf(m3, __uint_as_float(r[q][i + 3]));
              }
            }
          float* xm = xch + (j & 1) * 256;              // double buffered by job parity: one pair barrier per job suffices
          const float mloc = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
          xm[bsel * 128 + rloc] = mloc;
          named_bar_sync(1 + q4, 64);
          const float mc = fmaxf(mloc, xm[(bsel ^ 1) * 128 + rloc]);
          if (j == 0) {
            mx = mc;                                     // O is empty: nothing to rescale
            moff = mx * scale_log2;
          } else {
            const bool need = mc > mx + lazy_gap;        // both warps of the pair see the same mc and mx
            if (__any_sync(0xffffffffu, need)) {
              // rare: raise the reference of the rows that need it.  O holds the P V sums of jobs < j under the old
              // reference: wait for the previous job's MMAs (the control warp cannot have issued this job's yet), then
              // scale this warp's half of the O columns and the partial row sum
              const float f = need ? exp2f((mx - mc) * scale_log2) : 1.0f;
              mbar_wait(&bars[BAR_OFULL], static_cast<uint32_t>((gj - 1) & 1));
              tc_fence_after();
              const int pa = hh == 0 ? 0 : (KS + 1) / 2, pb = hh == 0 ? (KS + 1) / 2 : KS;
              for (int pz = pa; pz < pb; ++pz) {
                uint32_t ov[16];
                tmem_ld_32x16(t_lane + OCOL + pz * 16, ov);
                tmem_ld_wait();
                uint32_t lo[8], hi[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  lo[i] = __float_as_uint(__uint_as_float(ov[i]) * f);
                  hi[i] = __float_as_uint(__uint_as_float(ov[8 + i]) * f);
                }
                tmem_st_32x8(t_lane + OCOL + pz * 16, lo);
                tmem_st_32x8(t_lane + OCOL + pz * 16 + 8, hi);
              }
              tmem_st_wait();
              l *= f;
              if (need) { mx = mc; moff = mx * scale_log2; }
            }
          }
          // ---- p = exp2(s * c - ref * c), row sum, bf16 P in place ----
          float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
#pragma unroll
          for (int q = 0; q < QMAX; ++q)
            if (q < cnt) {
              float e[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) e[i] = exp2f(fmaf(__uint_as_float(r[q][i]), scale_log2, -moff));   // -inf -> 0
              uint32_t pk[8];
#pragma unroll
              for (int i = 0; i < 16; i += 4) {
                l0 += e[i]; l1 += e[i + 1]; l2 += e[i + 2]; l3 += e[i + 3];
                pk[i >> 1] = pack2_bf16(e[i], e[i + 1]);
                pk[(i >> 1) + 1] = pack2_bf16(e[i + 2], e[i + 3]);
              }
              tmem_st_32x8(ta + q * 8, pk);
            }
          l += (l0 + l1) + (l2 + l3);
          tmem_st_wait();
        }
        tc_fence_before();
        if (tid == 0) OCTIC_TRACE(1, 5);
        mbar_arrive(&bars[BAR_SDONE + buf]);
      }
      if (warp_valid) {
        // total row sum = both warps of the quarter (written before, read after the pair barrier)
        xcl[bsel * 128 + rloc] = l;
        named_bar_sync(1 + q4, 64);
        l += xcl[(bsel ^ 1) * 128 + rloc];
      }
      mbar_wait(&bars[BAR_OFULL], static_cast<uint32_t>((gj - 1) & 1));      // the tile's last P V job
      tc_fence_after();
      if (tid == 0) OCTIC_TRACE(1, 6);
      const int row = t * 128 + rloc;
      if (warp_valid) {
        const float inv = 1.0f / l;
        acc_half_to_stg<KS>(t_lane + OCOL, hh, inv, Qs + rloc * (HD * 2));
        if (hh == 0 && lse != nullptr && row < Nm)
          lse[(static_cast<long>(b) * H + h) * N + row] = (mx * scale_log2 + log2f(l)) * kLn2;
      }
      tc_fence_before();
      named_bar_sync(5, kFwdMathThreads);
      store_tile<HD, GRAN>(Qs, orows + static_cast<long>(t) * 128 * m.D, m.D, min(128, Nm - t * 128), ocb, nullptr, 0, tid,
                           kFwdMathThreads);
      fence_proxy_async_smem();      // the next Q tile arrives in Qs through the async proxy
      if (tid == 0) OCTIC_TRACE(1, 7);
      mbar_arrive(&bars[BAR_QFREE]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =====================================================================================================================
//  backward
// =====================================================================================================================
constexpr int kBwdMathThreads = 256;
constexpr int kBwdTailWarps = 3;                    // staged dQ: all three take the tail tokens as keys; else as key / as query / idle
constexpr int kBwdThreads = kBwdMathThreads + 32 + 32 * kBwdTailWarps;   // + control warp + tail-row warps

template <int HD, int GRAN>
__global__ void __launch_bounds__(kBwdThreads, 1) attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQKV,
                                                                     const __grid_constant__ CUtensorMap tmDO,
                                                                     const float* __restrict__ lse,
                                                                     const float* __restrict__ delta,
                                                                     __nv_bfloat16* __restrict__ dqkv, int N, int H, HeadMap m,
                                                                     float scale, float scale_log2,
                                                                     const __grid_constant__ ChunkPlan cp,
                                                                     int box_rows, int n_tail,
                                                                     const __grid_constant__ CUtensorMap tmDS,
                                                                     __nv_bfloat16* __restrict__ ds_ws, int* ds_slots,
                                                                     int n_slots, int ds_box_rows) {
  constexpr int KS = HD / 16, CW = tc_chunk_width(HD), ACC = 4 * CW, NU = HD / (GRAN / 2);
  constexpr int NPW = (CW / 16 + 1) / 2;        // max 16-column pieces per warp in the math step
  constexpr int KS0 = (KS + 1) / 2;             // epilogue: pieces of the accumulator handled by column-half 0
  constexpr uint32_t kTmemCols = 512;
  constexpr uint32_t stg_bytes = 128 * HD * 2;
  static_assert(ACC + 2 * HD <= 512, "TMEM budget");
  enum { BAR_KQ = 0, BAR_VDO = 1, BAR_LFULL = 2, BAR_MDONE = 4, BAR_ACC = 6, BAR_DS = 7, BAR_TAIL = 8, BAR_DSLOAD = 9,
         BAR_DQ = 10, BAR_DQFREE = 12, NBARS = 14 };
  // Staged dQ (ds_ws != nullptr): the query-major phase 1 (S, dP and the exponentials a second time) is replaced by
  //   phase 0  also writes dS^T (bf16, [key][query], rows/columns up to Rk) into this CTA's slot of an L2-resident scratch,
  //   phase 1' TMA-loads it back as the MN-major A operand of dQ_tile = dS[tile queries, all keys] K (Rk/16 K-steps).
  // One slot per resident CTA (claimed with an atomic CAS, released after the last TMA load): 2 x SM-count slots of
  // Rk x Rk bf16 stay in L2 (44 MB at N = 257), the data makes no HBM round trip.
  const bool staged = ds_ws != nullptr;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int Rk = cp.off[cp.n - 1] + cp.w[cp.n - 1];
  const uint32_t mat_bytes = static_cast<uint32_t>(Rk) * HD * 2;
  uint8_t* Qs = smem;
  uint8_t* Ks = Qs + mat_bytes;
  uint8_t* Vs = Ks + mat_bytes;
  uint8_t* dOs = Vs + mat_bytes;
  uint8_t* stg = dOs + mat_bytes;                 // 2 x [128][HD] bf16 staging; also absorbs the A-tile over-read of dOs
  float* lse_s = reinterpret_cast<float*>(stg + 2 * stg_bytes);
  float* del_s = lse_s + Rk;
  int* cb = reinterpret_cast<int*>(del_s + Rk);
  int* sm = cb + NU;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + NU + ((2 * NU) & 1));
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + NBARS);
  float* tail_red = reinterpret_cast<float*>(tmem_ptr + 4);      // two tail warps x [32][33] reduction scratch
  float* tail_xch = tail_red + 2 * 32 * 33;                      // staged: [tail warps][8 atom columns][32] partial sums

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x / H, h = blockIdx.x - b * H;
  const long ld3 = 3L * m.D;
  const int Nm = N - n_tail;                                     // rows (as keys and as queries) of the tensor path
  __nv_bfloat16* drows = dqkv + static_cast<long>(b) * N * ld3;

  if (tid < NU) {
    int base, smul;
    qkv_col(m, h, tid * (GRAN / 2), base, smul);
    cb[tid] = base; sm[tid] = smul;
  }
  if (tid == kBwdMathThreads) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    mbar_init(&bars[BAR_KQ], 1); mbar_init(&bars[BAR_VDO], 1);
    mbar_init(&bars[BAR_LFULL], 1); mbar_init(&bars[BAR_LFULL + 1], 1);
    mbar_init(&bars[BAR_MDONE], kBwdMathThreads); mbar_init(&bars[BAR_MDONE + 1], kBwdMathThreads);
    mbar_init(&bars[BAR_ACC], 1);
    mbar_init(&bars[BAR_DS], kBwdMathThreads + (n_tail > 0 ? 32 * kBwdTailWarps : 0));
    mbar_init(&bars[BAR_TAIL], 32 * kBwdTailWarps);
    mbar_init(&bars[BAR_DSLOAD], 1);
    mbar_init(&bars[BAR_DQ], 1); mbar_init(&bars[BAR_DQ + 1], 1);
    mbar_init(&bars[BAR_DQFREE], kBwdMathThreads); mbar_init(&bars[BAR_DQFREE + 1], kBwdMathThreads);
    fence_mbar_init();
    {
      // the operand loads go out before anything else (this thread initialised their barriers; nobody touches the tiles
      // before the __syncthreads below): the scratch-slot claim -- an atomic round trip to L2 -- and the TMEM allocation
      // then run under the DRAM latency of the loads instead of in front of it
      const uint32_t q_a = smem_u32(Qs), k_a = smem_u32(Ks), v_a = smem_u32(Vs), do_a = smem_u32(dOs);
      mbar_arrive_expect_tx(&bars[BAR_KQ], 2 * mat_bytes);
      tma_load_tile<HD>(k_a, &tmQKV, &bars[BAR_KQ], m.D + h * HD, 0, b, Rk, box_rows);
      tma_load_tile<HD>(q_a, &tmQKV, &bars[BAR_KQ], h * HD, 0, b, Rk, box_rows);
      mbar_arrive_expect_tx(&bars[BAR_VDO], 2 * mat_bytes);
      tma_load_tile<HD>(v_a, &tmQKV, &bars[BAR_VDO], 2 * m.D + h * HD, 0, b, Rk, box_rows);
      tma_load_tile<HD>(do_a, &tmDO, &bars[BAR_VDO], h * HD, 0, b, Rk, box_rows);
    }
    if (staged) {
      int sl = static_cast<int>(blockIdx.x % static_cast<unsigned>(n_slots));
      uint32_t spins = 0;
      while (atomicCAS(&ds_slots[sl], 0, 1) != 0) {
        sl = sl + 1 == n_slots ? 0 : sl + 1;
        if (++spins > OCTIC_WAIT_SPINS) __trap();
      }
      tmem_ptr[1] = static_cast<uint32_t>(sl);
    }
  }
  if (warp == 8) tmem_alloc(tmem_ptr, kTmemCols);
  if (tid < kBwdMathThreads) {
    for (int i = tid; i < Rk; i += kBwdMathThreads) {
      const long off = (static_cast<long>(b) * H + h) * N + i;
      lse_s[i] = i < N ? lse[off] * kLog2e : INFINITY;     // +inf -> P = 0 for padded queries
      del_s[i] = i < N ? delta[off] : 0.f;
    }
    for (int i = tid; i < static_cast<int>(2 * stg_bytes / 16); i += kBwdMathThreads)
      reinterpret_cast<uint4*>(stg)[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t q_addr = smem_u32(Qs), k_addr = smem_u32(Ks), v_addr = smem_u32(Vs), do_addr = smem_u32(dOs);
  const int nt = (Nm + 127) >> 7, nc = cp.n;
  const int jobs_per_phase = nt * nc, G = staged ? jobs_per_phase : 2 * jobs_per_phase;
  const int slot = staged ? static_cast<int>(tmem_ptr[1]) : 0;
  // dS^T [Rk keys][ldS queries].  Measured (tools/gpu/r2_ab.sh / r2_ad.sh): a 128-byte-multiple pitch (640 B at N = 257)
  // makes the TMA read faster (1.5 k vs 2.6 k cycles per tile) but the 32-byte-per-lane writes of the math warps slower
  // (jobs 1.4-1.6 k -> 1.8-2.4 k cycles): 421 vs 389 us per launch, so the pitch stays Rk.
  const int ldS = Rk;
  __nv_bfloat16* ds_mine = staged ? ds_ws + static_cast<long>(slot) * Rk * ldS : nullptr;

  if (warp >= 9) {
    // -------------------------------------------------- tail warps --------------------------------------------------
    // N = 128 k + a few rows (ViT: 257): the last n_tail tokens would cost a whole 128-lane tile in BOTH phases.  They
    // stay in the column (chunk) dimension of the tensor path; their own rows are done here on the CUDA cores from the
    // same shared-memory tiles: warp 9 takes them as keys (dK_j, dV_j over all queries), warp 10 as queries (dQ_i over
    // all keys).  lane = the other token (stride 32).  P and dS are rounded to bf16 like the tensor path's operands.
    if (n_tail > 0 && staged) {
      // Staged dQ: the tail tokens' dQ rows come from the tensor path (one more query tile in phase 1'), and ALL tail
      // warps take the tail tokens as keys, splitting the queries (warp 9 + p: lane groups p, p + 3, p + 6, ..) -- they
      // are on the critical path now: phase 1' needs their dS^T rows and the V | dO tiles they read.
      constexpr int TW = kBwdTailWarps, UPW = (kTailKpl + TW - 1) / TW;
      const int half = warp - 9;
      float* red = tail_red + half * (32 * 17);      // [32 lanes][16 columns + 1]: acc1 and acc2 go through it in turn
      const int kpl = (Rk + 31) >> 5;
      mbar_wait(&bars[BAR_KQ], 0);
      mbar_wait(&bars[BAR_VDO], 0);
      for (int r = Nm; r < N; ++r) {
        float sx[UPW], sy[UPW];
#pragma unroll
        for (int u = 0; u < UPW; ++u) { sx[u] = 0.f; sy[u] = 0.f; }
#pragma unroll 1
        for (int a = 0; a < KS; ++a) {
          float f1[16], f2[16];
          lds_row16(k_addr, Rk, a, r, f1);
          lds_row16(v_addr, Rk, a, r, f2);
#pragma unroll
          for (int u = 0; u < UPW; ++u) {
            const int i = lane + 32 * (TW * u + half);
            if (TW * u + half < kpl && i < Rk) {
              float g1[16], g2[16];
              lds_row16(q_addr, Rk, a, i, g1);
              lds_row16(do_addr, Rk, a, i, g2);
              float ax = sx[u], ay = sy[u];
#pragma unroll
              for (int c = 0; c < 16; ++c) { ax = fmaf(f1[c], g1[c], ax); ay = fmaf(f2[c], g2[c], ay); }
              sx[u] = ax; sy[u] = ay;
            }
          }
        }
        // sx = k_r . q_i, sy = v_r . dO_i  ->  sx = P[i, r], sy = dS[i, r] (rounded to bf16 like the tensor path's operands)
#pragma unroll
        for (int u = 0; u < UPW; ++u) {
          const int i = lane + 32 * (TW * u + half);
          float pv = 0.f, dv = 0.f;
          if (TW * u + half < kpl && i < N) {
            pv = exp2f(fmaf(sx[u], scale_log2, -lse_s[i]));
            dv = pv * (sy[u] - del_s[i]);
          }
          sx[u] = __bfloat162float(__float2bfloat16(pv));
          sy[u] = __bfloat162float(__float2bfloat16(dv));
          if (TW * u + half < kpl && i < Rk) ds_mine[static_cast<long>(r) * ldS + i] = __float2bfloat16(dv);
        }
#pragma unroll 1
        for (int a = 0; a < KS; ++a) {
          float acc1[16], acc2[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) { acc1[c] = 0.f; acc2[c] = 0.f; }
#pragma unroll
          for (int u = 0; u < UPW; ++u) {
            const int i = lane + 32 * (TW * u + half);
            if (TW * u + half < kpl && i < Rk) {
              float g1[16], g2[16];
              lds_row16(q_addr, Rk, a, i, g1);
              lds_row16(do_addr, Rk, a, i, g2);
#pragma unroll
              for (int c = 0; c < 16; ++c) { acc2[c] = fmaf(sy[u], g1[c], acc2[c]); acc1[c] = fmaf(sx[u], g2[c], acc1[c]); }
            }
          }
          // column sums over the 32 lanes: lane l adds rows (l >> 4), (l >> 4) + 2, .. of column l & 15, one shuffle joins
          // the two row halves
          float tot1, tot2;
#pragma unroll
          for (int c = 0; c < 16; ++c) red[lane * 17 + c] = acc1[c];
          __syncwarp();
          {
            float t0 = 0.f;
#pragma unroll
            for (int u = 0; u < 16; ++u) t0 += red[(2 * u + (lane >> 4)) * 17 + (lane & 15)];
            tot1 = t0 + __shfl_xor_sync(0xffffffffu, t0, 16);
          }
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 16; ++c) red[lane * 17 + c] = acc2[c];
          __syncwarp();
          {
            float t0 = 0.f;
#pragma unroll
            for (int u = 0; u < 16; ++u) t0 += red[(2 * u + (lane >> 4)) * 17 + (lane & 15)];
            tot2 = t0 + __shfl_xor_sync(0xffffffffu, t0, 16);
          }
          tail_xch[(half * 8 + a) * 32 + lane] = lane < 16 ? tot1 : tot2;     // lanes 0..15: dV column, lanes 16..31: dK column
          __syncwarp();
        }
        named_bar_sync(6, 32 * TW);
        if (half == 0) {
          __nv_bfloat16* drow = drows + static_cast<long>(r) * ld3;
          for (int a = 0; a < KS; ++a) {
            float tot = 0.f;
#pragma unroll
            for (int w = 0; w < TW; ++w) tot += tail_xch[(w * 8 + a) * 32 + lane];
            const int jc = a * 16 + (lane & 15);
            int base, smul;
            qkv_col(m, h, jc & ~1, base, smul);
            base += jc & 1;
            if (lane >= 16) drow[base + smul] = __float2bfloat16(tot * scale);
            else drow[base + 2 * smul] = __float2bfloat16(tot);
          }
        }
        named_bar_sync(6, 32 * TW);
      }
      if (half == 0) {
        // key rows [N, Rk) of the scratch: nobody computes them, the dQ contraction reads them (times zero rows of K)
        for (int r = N; r < Rk; ++r)
          for (int i = lane; i < Rk; i += 32) ds_mine[static_cast<long>(r) * ldS + i] = __float2bfloat16(0.f);
      }
      __threadfence();
      fence_proxy_async_all();
      mbar_arrive(&bars[BAR_DS]);
      mbar_arrive(&bars[BAR_TAIL]);      // this warp no longer reads the Q / K / V / dO tiles
    } else if (n_tail > 0 && warp <= 10) {
      const bool as_key = warp == 9;
      float* red = tail_red + (warp - 9) * (32 * 33);
      const int kpl = (Rk + 31) >> 5;
      mbar_wait(&bars[BAR_KQ], 0);
      mbar_wait(&bars[BAR_VDO], 0);
      // as key:   fixed row r of K / V, lanes run over rows of Q / dO;   as query: fixed row r of Q / dO, lanes over K / V
      const uint32_t fix1 = as_key ? k_addr : q_addr, fix2 = as_key ? v_addr : do_addr;
      const uint32_t run1 = as_key ? q_addr : k_addr, run2 = as_key ? do_addr : v_addr;
      for (int r = Nm; r < N; ++r) {
        float sx[kTailKpl], sy[kTailKpl];
#pragma unroll
        for (int u = 0; u < kTailKpl; ++u) { sx[u] = 0.f; sy[u] = 0.f; }
#pragma unroll 1
        for (int a = 0; a < KS; ++a) {
          float f1[16], f2[16];
          lds_row16(fix1, Rk, a, r, f1);
          lds_row16(fix2, Rk, a, r, f2);
#pragma unroll
          for (int u = 0; u < kTailKpl; ++u) {
            const int i = lane + 32 * u;
            if (u < kpl && i < Rk) {
              float g1[16], g2[16];
              lds_row16(run1, Rk, a, i, g1);
              lds_row16(run2, Rk, a, i, g2);
              float ax = sx[u], ay = sy[u];
#pragma unroll
              for (int c = 0; c < 16; ++c) { ax = fmaf(f1[c], g1[c], ax); ay = fmaf(f2[c], g2[c], ay); }
              sx[u] = ax; sy[u] = ay;
            }
          }
        }
        // sx = q.k, sy = dO.v  ->  sx = P, sy = dS
        const float lse_r = lse_s[r], del_r = del_s[r];
#pragma unroll
        for (int u = 0; u < kTailKpl; ++u) {
          const int i = lane + 32 * u;
          float pv = 0.f, dv = 0.f;
          if (u < kpl && i < N) {
            const float ls = as_key ? lse_s[i] : lse_r, dl = as_key ? del_s[i] : del_r;
            pv = exp2f(fmaf(sx[u], scale_log2, -ls));
            dv = pv * (sy[u] - dl);
          }
          sx[u] = __bfloat162float(__float2bfloat16(pv));
          sy[u] = __bfloat162float(__float2bfloat16(dv));
        }
        __nv_bfloat16* drow = drows + static_cast<long>(r) * ld3;
#pragma unroll 1
        for (int a = 0; a < KS; ++a) {
          // as key:   acc1 = sum_i P_i dO_i (dV), acc2 = sum_i dS_i q_i (dK);   as query: acc2 = sum_j dS_j k_j (dQ)
          float acc1[16], acc2[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) { acc1[c] = 0.f; acc2[c] = 0.f; }
#pragma unroll
          for (int u = 0; u < kTailKpl; ++u) {
            const int i = lane + 32 * u;
            if (u < kpl && i < Rk) {
              float g1[16];
              lds_row16(run1, Rk, a, i, g1);
#pragma unroll
              for (int c = 0; c < 16; ++c) acc2[c] = fmaf(sy[u], g1[c], acc2[c]);
              if (as_key) {
                float g2[16];
                lds_row16(run2, Rk, a, i, g2);
#pragma unroll
                for (int c = 0; c < 16; ++c) acc1[c] = fmaf(sx[u], g2[c], acc1[c]);
              }
            }
          }
#pragma unroll
          for (int c = 0; c < 16; ++c) { red[lane * 33 + c] = acc1[c]; red[lane * 33 + 16 + c] = acc2[c]; }
          __syncwarp();
          float t0 = 0.f, t1 = 0.f;
#pragma unroll
          for (int u = 0; u < 32; u += 2) { t0 += red[u * 33 + lane]; t1 += red[(u + 1) * 33 + lane]; }
          const float tot = t0 + t1;
          // lanes 0..15: acc1 column (dV), lanes 16..31: acc2 column (dK or dQ, scaled by 1/sqrt(hd))
          const int jc = a * 16 + (lane & 15);
          int base, smul;
          qkv_col(m, h, jc & ~1, base, smul);
          base += jc & 1;
          if (lane >= 16) drow[base + (as_key ? 1 : 0) * smul] = __float2bfloat16(tot * scale);
          else if (as_key) drow[base + 2 * smul] = __float2bfloat16(tot);
          __syncwarp();
        }
      }
    }
  } else if (warp == 8) {
    // ------------------------------------------------ control warp ------------------------------------------------
    // The whole warp runs the loops (so addresses and descriptors stay warp-uniform); lane 0 issues TMA / MMA / commit.
    const bool leader = lane == 0;
    OCTIC_TRACE_DECL;
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    // (the operand loads were issued by this warp's lane 0 in the prologue)
    // low descriptor words: K-major views (first level) and MN-major views (second level, LBO = atom-column stride)
    const uint32_t mstep = static_cast<uint32_t>(Rk * 32) >> 4;       // one K-step = next atom column
    const uint32_t qk = desc_lo_sw32(q_addr, 0), kk_ = desc_lo_sw32(k_addr, 0), vk = desc_lo_sw32(v_addr, 0),
                   dok = desc_lo_sw32(do_addr, 0);
    const uint32_t qm = desc_lo_sw32(q_addr, Rk * 32), km = desc_lo_sw32(k_addr, Rk * 32), dom = desc_lo_sw32(do_addr, Rk * 32);
    const uint32_t idesc_l2 = make_idesc_bf16(128, HD, 0, 1);

    // first level of job g: X = A1[tile rows] B1[chunk rows]^T -> buffer, Y = A2[tile rows] B2[chunk rows]^T -> +CW
    //   phase 0: lanes = keys,    X = S^T = K Q^T,  Y = dP^T = V dO^T
    //   phase 1: lanes = queries, X = S   = Q K^T,  Y = dP   = dO V^T
    auto issue_l1 = [&](int g) {
      const int phase = g >= jobs_per_phase, r = g - phase * jobs_per_phase, t = r / nc, c = r - t * nc, buf = g & 1;
      const uint32_t a1 = (phase == 0 ? kk_ : qk) + t * 256, b1 = (phase == 0 ? qk : kk_) + cp.off[c] * 2;
      const uint32_t a2 = (phase == 0 ? vk : dok) + t * 256, b2 = (phase == 0 ? dok : vk) + cp.off[c] * 2;
      const uint32_t idesc = make_idesc_bf16(128, cp.w[c], 0, 0);
      const uint32_t d = tb + buf * 2 * CW;
      if (elect_one()) {
        // the K-steps of X and Y alternate: consecutive MMAs into the SAME accumulator serialise on its latency (an
        // N = 80 MMA is ~40 cycles of work), two independent accumulation chains keep the pipe busy
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
          umma_ss_lohi(d, a1 + ks * mstep, b1 + ks * mstep, kDescHiSw32, idesc, ks != 0);
          umma_ss_lohi(d + CW, a2 + ks * mstep, b2 + ks * mstep, kDescHiSw32, idesc, ks != 0);
        }
        umma_commit(&bars[BAR_LFULL + buf]);
      }
    };
    // second level: acc (+)= (bf16 in TMEM at a_col) * B[chunk rows] (MN-major)
    // The bf16 A operand of K-step kk (written by the math warps): the first half of the pieces (warp set 0) sits at
    // columns kk * 8, the second half (warp set 1) at the start of that set's own column range, h * 16 + (kk - h) * 8.
    auto issue_l2 = [&](uint32_t acc_col, uint32_t a_col, uint32_t bm, int c, bool first) {
      const int nk = cp.w[c] >> 4, hsplit = (nk + 1) >> 1;
      const uint32_t bb = bm + cp.off[c] * 2;
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < CW / 16; ++kk)
          if (kk < nk) {
            const uint32_t ak = kk < hsplit ? kk * 8 : hsplit * 16 + (kk - hsplit) * 8;
            umma_ts_lohi(tb + acc_col, tb + a_col + ak, bb + kk * 32, kDescHiSw32, idesc_l2, !(first && kk == 0));
          }
      }
    };

    // phase 0: dV += P^T dO and dK += dS^T Q as two interleaved accumulation chains
    auto issue_l2_pair = [&](uint32_t acc0, uint32_t a_col0, uint32_t bm0, uint32_t acc1, uint32_t a_col1, uint32_t bm1, int c,
                             bool first) {
      const int nk = cp.w[c] >> 4, hsplit = (nk + 1) >> 1;
      const uint32_t bb0 = bm0 + cp.off[c] * 2, bb1 = bm1 + cp.off[c] * 2;
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < CW / 16; ++kk)
          if (kk < nk) {
            const uint32_t ak = kk < hsplit ? kk * 8 : hsplit * 16 + (kk - hsplit) * 8;
            umma_ts_lohi(tb + acc0, tb + a_col0 + ak, bb0 + kk * 32, kDescHiSw32, idesc_l2, !(first && kk == 0));
            umma_ts_lohi(tb + acc1, tb + a_col1 + ak, bb1 + kk * 32, kDescHiSw32, idesc_l2, !(first && kk == 0));
          }
      }
    };

    mbar_wait(&bars[BAR_KQ], 0);
    mbar_wait(&bars[BAR_VDO], 0);
    tc_fence_after();
    issue_l1(0);
    if (G > 1) issue_l1(1);
    uint32_t phd0 = 0u, phd1 = 0u;
    for (int g = 0; g < G; ++g) {
      const int phase = g >= jobs_per_phase, r = g - phase * jobs_per_phase, c = r % nc, buf = g & 1;
      if (buf == 0) { mbar_wait(&bars[BAR_MDONE], phd0); phd0 ^= 1u; }
      else { mbar_wait(&bars[BAR_MDONE + 1], phd1); phd1 ^= 1u; }
      tc_fence_after();
      if (leader) OCTIC_TRACE(0, 1);
      const uint32_t xcol = buf * 2 * CW, ycol = xcol + CW;
      if (phase == 0) {
        issue_l2_pair(ACC + HD, xcol, dom, ACC, ycol, qm, c, c == 0);    // dV += P^T dO, dK += dS^T Q
      } else {
        issue_l2(ACC, ycol, km, c, c == 0);          // dQ += dS K
      }
      if (c == nc - 1 && elect_one()) umma_commit(&bars[BAR_ACC]);
      if (g + 2 < G) issue_l1(g + 2);
      if (leader) OCTIC_TRACE(0, 2);
    }
    if (staged) {
      // ---- phase 1': dQ_tile = dS[tile queries, keys] K with dS^T streamed back from the L2 scratch ----
      // The V | dO tiles (contiguous, >= Rk * 256 bytes for hd >= 64) receive the operand: every MMA that read them has
      // completed (last BAR_ACC) and the tail warps are done with them (BAR_TAIL).
      mbar_wait(&bars[BAR_ACC], static_cast<uint32_t>((nt - 1) & 1));
      mbar_wait(&bars[BAR_DS], 0);
      if (n_tail > 0) mbar_wait(&bars[BAR_TAIL], 0);
      tc_fence_after();
      // operand tile: [Rk keys][128 queries] bf16 as two SWIZZLE_128B atom columns of 64 queries (Rk x 128 B each), used
      // MN-major (M = queries): LBO = atom-column stride, SBO = 8 key rows, one K-step = 16 key rows = 2048 B
      const uint64_t a_ds = make_smem_desc(v_addr, static_cast<uint32_t>(Rk) * 128u, 1024);
      const uint32_t idesc_q = make_idesc_bf16(128, HD, 1, 1);
      const int nks = Rk >> 4, ntq = (N + 127) >> 7;
      for (int t = 0; t < ntq; ++t) {
        const int ab = t & 1;
        if (t >= 1) mbar_wait(&bars[BAR_DQ + ((t - 1) & 1)], static_cast<uint32_t>(((t - 1) >> 1) & 1));   // operand tile free
        if (t >= 2) mbar_wait(&bars[BAR_DQFREE + ab], static_cast<uint32_t>(((t >> 1) - 1) & 1));          // accumulator drained
        const int natom = (N - t * 128) > 64 ? 2 : 1;        // a last tile of <= 64 queries needs one atom column only
        if (leader) {
          OCTIC_TRACE(0, 8);
          mbar_arrive_expect_tx(&bars[BAR_DSLOAD], static_cast<uint32_t>(natom * Rk) * 128u);
          for (int a = 0; a < natom; ++a)
            for (int r = 0; r < Rk; r += ds_box_rows)
              tma_load_3d(v_addr + a * (Rk * 128) + r * 128, &tmDS, &bars[BAR_DSLOAD], t * 128 + 64 * a, r, slot);
        }
        mbar_wait(&bars[BAR_DSLOAD], static_cast<uint32_t>(t & 1));
        tc_fence_after();
        if (leader) OCTIC_TRACE(0, 9);
        if (elect_one()) {
          for (int ks = 0; ks < nks; ++ks)
            umma_bf16(tb + ab * HD, a_ds + 128u * ks, desc_sw32_mn(k_addr, Rk, 16 * ks), idesc_q, ks != 0);
          umma_commit(&bars[BAR_DQ + ab]);
        }
        __syncwarp();
      }
      if (leader) {
        // every TMA read of the slot has landed: hand it to the next CTA
        __threadfence();
        atomicExch(&ds_slots[slot], 0);
      }
    }
  } else {
    // -------------------------------------------------- math warps --------------------------------------------------
    // Warp (q4, bsel) works on TMEM lane quarter q4 of EVERY job: set bsel = 0 takes the first half of the job's
    // 16-column pieces, set 1 the second half, so a job's math latency is half of what one warp per job gives and the
    // dependent chain math(g) -> second-level MMAs(g) + first-level MMAs(g+2) -> math(g+2) shortens accordingly (the
    // other buffer's job g+1 fills the tensor pipe meanwhile).  Each set streams its pieces (load of piece p+1 in flight
    // while piece p is computed) and writes the bf16 outputs at the start of ITS OWN column range: output piece q lands
    // on columns of the set's input piece q/2, which it has already consumed -- no barrier between the sets.
    // For the accumulator flush (once per tile) the pair splits the columns (hh = bsel).
    const int q4 = warp & 3, bsel = warp >> 2, hh = bsel;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    uint8_t* my_stg = stg + (q4 * 32 + lane) * (HD * 2);
    const uint32_t lse_sa = smem_u32(lse_s), del_sa = smem_u32(del_s);
    OCTIC_TRACE_DECL;
    uint32_t pha = 0u;
    int g = 0;
    const int nphase = staged ? 1 : 2;
    for (int phase = 0; phase < nphase; ++phase) {
      for (int t = 0; t < nt; ++t) {
        const int row0 = t * 128;
        const int my_row = row0 + q4 * 32 + lane;
        __nv_bfloat16* ds_row = staged ? ds_mine + static_cast<long>(my_row) * ldS : nullptr;
        const bool ds_store = staged && my_row < Rk;
        const bool ds_zero = my_row >= N;
        const bool warp_valid = row0 + q4 * 32 < Nm;
        float lse_r = 0.f, del_r = 0.f;
        if (phase == 1) {
          lse_r = my_row < Rk ? lse_s[my_row] : INFINITY;
          del_r = my_row < Rk ? del_s[my_row] : 0.f;
        }
        for (int c = 0; c < nc; ++c, ++g) {
          const int buf = g & 1;
          const uint32_t tx = t_lane + buf * 2 * CW, ty = tx + CW;
          mbar_wait(&bars[BAR_LFULL + buf], (g >> 1) & 1);
          tc_fence_after();
          if (tid == 0) OCTIC_TRACE(1, 3);
          if (warp_valid) {
            const int w = cp.w[c], k0 = cp.off[c];
            const int np = w >> 4, hsplit = (np + 1) >> 1;
            const int p0 = bsel ? hsplit : 0, cnt = bsel ? np - hsplit : hsplit;     // this set's pieces [p0, p0 + cnt)
            const uint32_t ix = tx + p0 * 16, iy = ty + p0 * 16;                      // inputs / outputs of the set start here
            // three register sets: the loads of pieces q+1 and q+2 are in flight while piece q is computed (a TMEM
            // round trip costs ~300 cycles, a piece of math ~150)
            uint32_t rx[3][16], ry[3][16];
            if (0 < cnt) {
              tmem_ld_32x16(ix, rx[0]);
              tmem_ld_32x16(iy, ry[0]);
            }
            if (1 < cnt) {
              tmem_ld_32x16(ix + 16, rx[1]);
              tmem_ld_32x16(iy + 16, ry[1]);
            }
#pragma unroll
            for (int q = 0; q < (CW / 16 + 1) / 2; ++q) {
              if (q < cnt) {
                // wait::ld retires every outstanding load, so piece q+1 is complete too; keep two loads in flight by
                // issuing piece q+2 right away
                tmem_ld_wait();
                if (q + 2 < cnt) {
                  tmem_ld_32x16(ix + (q + 2) * 16, rx[(q + 2) % 3]);
                  tmem_ld_32x16(iy + (q + 2) * 16, ry[(q + 2) % 3]);
                }
                const int col0 = k0 + (p0 + q) * 16;
                uint32_t pkp[8], pkd[8];
                if (phase == 0) {
                  // padded query columns carry lse = +inf (p = 0) and delta = 0: no explicit mask
                  bwd_piece<true>(rx[q % 3], ry[q % 3], pkp, pkd, scale_log2, lse_sa + col0 * 4, del_sa + col0 * 4, 0.f, 0.f, 16);
                  tmem_st_32x8(ix + q * 8, pkp);
                  if (ds_store) {
                    uint4 v0 = make_uint4(pkd[0], pkd[1], pkd[2], pkd[3]), v1 = make_uint4(pkd[4], pkd[5], pkd[6], pkd[7]);
                    if (ds_zero) { v0 = make_uint4(0u, 0u, 0u, 0u); v1 = v0; }
                    uint4* dst = reinterpret_cast<uint4*>(ds_row + col0);
                    dst[0] = v0; dst[1] = v1;
                  }
                } else {
                  bwd_piece<false>(rx[q % 3], ry[q % 3], pkp, pkd, scale_log2, 0u, 0u, lse_r, del_r, N - col0);
                }
                tmem_st_32x8(iy + q * 8, pkd);
              }
            }
            tmem_st_wait();
          }
          tc_fence_before();
          if (tid == 0) OCTIC_TRACE(1, 5);
          mbar_arrive(&bars[BAR_MDONE + buf]);
        }
        if (staged && t == nt - 1) {
          // this thread's part of dS^T is written: make it visible to the TMA (async proxy) reads of phase 1'
          __threadfence();
          fence_proxy_async_all();
          mbar_arrive(&bars[BAR_DS]);
        }
        // ---- flush the accumulators of this tile: TMEM -> bf16 staging -> packed global rows ----
        mbar_wait(&bars[BAR_ACC], pha);
        pha ^= 1u;
        tc_fence_after();
        if (tid == 0) OCTIC_TRACE(1, 6);
        named_bar_sync(5, kBwdMathThreads);          // the previous flush's global stores have read the staging tiles
        if (tid == 0) OCTIC_TRACE(1, 10);
        if (warp_valid) {
          acc_half_to_stg<KS>(t_lane + ACC, hh, scale, my_stg);                               // dK or dQ
          if (phase == 0) acc_half_to_stg<KS>(t_lane + ACC + HD, hh, 1.0f, my_stg + stg_bytes);   // dV
        }
        tc_fence_before();
        if (tid == 0) OCTIC_TRACE(1, 11);
        named_bar_sync(5, kBwdMathThreads);
        if (tid == 0) OCTIC_TRACE(1, 12);
        const int nvalid = min(128, Nm - row0);
        store_tile<HD, GRAN>(stg, drows + static_cast<long>(row0) * ld3, ld3, nvalid, cb, sm, phase == 0 ? 1 : 0, tid,
                             kBwdMathThreads);
        if (phase == 0)
          store_tile<HD, GRAN>(stg + stg_bytes, drows + static_cast<long>(row0) * ld3, ld3, nvalid, cb, sm, 2, tid,
                               kBwdMathThreads);
        if (tid == 0) OCTIC_TRACE(1, 7);
      }
    }
    if (staged) {
      // ---- phase 1': drain dQ of every query tile (accumulators ping-pong in the columns the S / dP buffers used) ----
      // The tiles cover ALL N queries here (a tail token is one more, nearly empty, tile: its cost is one operand load
      // and Rk/16 MMAs, not a pass of jobs), rows past N hold garbage and are not stored.
      const int ntq = (N + 127) >> 7;
      for (int t = 0; t < ntq; ++t) {
        const int row0 = t * 128, ab = t & 1;
        const bool warp_valid = row0 + q4 * 32 < N;
        mbar_wait(&bars[BAR_DQ + ab], static_cast<uint32_t>((t >> 1) & 1));
        tc_fence_after();
        if (tid == 0) OCTIC_TRACE(1, 6);
        named_bar_sync(5, kBwdMathThreads);          // the previous flush's global stores have read the staging tile
        if (tid == 0) OCTIC_TRACE(1, 10);
        if (warp_valid) acc_half_to_stg<KS>(t_lane + ab * HD, hh, scale, my_stg);
        tc_fence_before();
        if (tid == 0) OCTIC_TRACE(1, 11);
        named_bar_sync(5, kBwdMathThreads);
        if (tid == 0) OCTIC_TRACE(1, 12);
        if (ntq > 2) mbar_arrive(&bars[BAR_DQFREE + ab]);
        store_tile<HD, GRAN>(stg, drows + static_cast<long>(row0) * ld3, ld3, min(128, N - row0), cb, sm, 0, tid,
                             kBwdMathThreads);
        if (tid == 0) OCTIC_TRACE(1, 7);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =====================================================================================================================
//  streamed kernels: sequences too long for the resident kernels above
// =====================================================================================================================
// One CTA owns a 128-row tile of one (image, head) and streams 64-row chunks of the other side through a TMA ring, so
// nothing in shared memory grows with N.  One template, three modes:
//   kStreamFwd    tile = queries, chunks = K | V:   X = S = Q K^T -> P (bf16, in place) -> O += P V
//   kStreamBwdKV  tile = keys,    chunks = Q | dO:  X = S^T = K Q^T, Y = dP^T = V dO^T -> P^T, dS^T (bf16, in place)
//                                                   -> dV += P^T dO, dK += dS^T Q
//   kStreamBwdQ   tile = queries, chunks = K | V:   X = S = Q K^T, Y = dP = dO V^T -> dS (bf16, in place) -> dQ += dS K
// The backward runs the key-major and the query-major kernel one after the other: dQ is recomputed from S and dP
// instead of reduced across key tiles, so it needs no workspace sized by B * H * N and no atomics (deterministic).
// Warp roles: warps 0-3 do the math (thread = TMEM lane = tile row), warp 4 issues every tcgen05.mma, warp 5 every
// chunk load.  X / Y live in two ping-pong TMEM buffers: the first-level MMAs of chunk c + 2 are issued right after the
// second-level MMAs of chunk c (same buffer; tcgen05.mma of one thread run in issue order), while the math warps work
// on chunk c + 1.  Operand tiles use the SWIZZLE_32B atom-column format of the resident kernels.
enum { kStreamFwd = 0, kStreamBwdKV = 1, kStreamBwdQ = 2 };
constexpr int kStreamCW = 64;                         // rows per streamed chunk (= TMA box rows)
constexpr int kStreamStages = 3;
constexpr int kStreamMath = 128;
constexpr int kStreamThreads = kStreamMath + 64;

template <int HD, int GRAN, int MODE>
__global__ void __launch_bounds__(kStreamThreads, 1) attn_stream_tc_kernel(const __grid_constant__ CUtensorMap tmQKV,
                                                                           const __grid_constant__ CUtensorMap tmDO,
                                                                           __nv_bfloat16* __restrict__ out,
                                                                           const float* __restrict__ lse_in,
                                                                           float* __restrict__ lse_out,
                                                                           const float* __restrict__ delta, int N, int H,
                                                                           HeadMap m, float scale, float scale_log2) {
  constexpr bool HAS_Y = MODE != kStreamFwd;          // second first-level product (dP / dP^T)
  constexpr bool X_CHAIN = MODE != kStreamBwdQ;       // second level with the bf16 X as A operand (O or dV)
  constexpr int KS = HD / 16, CW = kStreamCW, NP = CW / 16, NS = kStreamStages, NU = HD / (GRAN / 2);
  constexpr int XS = HAS_Y ? 2 * CW : CW;             // TMEM columns of one ping-pong buffer (X, then Y)
  constexpr int ACC = 2 * XS;                         // first accumulator column
  constexpr int NRES = MODE == kStreamFwd ? 1 : 2;    // resident 128-row tiles
  constexpr uint32_t kTmemCols = ACC + (MODE == kStreamBwdKV ? 2 : 1) * HD <= 256 ? 256 : 512;
  constexpr uint32_t tile_bytes = 128 * HD * 2, chunk_bytes = CW * HD * 2;
  enum { BAR_RES = 0, BAR_FULL = 1, BAR_EMPTY = BAR_FULL + NS, BAR_LFULL = BAR_EMPTY + NS, BAR_MDONE = BAR_LFULL + 2,
         BAR_OFULL = BAR_MDONE + 2, BAR_ACC = BAR_OFULL + 1, NBARS = BAR_ACC + 1 };
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int nt = (N + 127) >> 7, nc = (N + CW - 1) / CW;
  const int tile = blockIdx.x % nt, bh = blockIdx.x / nt, b = bh / H, h = bh - b * H, row0 = tile * 128;
  const int npad = MODE == kStreamBwdKV ? nc * CW : 0;
  uint8_t* A1 = smem;
  uint8_t* A2 = A1 + (NRES - 1) * tile_bytes;
  uint8_t* stages = A1 + NRES * tile_bytes;           // stage s: B1 chunk, then B2 chunk
  float* lse_s = reinterpret_cast<float*>(stages + NS * 2 * chunk_bytes);   // key-major: per query column, log2 units
  float* del_s = lse_s + npad;
  int* cb = reinterpret_cast<int*>(del_s + npad);
  int* sm = cb + NU;
  uint64_t* bars = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(sm + NU) + 7) & ~uintptr_t(7));
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + NBARS);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long ld_out = MODE == kStreamFwd ? m.D : 3L * m.D;
  const long soff = static_cast<long>(bh) * N;        // (b, h) row of lse / delta [B, H, N]

  if (tid < NU) {
    if (MODE == kStreamFwd) {
      cb[tid] = o_col(m, h, tid * (GRAN / 2));
    } else {
      int base, smul;
      qkv_col(m, h, tid * (GRAN / 2), base, smul);
      cb[tid] = base; sm[tid] = smul;
    }
  }
  if (MODE == kStreamBwdKV && tid < kStreamMath) {
    for (int i = tid; i < npad; i += kStreamMath) {
      lse_s[i] = i < N ? lse_in[soff + i] * kLog2e : INFINITY;      // +inf -> P = 0 for padded queries
      del_s[i] = i < N ? delta[soff + i] : 0.f;
    }
  }
  if (tid == kStreamMath) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    mbar_init(&bars[BAR_RES], 1);
    for (int s = 0; s < NS; ++s) { mbar_init(&bars[BAR_FULL + s], 1); mbar_init(&bars[BAR_EMPTY + s], 1); }
    mbar_init(&bars[BAR_LFULL], 1); mbar_init(&bars[BAR_LFULL + 1], 1);
    mbar_init(&bars[BAR_MDONE], kStreamMath); mbar_init(&bars[BAR_MDONE + 1], kStreamMath);
    mbar_init(&bars[BAR_OFULL], 1);
    mbar_init(&bars[BAR_ACC], 1);
    fence_mbar_init();
  }
  if (warp == 4) tmem_alloc(tmem_ptr, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t stages_addr = smem_u32(stages);

  if (warp == 5) {
    // ------------------------------------------------- load warp -------------------------------------------------
    // head-major columns: q at h*HD, k at D + h*HD, v at 2D + h*HD of a qkv row; dO at h*HD of a dO row
    if (lane == 0) {
      const int colq = h * HD, colk = m.D + h * HD, colv = 2 * m.D + h * HD;
      mbar_arrive_expect_tx(&bars[BAR_RES], NRES * tile_bytes);
      if (MODE == kStreamBwdKV) {
        tma_load_tile<HD>(smem_u32(A1), &tmQKV, &bars[BAR_RES], colk, row0, b, 128, CW);
        tma_load_tile<HD>(smem_u32(A2), &tmQKV, &bars[BAR_RES], colv, row0, b, 128, CW);
      } else {
        tma_load_tile<HD>(smem_u32(A1), &tmQKV, &bars[BAR_RES], colq, row0, b, 128, CW);
        if (MODE == kStreamBwdQ) tma_load_tile<HD>(smem_u32(A2), &tmDO, &bars[BAR_RES], colq, row0, b, 128, CW);
      }
      const CUtensorMap* mb2 = MODE == kStreamBwdKV ? &tmDO : &tmQKV;
      const int c1 = MODE == kStreamBwdKV ? colq : colk, c2 = MODE == kStreamBwdKV ? colq : colv;
      for (int c = 0; c < nc; ++c) {
        const int s = c % NS;
        if (c >= NS) mbar_wait(&bars[BAR_EMPTY + s], static_cast<uint32_t>((c / NS - 1) & 1));
        const uint32_t dst = stages_addr + s * 2 * chunk_bytes;
        mbar_arrive_expect_tx(&bars[BAR_FULL + s], 2 * chunk_bytes);
        tma_load_tile<HD>(dst, &tmQKV, &bars[BAR_FULL + s], c1, c * CW, b, CW, CW);
        tma_load_tile<HD>(dst + chunk_bytes, mb2, &bars[BAR_FULL + s], c2, c * CW, b, CW, CW);
      }
    }
    __syncwarp();
  } else if (warp == 4) {
    // -------------------------------------------------- MMA warp --------------------------------------------------
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t a1 = desc_lo_sw32(smem_u32(A1), 0), a2 = desc_lo_sw32(smem_u32(A2), 0);
    constexpr uint32_t a_step = (128 * 32) >> 4, c_step = (CW * 32) >> 4;   // K-step = next atom column
    const uint32_t idesc1 = make_idesc_bf16(128, CW, 0, 0), idesc2 = make_idesc_bf16(128, HD, 0, 1);
    // first level of chunk c: X = A1 B1^T, Y = A2 B2^T (contraction over the head dim, both K-major)
    auto issue_l1 = [&](int c) {
      const int s = c % NS;
      mbar_wait(&bars[BAR_FULL + s], static_cast<uint32_t>((c / NS) & 1));
      tc_fence_after();
      const uint32_t b1 = desc_lo_sw32(stages_addr + s * 2 * chunk_bytes, 0), b2 = b1 + (chunk_bytes >> 4);
      const uint32_t d = tb + (c & 1) * XS;
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
          umma_ss_lohi(d, a1 + ks * a_step, b1 + ks * c_step, kDescHiSw32, idesc1, ks != 0);
          if (HAS_Y) umma_ss_lohi(d + CW, a2 + ks * a_step, b2 + ks * c_step, kDescHiSw32, idesc1, ks != 0);
        }
        umma_commit(&bars[BAR_LFULL + (c & 1)]);
      }
      __syncwarp();
    };
    // second level of chunk c: acc += (bf16 X or Y in TMEM, K-step kk at column kk * 8) * chunk (MN-major, over rows)
    auto issue_l2 = [&](int c) {
      const int s = c % NS;
      const uint32_t xa = tb + (c & 1) * XS, ya = xa + CW;
      const uint32_t b1 = desc_lo_sw32(stages_addr + s * 2 * chunk_bytes, CW * 32), b2 = b1 + (chunk_bytes >> 4);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < NP; ++kk) {
          const uint32_t acc = (c > 0 || kk > 0) ? 1u : 0u;
          if (X_CHAIN)      // O += P V   or   dV += P^T dO
            umma_ts_lohi(tb + ACC + (MODE == kStreamBwdKV ? HD : 0), xa + kk * 8, b2 + kk * 32, kDescHiSw32, idesc2, acc);
          if (HAS_Y)        // dK += dS^T Q   or   dQ += dS K
            umma_ts_lohi(tb + ACC, ya + kk * 8, b1 + kk * 32, kDescHiSw32, idesc2, acc);
        }
        umma_commit(&bars[BAR_EMPTY + s]);
        if (MODE == kStreamFwd) umma_commit(&bars[BAR_OFULL]);
        if (c == nc - 1) umma_commit(&bars[BAR_ACC]);
      }
      __syncwarp();
    };
    mbar_wait(&bars[BAR_RES], 0);
    tc_fence_after();
    issue_l1(0);
    if (nc > 1) issue_l1(1);
    for (int c = 0; c < nc; ++c) {
      mbar_wait(&bars[BAR_MDONE + (c & 1)], static_cast<uint32_t>((c >> 1) & 1));
      tc_fence_after();
      issue_l2(c);
      if (c + 2 < nc) issue_l1(c + 2);
    }
  } else {
    // ------------------------------------------------- math warps -------------------------------------------------
    const int rloc = tid, my_row = row0 + rloc;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const uint32_t lse_sa = smem_u32(lse_s), del_sa = smem_u32(del_s);
    float lse_r = INFINITY, del_r = 0.f;                // query-major backward: this row's lse (log2 units) and delta
    if (MODE == kStreamBwdQ && my_row < N) { lse_r = lse_in[soff + my_row] * kLog2e; del_r = delta[soff + my_row]; }
    // forward: the row's reference maximum, raised lazily as in attn_fwd_tc_kernel (p <= 2^8 between raises)
    const float lazy_gap = 8.0f / scale_log2;
    float mx = -INFINITY, moff = 0.f, l = 0.f;
    for (int c = 0; c < nc; ++c) {
      const int buf = c & 1, k0 = c * CW;
      mbar_wait(&bars[BAR_LFULL + buf], static_cast<uint32_t>((c >> 1) & 1));
      tc_fence_after();
      const uint32_t tx = t_lane + buf * XS, ty = tx + CW;
      if (MODE == kStreamFwd) {
        uint32_t r[NP][16];
#pragma unroll
        for (int q = 0; q < NP; ++q) tmem_ld_32x16(tx + q * 16, r[q]);
        tmem_ld_wait();
        float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
        for (int q = 0; q < NP; ++q) {
          const int nvalid = N - (k0 + q * 16);
          if (nvalid < 16) {
#pragma unroll
            for (int i = 0; i < 16; ++i) r[q][i] = i < nvalid ? r[q][i] : 0xff800000u;      // -inf
          }
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            m0 = fmaxf(m0, __uint_as_float(r[q][i]));
            m1 = fmaxf(m1, __uint_as_float(r[q][i + 1]));
          }
        }
        const float mc = fmaxf(m0, m1);
        if (c == 0) {
          mx = mc;
          moff = mx * scale_log2;
        } else {
          const bool need = mc > mx + lazy_gap;
          if (__any_sync(0xffffffffu, need)) {
            // O holds the P V sums of chunks < c under the old reference: wait for chunk c - 1's MMAs (chunk c's cannot
            // have been issued), then rescale this row of O and its partial sum
            const float f = need ? exp2f((mx - mc) * scale_log2) : 1.0f;
            mbar_wait(&bars[BAR_OFULL], static_cast<uint32_t>((c - 1) & 1));
            tc_fence_after();
#pragma unroll 1
            for (int pz = 0; pz < KS; ++pz) {
              uint32_t ov[16];
              tmem_ld_32x16(t_lane + ACC + pz * 16, ov);
              tmem_ld_wait();
              uint32_t lo[8], hi[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                lo[i] = __float_as_uint(__uint_as_float(ov[i]) * f);
                hi[i] = __float_as_uint(__uint_as_float(ov[8 + i]) * f);
              }
              tmem_st_32x8(t_lane + ACC + pz * 16, lo);
              tmem_st_32x8(t_lane + ACC + pz * 16 + 8, hi);
            }
            tmem_st_wait();
            l *= f;
            if (need) { mx = mc; moff = mx * scale_log2; }
          }
        }
        float l0 = 0.f, l1 = 0.f;
#pragma unroll
        for (int q = 0; q < NP; ++q) {
          uint32_t pk[8];
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const float e0 = exp2f(fmaf(__uint_as_float(r[q][i]), scale_log2, -moff));       // -inf -> 0
            const float e1 = exp2f(fmaf(__uint_as_float(r[q][i + 1]), scale_log2, -moff));
            l0 += e0; l1 += e1;
            pk[i >> 1] = pack2_bf16(e0, e1);
          }
          tmem_st_32x8(tx + q * 8, pk);       // bf16 P of piece q over columns of piece q / 2, already in registers
        }
        l += l0 + l1;
      } else {
        uint32_t rx[NP][16], ry[NP][16];
#pragma unroll
        for (int q = 0; q < NP; ++q) { tmem_ld_32x16(tx + q * 16, rx[q]); tmem_ld_32x16(ty + q * 16, ry[q]); }
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < NP; ++q) {
          const int col0 = k0 + q * 16;
          uint32_t pkp[8], pkd[8];
          if (MODE == kStreamBwdKV) {
            // columns are queries: padded ones carry lse = +inf (p = 0) and delta = 0
            bwd_piece<true>(rx[q], ry[q], pkp, pkd, scale_log2, lse_sa + col0 * 4, del_sa + col0 * 4, 0.f, 0.f, 16);
            tmem_st_32x8(tx + q * 8, pkp);
          } else {
            bwd_piece<false>(rx[q], ry[q], pkp, pkd, scale_log2, 0u, 0u, lse_r, del_r, N - col0);
          }
          tmem_st_32x8(ty + q * 8, pkd);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&bars[BAR_MDONE + buf]);
    }
    // ---- epilogue: accumulators -> bf16 row-major staging over the resident tiles (no MMA reads them any more) ----
    mbar_wait(&bars[BAR_ACC], 0);
    tc_fence_after();
    if (MODE == kStreamFwd) {
      acc_pieces_to_stg<0, KS>(t_lane + ACC, 1.0f / l, A1 + rloc * (HD * 2));
      if (lse_out != nullptr && my_row < N) lse_out[soff + my_row] = (mx * scale_log2 + log2f(l)) * kLn2;
    } else {
      acc_pieces_to_stg<0, KS>(t_lane + ACC, scale, A1 + rloc * (HD * 2));                 // dK or dQ
      if (MODE == kStreamBwdKV) acc_pieces_to_stg<0, KS>(t_lane + ACC + HD, 1.0f, A2 + rloc * (HD * 2));   // dV
    }
    tc_fence_before();
    named_bar_sync(1, kStreamMath);
    const int nvalid = min(128, N - row0);
    __nv_bfloat16* dst = out + (static_cast<long>(b) * N + row0) * ld_out;
    if (MODE == kStreamFwd) {
      store_tile<HD, GRAN>(A1, dst, ld_out, nvalid, cb, nullptr, 0, tid, kStreamMath);
    } else {
      store_tile<HD, GRAN>(A1, dst, ld_out, nvalid, cb, sm, MODE == kStreamBwdKV ? 1 : 0, tid, kStreamMath);
      if (MODE == kStreamBwdKV) store_tile<HD, GRAN>(A2, dst, ld_out, nvalid, cb, sm, 2, tid, kStreamMath);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =====================================================================================================================
//  host
// =====================================================================================================================
constexpr int kMaxSmem = 232448;   // 227 KiB

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn attn_encode_fn() {
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
// bf16 [B][N][cols] (contiguous); box = 16 columns x box_rows rows x 1 image, SWIZZLE_32B, zero fill out of bounds
static int make_map_rows(CUtensorMap* map, const void* base, int B, int N, long cols, int box_rows) {
  EncodeTiledFn enc = attn_encode_fn();
  if (enc == nullptr) return OCTIC_ERR_DRIVER;
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (cols * 2) % 16 != 0) return OCTIC_ERR_ALIGN;
  if (box_rows < 1 || box_rows > 256) return OCTIC_ERR_ARG;
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(B)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(cols) * 2, static_cast<cuuint64_t>(cols) * 2 * static_cast<cuuint64_t>(N)};
  cuuint32_t box[3] = {16, static_cast<cuuint32_t>(box_rows), 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? OCTIC_OK : OCTIC_ERR_TMAP;
}
static int pick_box_rows(int Rk) { return Rk > 256 ? Rk / 2 : Rk; }
// staged-dQ scratch, bf16 [slots][Rk][Rk]: box = 64 columns (128 B) x box_rows rows, SWIZZLE_128B
static int ds_pitch(int Rk) { return Rk; }   // = ldS of the kernel
static int make_map_ds(CUtensorMap* map, const void* base, int slots, int Rk, int box_rows) {
  EncodeTiledFn enc = attn_encode_fn();
  if (enc == nullptr) return OCTIC_ERR_DRIVER;
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || box_rows < 1 || box_rows > 256) return OCTIC_ERR_ARG;
  const cuuint64_t ld = static_cast<cuuint64_t>(ds_pitch(Rk));
  cuuint64_t dims[3] = {ld, static_cast<cuuint64_t>(Rk), static_cast<cuuint64_t>(slots)};
  cuuint64_t strides[2] = {ld * 2, ld * 2 * static_cast<cuuint64_t>(Rk)};
  cuuint32_t box[3] = {64, static_cast<cuuint32_t>(box_rows), 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? OCTIC_OK : OCTIC_ERR_TMAP;
}

static size_t fwd_smem(int Rk, int hd, int gran) {
  const int nu = hd / (gran / 2);
  return static_cast<size_t>(2 * Rk + 128) * hd * 2 + 768 * 4 + (nu + 1) * 4 + 9 * 8 + 16 + 16 + (hd + 32 * 17) * 4 + 1024;
}
static size_t bwd_smem(int Rk, int hd, int gran) {
  const int nu = hd / (gran / 2);
  return static_cast<size_t>(4 * Rk + 256) * hd * 2 + 2 * Rk * 4 + (2 * nu + 1) * 4 + 14 * 8 + 16 + 2 * 32 * 33 * 4 +
         3 * 8 * 32 * 4 + 1024;
}

// ---- staged-dQ workspace: [kDsHeader bytes of slot flags (int, 0 = free)] [n_slots x Rk x ds_pitch(Rk) bf16] ----
constexpr size_t kDsHeader = 4096;
constexpr int kDsMaxSlots = static_cast<int>(kDsHeader / sizeof(int));
static int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n = 0;
  }
  return n;
}
bool attn_tc_supported(int N, int hd, bool backward);
// the operand tile [Rk keys][128 queries] must fit into the V | dO tiles of the backward kernel
static bool ds_staging_applies(int N, int hd) { return hd >= 64 && attn_tc_supported(N, hd, true); }
size_t attn_bwd_tc_workspace_bytes(int N, int hd) {
  if (!ds_staging_applies(N, hd) || sm_count() <= 0) return 0;
  const size_t Rk = static_cast<size_t>((N + 15) / 16 * 16);
  const int slots = 2 * sm_count() < kDsMaxSlots ? 2 * sm_count() : kDsMaxSlots;
  return kDsHeader + static_cast<size_t>(slots) * Rk * ds_pitch(static_cast<int>(Rk)) * 2;
}

bool attn_tc_supported(int N, int hd, bool backward) {
  if (hd != 64 && hd != 80 && hd != 32 && hd != 96 && hd != 128) return false;
  ChunkPlan p;
  if (N < 1 || !make_plan(&p, N, hd)) return false;
  const int Rk = (N + 15) / 16 * 16;
  if (Rk > 512) return false;
  return (backward ? bwd_smem(Rk, hd, 4) : fwd_smem(Rk, hd, 4)) <= static_cast<size_t>(kMaxSmem);
}

static int pick_gran(const HeadMap& m) { return (!m.octic || (m.ch % 8) == 0) ? 16 : 4; }

template <int HD, int GRAN>
static int launch_fwd_t(const void* qkv, void* o, float* lse, int B, int N, int H, const HeadMap& m, const ChunkPlan& cp,
                        cudaStream_t s) {
  const int Rk = (N + 15) / 16 * 16;
  const size_t smem = fwd_smem(Rk, HD, GRAN);
  static bool done = false;
  if (!done) {
    if (cudaFuncSetAttribute(attn_fwd_tc_kernel<HD, GRAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem) != cudaSuccess)
      return OCTIC_ERR_CUDA;
    done = true;
  }
  CUtensorMap tmKV, tmQ;
  const int br = pick_box_rows(Rk);
  int rc = make_map_rows(&tmKV, qkv, B, N, 3L * m.D, br);
  if (rc) return rc;
  rc = make_map_rows(&tmQ, qkv, B, N, 3L * m.D, 128);
  if (rc) return rc;
  const float scale_log2 = kLog2e / sqrtf(static_cast<float>(HD));
  attn_fwd_tc_kernel<HD, GRAN><<<B * H, kFwdThreads, smem, s>>>(tmKV, tmQ, static_cast<__nv_bfloat16*>(o), lse, N, H, m,
                                                                scale_log2, cp, br, static_cast<const __nv_bfloat16*>(qkv),
                                                                attn_tail_rows(N));
  return cudaGetLastError() == cudaSuccess ? OCTIC_OK : OCTIC_ERR_CUDA;
}
template <int HD, int GRAN>
static int launch_bwd_t(const void* qkv, const void* d_o, const float* lse, const float* delta, void* dqkv, int B, int N,
                        int H, const HeadMap& m, const ChunkPlan& cp, void* ws, size_t ws_bytes, cudaStream_t s) {
  const int Rk = (N + 15) / 16 * 16;
  const size_t smem = bwd_smem(Rk, HD, GRAN);
  static bool done = false;
  if (!done) {
    if (cudaFuncSetAttribute(attn_bwd_tc_kernel<HD, GRAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem) != cudaSuccess)
      return OCTIC_ERR_CUDA;
    done = true;
  }
  CUtensorMap tmQKV, tmDO;
  const int br = pick_box_rows(Rk);
  int rc = make_map_rows(&tmQKV, qkv, B, N, 3L * m.D, br);
  if (rc) return rc;
  rc = make_map_rows(&tmDO, d_o, B, N, m.D, br);
  if (rc) return rc;
  // staged dQ when the caller's workspace holds a slot for every CTA that can be resident (one per SM)
  CUtensorMap tmDS = tmDO;
  __nv_bfloat16* ds_ws = nullptr;
  int* ds_slots = nullptr;
  int n_slots = 0, ds_br = br;
  if (ws != nullptr && ws_bytes > kDsHeader && ds_staging_applies(N, HD) && (reinterpret_cast<uintptr_t>(ws) & 255) == 0) {
    const size_t per = static_cast<size_t>(Rk) * ds_pitch(Rk) * 2;
    size_t fit = (ws_bytes - kDsHeader) / per;
    if (fit > static_cast<size_t>(kDsMaxSlots)) fit = kDsMaxSlots;
    if (sm_count() > 0 && fit >= static_cast<size_t>(sm_count())) {
      n_slots = static_cast<int>(fit);
      ds_slots = static_cast<int*>(ws);
      ds_ws = reinterpret_cast<__nv_bfloat16*>(static_cast<uint8_t*>(ws) + kDsHeader);
      static int env_rows = -1;
      if (env_rows < 0) { const char* e = getenv("OCTIC_DS_BOX_ROWS"); env_rows = e ? atoi(e) : 0; }
      if (env_rows > 0 && env_rows <= 256 && Rk % env_rows == 0) ds_br = env_rows;
      rc = make_map_ds(&tmDS, ds_ws, n_slots, Rk, ds_br);
      if (rc) return rc;
    }
  }
  const float scale = 1.0f / sqrtf(static_cast<float>(HD));
  attn_bwd_tc_kernel<HD, GRAN><<<B * H, kBwdThreads, smem, s>>>(tmQKV, tmDO, lse, delta, static_cast<__nv_bfloat16*>(dqkv),
                                                                N, H, m, scale, kLog2e * scale, cp, br, attn_tail_rows(N),
                                                                tmDS, ds_ws, ds_slots, n_slots, ds_br);
  return cudaGetLastError() == cudaSuccess ? OCTIC_OK : OCTIC_ERR_CUDA;
}

#define OCTIC_TC_DISPATCH(FN, ...)                                                     \
  switch (m.hd) {                                                                      \
    case 32: return gran == 16 ? FN<32, 16>(__VA_ARGS__) : FN<32, 4>(__VA_ARGS__);    \
    case 64: return gran == 16 ? FN<64, 16>(__VA_ARGS__) : FN<64, 4>(__VA_ARGS__);    \
    case 80: return gran == 16 ? FN<80, 16>(__VA_ARGS__) : FN<80, 4>(__VA_ARGS__);    \
    case 96: return gran == 16 ? FN<96, 16>(__VA_ARGS__) : FN<96, 4>(__VA_ARGS__);    \
    case 128: return gran == 16 ? FN<128, 16>(__VA_ARGS__) : FN<128, 4>(__VA_ARGS__); \
    default: return OCTIC_ERR_ARG;                                                     \
  }

// m describes the OUTPUT rows (o / dqkv: packed octic or dense); the inputs qkv (and d_o) are head-major.
int launch_attn_fwd_tc(const void* qkv, void* o, float* lse, int B, int N, int H, const HeadMap& m, cudaStream_t s) {
  ChunkPlan cp;
  if (!attn_tc_supported(N, m.hd, false) || !make_plan(&cp, N, m.hd)) return OCTIC_ERR_ARG;
  const int gran = pick_gran(m);
  OCTIC_TC_DISPATCH(launch_fwd_t, qkv, o, lse, B, N, H, m, cp, s)
}

int launch_attn_bwd_tc(const void* qkv, const void* d_o, const float* lse, const float* delta, void* dqkv, int B, int N,
                       int H, const HeadMap& m, void* ws, size_t ws_bytes, cudaStream_t s) {
  ChunkPlan cp;
  if (!attn_tc_supported(N, m.hd, true) || !make_plan(&cp, N, m.hd)) return OCTIC_ERR_ARG;
  const int gran = pick_gran(m);
  OCTIC_TC_DISPATCH(launch_bwd_t, qkv, d_o, lse, delta, dqkv, B, N, H, m, cp, ws, ws_bytes, s)
}


// ---- streamed kernels ----
static size_t stream_smem(int N, int hd, int gran, int mode) {
  const int nu = hd / (gran / 2), nres = mode == kStreamFwd ? 1 : 2;
  const size_t npad = mode == kStreamBwdKV ? static_cast<size_t>((N + kStreamCW - 1) / kStreamCW) * kStreamCW : 0;
  return 1024 + static_cast<size_t>(nres * 128 + kStreamStages * 2 * kStreamCW) * hd * 2 + 2 * npad * 4 + 2 * nu * 4 + 8 +
         (1 + 2 * kStreamStages + 6) * 8 + 16;
}

bool attn_stream_supported(int N, int hd) {
  if (hd != 64 && hd != 80 && hd != 32 && hd != 96 && hd != 128) return false;
  return N >= 1 && stream_smem(N, hd, 4, kStreamBwdKV) <= static_cast<size_t>(kMaxSmem);
}

template <int HD, int GRAN, int MODE>
static int launch_stream_mode(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, void* out, const float* lse_in,
                              float* lse_out, const float* delta, int B, int N, int H, const HeadMap& m, cudaStream_t s) {
  static bool done = false;
  if (!done) {
    if (cudaFuncSetAttribute(attn_stream_tc_kernel<HD, GRAN, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             kMaxSmem) != cudaSuccess)
      return OCTIC_ERR_CUDA;
    done = true;
  }
  const float scale = 1.0f / sqrtf(static_cast<float>(HD));
  const long grid = static_cast<long>(B) * H * ((N + 127) / 128);
  if (grid > 0x7fffffffL) return OCTIC_ERR_ARG;
  attn_stream_tc_kernel<HD, GRAN, MODE><<<static_cast<unsigned>(grid), kStreamThreads, stream_smem(N, HD, GRAN, MODE), s>>>(
      tmQKV, tmDO, static_cast<__nv_bfloat16*>(out), lse_in, lse_out, delta, N, H, m, scale, kLog2e * scale);
  return cudaGetLastError() == cudaSuccess ? OCTIC_OK : OCTIC_ERR_CUDA;
}

template <int HD, int GRAN>
static int launch_stream_fwd_t(const void* qkv, void* o, float* lse, int B, int N, int H, const HeadMap& m, cudaStream_t s) {
  CUtensorMap tmQKV;
  const int rc = make_map_rows(&tmQKV, qkv, B, N, 3L * m.D, kStreamCW);
  if (rc) return rc;
  return launch_stream_mode<HD, GRAN, kStreamFwd>(tmQKV, tmQKV, o, nullptr, lse, nullptr, B, N, H, m, s);
}

template <int HD, int GRAN>
static int launch_stream_bwd_t(const void* qkv, const void* d_o, const float* lse, const float* delta, void* dqkv, int B,
                               int N, int H, const HeadMap& m, cudaStream_t s) {
  CUtensorMap tmQKV, tmDO;
  int rc = make_map_rows(&tmQKV, qkv, B, N, 3L * m.D, kStreamCW);
  if (rc) return rc;
  rc = make_map_rows(&tmDO, d_o, B, N, m.D, kStreamCW);
  if (rc) return rc;
  rc = launch_stream_mode<HD, GRAN, kStreamBwdKV>(tmQKV, tmDO, dqkv, lse, nullptr, delta, B, N, H, m, s);
  if (rc) return rc;
  return launch_stream_mode<HD, GRAN, kStreamBwdQ>(tmQKV, tmDO, dqkv, lse, nullptr, delta, B, N, H, m, s);
}

int launch_attn_fwd_stream(const void* qkv, void* o, float* lse, int B, int N, int H, const HeadMap& m, cudaStream_t s) {
  if (!attn_stream_supported(N, m.hd)) return OCTIC_ERR_ARG;
  const int gran = pick_gran(m);
  OCTIC_TC_DISPATCH(launch_stream_fwd_t, qkv, o, lse, B, N, H, m, s)
}

int launch_attn_bwd_stream(const void* qkv, const void* d_o, const float* lse, const float* delta, void* dqkv, int B,
                           int N, int H, const HeadMap& m, cudaStream_t s) {
  if (!attn_stream_supported(N, m.hd)) return OCTIC_ERR_ARG;
  const int gran = pick_gran(m);
  OCTIC_TC_DISPATCH(launch_stream_bwd_t, qkv, d_o, lse, delta, dqkv, B, N, H, m, s)
}

}  // namespace octic
