// Internal declarations shared by the .cu files of liboctic_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string.h>
#include "../../include/octic_b200.h"

namespace octic {

enum { EPI_BF16 = OCTIC_EPI_BF16, EPI_RESID = OCTIC_EPI_RESID, EPI_F32 = OCTIC_EPI_F32, EPI_GELU_BF16 = OCTIC_EPI_GELU_BF16,
       EPI_GELU_BWD = OCTIC_EPI_GELU_BWD };

struct GemmGroup {
  int a_col, k_blocks, b_map, b_row, n, n_tiles, c_col, bias_off, tile_begin, head_off;
};
struct GemmParams {
  int M, num_groups, block_n, tiles_per_m, num_m_blocks, num_stages, mode;
  GemmGroup g[OCTIC_MAX_GROUPS];
  void* out;
  long ldo;
  const float* bias;
  const float* gamma;
  const float* resid_in;
  float* resid_out;
  long ldr;
  const float* row_scale;
  int rows_per_sample;
  void* branch_out;
  long ldb;
  int remap_group, remap_extra, remap_off;
  int head_H, head_S, head_D;
  const void* gelu_pre;
  float* colsum;
  int direct;   // 1: full aligned chunks go registers -> global without the shared-memory transpose
  int ws;       // weight-stationary tile order (CTA pairs, small-K groups): see gemm_tn_kernel
  int ws_kb_max;
  int packed;      // 1: bf16-packed epilogue staging where it applies (gemm_tn_kernel process_packed)
  int roles_low;   // 1: TMA producer / MMA issuer on warps 0 / 1 (round-1 order) instead of the two highest warp ids
};

struct WgradGroup {
  int dy_col, x_col, n_out, k_in, n_tiles, m_tiles, tile_begin;
  float* dw;
  long ldw;
};
struct WgradParams {
  int T, num_groups, block_n, total_tiles, splits, num_stages, rem_splits, roles_low;
  WgradGroup g[OCTIC_MAX_GROUPS];
};

int launch_gemm_tn(const octic_gemm_desc* d, cudaStream_t stream);
int launch_gemm_wgrad(const octic_wgrad_desc* d, cudaStream_t stream);
int gemm_last_plan(octic_gemm_plan* out);

inline int roundup64(int x) { return (x + 63) / 64 * 64; }

// largest multiple of 16 that is <= 256 and divides every n in ns[]; falls back to min(256, roundup16(max n)).
int pick_block_n(const int* ns, int count);

}  // namespace octic
