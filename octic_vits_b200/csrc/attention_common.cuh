// Shared by the attention kernels (attention.cu: legacy mma.sync path for long sequences; attention_tc.cu: tcgen05
// path): the map from a head vector to columns of the packed qkv / attention-output rows.
// Reference: AttentionD8.forward (octic_vits/d8_layers.py:632-656) -- per head [A1(c_h) | A2 | B1 | B2 | E row0 (2c_h) |
// E row1 (2c_h)]; the dense layout (deit/vit.py:36-50) is [3][H][hd].
#pragma once
#include "octic_capi_internal.h"

namespace octic {

struct HeadMap {
  int octic;   // 1: packed LinearD8 layout, 0: dense [3][H][hd]
  int D;       // embed dim
  int C;       // D / 8
  int ch;      // hd / 8 = C / H
  int hd;
};

// column of element j (even) of the head vector of (s, h) inside a qkv row, split as base + s * smul
__device__ __forceinline__ void qkv_col(const HeadMap& m, int h, int j, int& base, int& smul) {
  if (!m.octic) { base = h * m.hd + j; smul = m.D; return; }
  if (j < 4 * m.ch) {
    const int g = j / m.ch, jj = j - g * m.ch;
    base = g * 3 * m.C + h * m.ch + jj; smul = m.C;
  } else {
    const int j2 = j - 4 * m.ch, r = j2 / (2 * m.ch), jj = j2 - r * 2 * m.ch;
    base = 12 * m.C + r * 6 * m.C + h * 2 * m.ch + jj; smul = 2 * m.C;
  }
}
// column of element j of head h inside an attention-output row (packed 5-tuple order, d8_layers.py:650-656)
__device__ __forceinline__ int o_col(const HeadMap& m, int h, int j) {
  if (!m.octic) return h * m.hd + j;
  if (j < 4 * m.ch) {
    const int g = j / m.ch, jj = j - g * m.ch;
    return g * m.C + h * m.ch + jj;
  }
  const int j2 = j - 4 * m.ch, r = j2 / (2 * m.ch), jj = j2 - r * 2 * m.ch;
  return 4 * m.C + r * 2 * m.C + h * 2 * m.ch + jj;
}


constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// launchers of the tcgen05 path (attention_tc.cu); return OCTIC_ERR_ARG when the shape is outside its envelope
bool attn_tc_supported(int N, int hd, bool backward);
int launch_attn_fwd_tc(const void* qkv, void* o, float* lse, int B, int N, int H, const HeadMap& m, cudaStream_t s);
// ws: optional staged-dQ workspace (attn_bwd_tc_workspace_bytes(N, hd) bytes, 256-byte aligned, slot flags zeroed
// once); nullptr = the two-phase kernel that recomputes S and dP for dQ.
int launch_attn_bwd_tc(const void* qkv, const void* d_o, const float* lse, const float* delta, void* dqkv, int B, int N,
                       int H, const HeadMap& m, void* ws, size_t ws_bytes, cudaStream_t s);
size_t attn_bwd_tc_workspace_bytes(int N, int hd);
// streamed tcgen05 kernels (attention_tc.cu): head-major inputs of any length whose shared-memory needs fit (checked by
// attn_stream_supported); the backward needs no workspace.  delta must already hold rowsum(dO * O).
bool attn_stream_supported(int N, int hd);
int launch_attn_fwd_stream(const void* qkv, void* o, float* lse, int B, int N, int H, const HeadMap& m, cudaStream_t s);
int launch_attn_bwd_stream(const void* qkv, const void* d_o, const float* lse, const float* delta, void* dqkv, int B,
                           int N, int H, const HeadMap& m, cudaStream_t s);

}  // namespace octic
