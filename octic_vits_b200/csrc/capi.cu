// extern "C" entry points of liboctic_b200.so that are thin glue: error strings, device probe, the generic
// grouped GEMM, and the LinearD8 / nn.Linear wrappers that turn reference-level arguments into GEMM groups.
#include "octic_capi_internal.h"
#include <stdlib.h>

namespace octic {

int pick_block_n(const int* ns, int count) {
  int maxn = 0;
  for (int i = 0; i < count; ++i) maxn = ns[i] > maxn ? ns[i] : maxn;
  {
    // OCTIC_BLOCK_N=n forces the N tile of the grouped (LinearD8) launches: tile-shape experiments (ragged last tiles
    // are handled by the kernels)
    static int forced = -1;
    if (forced < 0) {
      const char* e = getenv("OCTIC_BLOCK_N");
      forced = e != nullptr ? atoi(e) : 0;
    }
    if (forced >= 32 && forced <= 256 && forced % 16 == 0) return forced;
  }
  for (int bn = 256; bn >= 16; bn -= 16) {
    bool ok = true;
    for (int i = 0; i < count; ++i) ok = ok && (ns[i] % bn == 0);
    if (ok && bn >= 32) return bn;
  }
  int bn = (maxn + 15) / 16 * 16;
  return bn > 256 ? 256 : bn;
}

// fp32 [N, K] -> bf16 [N, ldp] (zero padded to ldp columns) and bf16 transpose [K, ldt] (zero padded).
// row_scale (optional, fp32 [N]) multiplies row n before rounding: diag(gamma) W of the gamma-folded layer-scale backward.
__global__ void pack_weight_kernel(const float* __restrict__ w, int N, int K, __nv_bfloat16* __restrict__ dst,
                                   long ldp, int Kp, __nv_bfloat16* __restrict__ dst_t, long ldt, int Np,
                                   const float* __restrict__ row_scale) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int n = n0 + i, k = k0 + tx;
    float v = (n < N && k < K) ? w[static_cast<long>(n) * K + k] : 0.f;
    if (row_scale != nullptr && n < N) v *= row_scale[n];
    tile[i][tx] = v;
    if (dst != nullptr && n < N && k < Kp) dst[static_cast<long>(n) * ldp + k] = __float2bfloat16(v);
  }
  __syncthreads();
  if (dst_t != nullptr) {
    for (int i = ty; i < 32; i += 8) {
      const int k = k0 + i, n = n0 + tx;
      if (k < K && n < Np) dst_t[static_cast<long>(k) * ldt + n] = __float2bfloat16(tile[tx][i]);
    }
  }
}

static int pack_one(const float* w, int N, int K, __nv_bfloat16* dst, long ldp, __nv_bfloat16* dst_t, long ldt,
                    cudaStream_t s, const float* row_scale = nullptr) {
  const int Kp = roundup64(K), Np = roundup64(N);
  dim3 grid((Kp + 31) / 32, (Np + 31) / 32), block(32, 8);
  pack_weight_kernel<<<grid, block, 0, s>>>(w, N, K, dst, ldp, Kp, dst_t, ldt, Np, row_scale);
  return cudaGetLastError() == cudaSuccess ? OCTIC_OK : OCTIC_ERR_CUDA;
}

}  // namespace octic

using namespace octic;

extern "C" {

const char* octic_strerror(int code) {
  switch (code) {
    case OCTIC_OK: return "ok";
    case OCTIC_ERR_ARG: return "invalid argument (size, null pointer or unsupported shape)";
    case OCTIC_ERR_ALIGN: return "pointer or leading dimension is not 16-byte aligned";
    case OCTIC_ERR_DRIVER: return "cuTensorMapEncodeTiled driver entry point unavailable";
    case OCTIC_ERR_TMAP: return "cuTensorMapEncodeTiled failed";
    case OCTIC_ERR_CUDA: return "CUDA launch failed or no sm_100 device";
    default: return "unknown octic error";
  }
}

int octic_version(void) { return 202; }   // 202: streamed tcgen05 attention for long head-major sequences; 201: octic_gemm_last_plan added; 200: round 2 (octic_attention_bwd_ws, octic_sparse_rowmap / posmap added; no entry point changed)

int octic_device_ok(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

int octic_gemm_bf16(const octic_gemm_desc* desc, void* stream) {
  if (desc == nullptr || desc->a == nullptr || desc->b0 == nullptr) return OCTIC_ERR_ARG;
  return launch_gemm_tn(desc, static_cast<cudaStream_t>(stream));
}

int octic_gemm_wgrad_bf16(const octic_wgrad_desc* desc, void* stream) {
  if (desc == nullptr || desc->dy == nullptr || desc->x == nullptr) return OCTIC_ERR_ARG;
  return launch_gemm_wgrad(desc, static_cast<cudaStream_t>(stream));
}

int octic_gemm_last_plan(octic_gemm_plan* out) { return gemm_last_plan(out); }

int octic_linear_d8_pack_weights(const float* wA1, const float* wA2, const float* wB1, const float* wB2,
                                 const float* wE, int Din, int Dout, void* w1d, void* wE_packed, void* w1d_t,
                                 void* wE_t, void* stream) {
  if (Din % 8 || Dout % 8 || !wA1 || !wA2 || !wB1 || !wB2 || !wE) return OCTIC_ERR_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int Ci = Din / 8, Co = Dout / 8;
  const long ld1 = roundup64(Ci), ldE = roundup64(2 * Ci), ld1t = roundup64(Co), ldEt = roundup64(2 * Co);
  const float* w[4] = {wA1, wA2, wB1, wB2};
  for (int g = 0; g < 4; ++g) {
    __nv_bfloat16* d = w1d ? static_cast<__nv_bfloat16*>(w1d) + static_cast<long>(g) * Co * ld1 : nullptr;
    __nv_bfloat16* dt = w1d_t ? static_cast<__nv_bfloat16*>(w1d_t) + static_cast<long>(g) * Ci * ld1t : nullptr;
    int rc = pack_one(w[g], Co, Ci, d, ld1, dt, ld1t, s);
    if (rc) return rc;
  }
  return pack_one(wE, 2 * Co, 2 * Ci, static_cast<__nv_bfloat16*>(wE_packed), ldE,
                  static_cast<__nv_bfloat16*>(wE_t), ldEt, s);
}

int octic_linear_d8_pack_weights_scaled(const float* wA1, const float* wA2, const float* wB1, const float* wB2,
                                        const float* wE, const float* gamma, int Din, int Dout, void* w1d_t, void* wE_t,
                                        void* stream) {
  if (Din % 8 || Dout % 8 || !wA1 || !wA2 || !wB1 || !wB2 || !wE || !gamma || !w1d_t || !wE_t) return OCTIC_ERR_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int Ci = Din / 8, Co = Dout / 8;
  const long ld1t = roundup64(Co), ldEt = roundup64(2 * Co);
  const float* w[4] = {wA1, wA2, wB1, wB2};
  for (int g = 0; g < 4; ++g) {
    int rc = pack_one(w[g], Co, Ci, nullptr, 0, static_cast<__nv_bfloat16*>(w1d_t) + static_cast<long>(g) * Ci * ld1t, ld1t, s,
                      gamma + g * Co);
    if (rc) return rc;
  }
  return pack_one(wE, 2 * Co, 2 * Ci, nullptr, 0, static_cast<__nv_bfloat16*>(wE_t), ldEt, s, gamma + 4 * Co);
}

int octic_linear_pack_weights_scaled(const float* w, const float* gamma, int N, int K, void* w_t_packed, void* stream) {
  if (!w || !gamma || !w_t_packed || N <= 0 || K <= 0) return OCTIC_ERR_ARG;
  return pack_one(w, N, K, nullptr, 0, static_cast<__nv_bfloat16*>(w_t_packed), roundup64(N),
                  static_cast<cudaStream_t>(stream), gamma);
}

int octic_linear_pack_weights(const float* w, int N, int K, void* w_packed, void* w_t_packed, void* stream) {
  if (!w || N <= 0 || K <= 0) return OCTIC_ERR_ARG;
  return pack_one(w, N, K, static_cast<__nv_bfloat16*>(w_packed), roundup64(K),
                  static_cast<__nv_bfloat16*>(w_t_packed), roundup64(N), static_cast<cudaStream_t>(stream));
}

// Six groups over the packed row: A1, A2, B1, B2 (K = Ci, N = Co) and the two E rows (K = 2Ci, N = 2Co, shared W_E).
static void fill_d8_groups(octic_gemm_desc* d, int Ci, int Co, bool has_bias) {
  d->num_groups = 6;
  for (int g = 0; g < 4; ++g) {
    octic_gemm_group& G = d->groups[g];
    G.a_col = g * Ci; G.k = Ci; G.b_map = 0; G.b_row = g * Co; G.n = Co; G.c_col = g * Co;
    G.bias_off = (g == 0 && has_bias) ? 0 : -1;
  }
  for (int r = 0; r < 2; ++r) {
    octic_gemm_group& G = d->groups[4 + r];
    G.a_col = 4 * Ci + r * 2 * Ci; G.k = 2 * Ci; G.b_map = 1; G.b_row = 0; G.n = 2 * Co;
    G.c_col = 4 * Co + r * 2 * Co; G.bias_off = -1;
  }
  if (d->head_H > 0 && d->head_S > 0) {
    // head vector [A1 | A2 | B1 | B2 | E row 0 | E row 1], c_h = Co / (S * H) columns per 1-D irrep
    const int ch = Co / (d->head_S * d->head_H);
    d->head_D = 8 * Co / d->head_S;
    for (int g = 0; g < 4; ++g) d->head_off[g] = g * ch;
    d->head_off[4] = 4 * ch;
    d->head_off[5] = 6 * ch;
  }
}

// N-tile width of a LinearD8 launch (Co output channels per 1-D irrep, Ci input channels).  Measured on B200 at the
// ViT-H/14 shapes (tools/gpu/r2_u.sh, profiles/r02_gemm_block_n.txt): wide outputs with a short contraction (qkv, fc1 and
// the fc2 dgrad: K = 160 / 320) are bound by operand traffic per tile and want the largest tile, 256 columns, even with a
// ragged last tile (fc1 126 -> 116 us, fc2 dgrad 127 -> 116, qkv 100 -> 90); the head-major scatter epilogue is bound by
// its own latency per warp and wants 128 columns = one 32-column chunk per epilogue warp (qkv head-major 232 -> 175 us);
// everything else keeps the largest exact divisor (proj / fc2 + residual and the long-K dgrads lose with ragged tiles).
static int pick_block_n_d8(int Co, int Ci, bool head_major) {
  const int ns[2] = {Co, 2 * Co};
  const int exact = pick_block_n(ns, 2);
  if (getenv("OCTIC_BLOCK_N") != nullptr) return exact;       // forced (pick_block_n honours it)
  if (Co >= 480 && Ci <= 160) return head_major ? 128 : 256;
  return exact;
}

int octic_linear_d8_fwd(const void* x, int T, int Din, int Dout, const void* w1d, const void* wE_packed,
                        const float* bias, const octic_gemm_desc* epi, void* stream) {
  if (!x || !w1d || !wE_packed || !epi || Din % 8 || Dout % 8) return OCTIC_ERR_ARG;
  const int Ci = Din / 8, Co = Dout / 8;
  octic_gemm_desc d = *epi;
  d.a = x; d.lda = Din; d.a_cols = Din; d.M = T;
  d.b0 = w1d; d.b0_rows = 4L * Co; d.b0_cols = roundup64(Ci); d.b0_ld = roundup64(Ci);
  d.b1 = wE_packed; d.b1_rows = 2L * Co; d.b1_cols = roundup64(2 * Ci); d.b1_ld = roundup64(2 * Ci);
  d.bias = bias;
  fill_d8_groups(&d, Ci, Co, bias != nullptr);
  d.block_n = pick_block_n_d8(Co, Ci, d.head_H > 0);
  return launch_gemm_tn(&d, static_cast<cudaStream_t>(stream));
}

int octic_linear_d8_dgrad(const void* dy, int T, int Din, int Dout, const void* w1d_t, const void* wE_t, void* dx,
                          int head_H, void* stream) {
  if (!dy || !w1d_t || !wE_t || !dx || Din % 8 || Dout % 8 || head_H < 0) return OCTIC_ERR_ARG;
  const int Ci = Din / 8, Co = Dout / 8;
  octic_gemm_desc d;
  memset(&d, 0, sizeof(d));
  d.a = dy; d.lda = Dout; d.a_cols = Dout; d.M = T;
  d.b0 = w1d_t; d.b0_rows = 4L * Ci; d.b0_cols = roundup64(Co); d.b0_ld = roundup64(Co);
  d.b1 = wE_t; d.b1_rows = 2L * Ci; d.b1_cols = roundup64(2 * Co); d.b1_ld = roundup64(2 * Co);
  // roles of (Ci, Co) swap: contraction over the output features, result has Din columns
  d.mode = OCTIC_EPI_BF16;
  d.head_H = head_H;
  d.head_S = 1;
  fill_d8_groups(&d, Co, Ci, false);
  d.block_n = pick_block_n_d8(Ci, Co, head_H > 0);
  d.mode = OCTIC_EPI_BF16;
  d.out = dx; d.ldo = Din;
  return launch_gemm_tn(&d, static_cast<cudaStream_t>(stream));
}

int octic_linear_d8_wgrad(const void* dy, const void* x, int T, int Din, int Dout, float* dwA1, float* dwA2,
                          float* dwB1, float* dwB2, float* dwE, void* stream) {
  if (!dy || !x || !dwA1 || !dwA2 || !dwB1 || !dwB2 || !dwE || Din % 8 || Dout % 8) return OCTIC_ERR_ARG;
  const int Ci = Din / 8, Co = Dout / 8;
  octic_wgrad_desc d;
  memset(&d, 0, sizeof(d));
  d.dy = dy; d.ld_dy = Dout; d.dy_cols = Dout;
  d.x = x; d.ld_x = Din; d.x_cols = Din;
  d.T = T;
  d.num_groups = 6;
  float* dw[4] = {dwA1, dwA2, dwB1, dwB2};
  for (int g = 0; g < 4; ++g) {
    octic_wgrad_group& G = d.groups[g];
    G.dy_col = g * Co; G.x_col = g * Ci; G.n_out = Co; G.k_in = Ci; G.dw = dw[g]; G.ldw = Ci;
  }
  for (int r = 0; r < 2; ++r) {   // both E rows accumulate into the same dW_E
    octic_wgrad_group& G = d.groups[4 + r];
    G.dy_col = 4 * Co + r * 2 * Co; G.x_col = 4 * Ci + r * 2 * Ci; G.n_out = 2 * Co; G.k_in = 2 * Ci;
    G.dw = dwE; G.ldw = 2 * Ci;
  }
  int bn = roundup64(Ci);
  d.block_n = bn > 256 ? 256 : bn;
  d.splits = 0;
  return launch_gemm_wgrad(&d, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
