/*
 * octic_b200.h -- C ABI of the B200-native octic ViT block hot path (liboctic_b200.so).
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream handle (cudaStream_t passed as
 * void*), returns 0 (OCTIC_OK) or a negative OCTIC_ERR_* code, never allocates device memory and never
 * synchronises.  Outputs and workspaces are owned by the caller.  There is no CPU path: without a sm_100
 * device every compute entry point fails with OCTIC_ERR_CUDA.
 *
 * Data layout ("packed octic row").  The reference keeps an octic feature of width D = 8C as a 5-tuple
 * (A1, A2, B1, B2, E) of tensors [B,N,C] x4 and [B,N,2,2C] (reference octic_vits/d8_layers.py:64-82,111-112,
 * octic_vits/d8_utils.py:358-385).  Here one token is one contiguous row of D elements
 *
 *        [ A1 (C) | A2 (C) | B1 (C) | B2 (C) | E row 0 (2C) | E row 1 (2C) ]
 *
 * so the reference's five tensors are strided views of a single [T, D] matrix (T = B*N tokens), and the
 * reference 8-tuple component k of channel c sits at column offset {0,1,2,3,4,6,5,7}[k]*C + c.
 *
 * Each function cites the reference interface it replaces (file:line relative to the reference repo).
 */
#ifndef OCTIC_B200_H_
#define OCTIC_B200_H_

#include <stdint.h>

#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

#define OCTIC_OK 0
#define OCTIC_ERR_ARG (-1)     /* bad size / null pointer / unsupported shape            */
#define OCTIC_ERR_ALIGN (-2)   /* pointer or leading dimension not 16-byte aligned       */
#define OCTIC_ERR_DRIVER (-3)  /* cuTensorMapEncodeTiled entry point not available       */
#define OCTIC_ERR_TMAP (-4)    /* tensor-map encode failed                               */
#define OCTIC_ERR_CUDA (-5)    /* launch failed / no sm_100 device                       */

#define OCTIC_MAX_GROUPS 8

/* element types for the pointwise kernels */
#define OCTIC_F32 0
#define OCTIC_BF16 1

/* GEMM epilogues */
#define OCTIC_EPI_BF16 0       /* out_bf16 = acc + bias                                                       */
#define OCTIC_EPI_RESID 1      /* resid_out_f32 = resid_in + row_scale[m/rows_per_sample]*gamma[c]*bf16(acc+bias); */
                               /* optional branch_out_bf16 = acc + bias (saved for the layer-scale gradient)  */
#define OCTIC_EPI_F32 2        /* out_f32 = acc + bias                                                        */
#define OCTIC_EPI_GELU_BF16 3  /* out_bf16 = gelu(bf16(acc + bias)); optional branch_out_bf16 = acc + bias    */
#define OCTIC_EPI_GELU_BWD 4   /* out_bf16 = acc * gelu'(gelu_pre[m, c]) -- the fc2 dgrad with the nn.GELU backward of */
                               /* deit/vit.py:126-129 fused; optional colsum[c] += sum_m out (the fc1 bias gradient)  */

const char* octic_strerror(int code);
int octic_version(void);
/* 1 when a CUDA device with compute capability 10.x is current, else 0. */
int octic_device_ok(void);

/* ---------------------------------------------------------------------------------------------------------
 * Grouped bf16 GEMM on tcgen05 (the engine under LinearD8 / nn.Linear).
 *   C[m, c_col + n] = sum_k A[m, a_col + k] * B[b_row + n, k]      for every group, m < M
 * A is [M, a_cols] bf16 row-major (lda elements); B0/B1 are bf16 weight matrices [rows, cols] whose K extent is
 * zero-padded to a multiple of 64; a group picks B0 or B1 with b_map.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
  int a_col;    /* first column of A used by this group (multiple of 8)     */
  int k;        /* contraction length (<= padded weight columns)            */
  int b_map;    /* 0 -> b0, 1 -> b1                                         */
  int b_row;    /* first weight row of this group                           */
  int n;        /* output features of this group                            */
  int c_col;    /* first output column                                      */
  int bias_off; /* offset into bias[], or -1 for "no bias on this group"    */
} octic_gemm_group;

typedef struct {
  const void* a; long lda; long a_cols; int M;
  const void* b0; long b0_rows; long b0_cols; long b0_ld;
  const void* b1; long b1_rows; long b1_cols; long b1_ld;   /* b1 may be NULL */
  int num_groups;
  octic_gemm_group groups[OCTIC_MAX_GROUPS];
  int block_n;                /* N tile, multiple of 16, <= 256                                        */
  int mode;                   /* OCTIC_EPI_*                                                           */
  void* out; long ldo;        /* EPI_BF16 / EPI_F32 / EPI_GELU_BF16 destination                        */
  const float* bias;          /* fp32, indexed bias_off + n                                            */
  const float* gamma;         /* EPI_RESID: fp32 per output column (c_col + n), NULL = 1               */
  const float* resid_in;      /* EPI_RESID: fp32 [M', ldr], NULL = 0                                   */
  float* resid_out; long ldr; /* EPI_RESID destination (may alias resid_in)                            */
  const float* row_scale;     /* EPI_RESID: per-sample scale (DropPath keep-mask / keep_prob), or NULL */
  int rows_per_sample;
  void* branch_out; long ldb; /* optional bf16 copy of acc + bias (EPI_GELU_BF16: row stride ldo; ldb 0 or ldo) */
  int remap_group; int remap_extra; int remap_off; /* EPI_RESID/EPI_F32 row remap: m' = m + (m/remap_group)*remap_extra + remap_off (0 = identity) */
  /* EPI_BF16 head remap (0 heads = off).  Feature n of a group with n_g outputs is read as [S][H][c_g]
   * (c_g = n_g / (S*H), even) and stored at column s*head_D + h*(head_D/H) + head_off[group] + j instead of
   * c_col + n: the qkv LinearD8 (S = 3) and the proj dgrad (S = 1) emit head-major rows for the attention kernels
   * (reference pack step octic_vits/d8_layers.py:632-641) straight from the GEMM epilogue. */
  int head_H; int head_S; int head_D; int head_off[OCTIC_MAX_GROUPS];
  const void* gelu_pre;       /* EPI_GELU_BWD: bf16 pre-activation, same shape and row stride (ldo) as out */
  float* colsum;              /* EPI_GELU_BWD: optional fp32 [>= c_col + n], accumulated with red.add      */
} octic_gemm_desc;

int octic_gemm_bf16(const octic_gemm_desc* desc, void* stream);

/* Weight gradient: dW_g[n, k] += sum_t dY[t, dy_col + n] * X[t, x_col + k], fp32, accumulated with red.add
 * (the caller zeroes or pre-loads dW).  Replaces the autograd wgrad of nn.Linear inside LinearD8
 * (octic_vits/d8_layers.py:117-127). */
typedef struct {
  int dy_col; int x_col; int n_out; int k_in;   /* dy_col, x_col: multiples of 8 */
  float* dw; long ldw;
} octic_wgrad_group;

typedef struct {
  const void* dy; long ld_dy; long dy_cols;
  const void* x; long ld_x; long x_cols;
  int T;
  int num_groups;
  octic_wgrad_group groups[OCTIC_MAX_GROUPS];
  int block_n;  /* tile over k_in: multiple of 64, <= 256 */
  int splits;   /* token-range splits; 0 = choose          */
} octic_wgrad_desc;

int octic_gemm_wgrad_bf16(const octic_wgrad_desc* desc, void* stream);

/* Launch plan of the last GEMM this host thread launched (octic_gemm_bf16, octic_gemm_wgrad_bf16 or a wrapper over them:
 * LinearD8 forward / dgrad / wgrad, the dense helpers).  It is recorded from the same values the launch uses, right
 * before the kernel is launched, so a test can assert which code path a shape takes.  Returns OCTIC_ERR_ARG when this
 * thread has launched no GEMM yet.  A refused call (a negative return before the launch) leaves the previous plan. */
#define OCTIC_GEMM_PLAN_TN 0
#define OCTIC_GEMM_PLAN_WGRAD 1
typedef struct {
  int kind;          /* OCTIC_GEMM_PLAN_TN or OCTIC_GEMM_PLAN_WGRAD                                              */
  int mode;          /* tn: OCTIC_EPI_*; wgrad: -1                                                                 */
  int ncta;          /* 1 = single CTAs, 2 = CTA pairs (cta_group::2, 256-row tiles)                              */
  int num_stages;    /* TMA ring depth                                                                            */
  int ws;            /* tn: weight-stationary tile order                                                          */
  int block_n;       /* N tile (tn: output columns; wgrad: X columns)                                              */
  int grid;          /* CTAs launched (pairs count twice)                                                          */
  int num_m_blocks;  /* tn: blocks of 128 * ncta rows                                                              */
  int total_tiles;   /* output tiles of the launch                                                                */
  int kb_total;      /* wgrad: 64-token k-blocks                                                                  */
  int full_rounds;   /* wgrad: rounds in which every CTA (pair) takes one whole tile                               */
  int rem_tiles;     /* wgrad: tiles left after the full rounds                                                    */
  int rem_splits;    /* wgrad: > 0 = each remaining tile cut into this many token ranges; 0 = one stream-K line     */
  int splits;        /* wgrad: the descriptor's splits                                                             */
  int packed;        /* tn: 1 = bf16-packed epilogue staging where it applies (OCTIC_GEMM_PACKED unset)            */
  int direct;        /* tn: 1 = register-direct epilogue for this launch's mode (OCTIC_GEMM_DIRECT mask)           */
  int roles_low;     /* 1 = TMA producer / MMA issuer on warps 0 / 1 (OCTIC_GEMM_ROLES_HIGH unset)                 */
} octic_gemm_plan;

int octic_gemm_last_plan(octic_gemm_plan* out);

/* ---------------------------------------------------------------------------------------------------------
 * LinearD8 (octic_vits/d8_layers.py:104-127): 5 block-diagonal linears = 6 GEMM groups over packed rows.
 * Packed weights: w1d = [A1;A2;B1;B2] rows, each [Dout/8, roundup64(Din/8)], wE = [Dout/4, roundup64(Din/4)];
 * the *_t buffers hold the transposes ([Din/8 rows..] x roundup64(Dout/8) etc.) used by dgrad.
 * --------------------------------------------------------------------------------------------------------- */
int octic_linear_d8_pack_weights(const float* wA1, const float* wA2, const float* wB1, const float* wB2,
                                 const float* wE, int Din, int Dout, void* w1d, void* wE_packed, void* w1d_t,
                                 void* wE_t, void* stream);

/* y = LinearD8(x): x bf16 [T, Din] packed rows, bias fp32 [Dout/8] (A1 only) or NULL.  The epilogue fields of
 * `epi` (mode/out/ldo/gamma/resid/row_scale/branch_out, head_H/head_S) are honoured; a/b/groups/bias and the
 * head_D/head_off fields are filled in here. */
int octic_linear_d8_fwd(const void* x, int T, int Din, int Dout, const void* w1d, const void* wE_packed,
                        const float* bias, const octic_gemm_desc* epi, void* stream);
/* dx = LinearD8^T(dy): dy bf16 [T, Dout] -> dx bf16 [T, Din] using the transposed packs.  head_H > 0: dx rows are
 * written head-major ([H][hd], head vector [A1|A2|B1|B2|E0|E1]) instead of packed -- the d_o operand of
 * octic_attention_bwd(OCTIC_ATTN_OCTIC_HEADMAJOR). */
int octic_linear_d8_dgrad(const void* dy, int T, int Din, int Dout, const void* w1d_t, const void* wE_t,
                          void* dx, int head_H, void* stream);
/* dW_* += dy^T x per irrep (fp32 [Dout/8, Din/8] x4 and [Dout/4, Din/4]). */
int octic_linear_d8_wgrad(const void* dy, const void* x, int T, int Din, int Dout, float* dwA1, float* dwA2,
                          float* dwB1, float* dwB2, float* dwE, void* stream);

/* Dense nn.Linear helpers (deit/vit.py:29-33): pack fp32 [N, K] -> bf16 [N, roundup64(K)] and its transpose. */
int octic_linear_pack_weights(const float* w, int N, int K, void* w_packed, void* w_t_packed, void* stream);
/* Transposed packs of diag(gamma) W (dgrad operand of the gamma-folded layer-scale backward, see
 * octic_layerscale_wgrad_finalize): gamma fp32 [N] (dense) or the packed [Dout] vector (octic, alpha_E repeated). */
int octic_linear_pack_weights_scaled(const float* w, const float* gamma, int N, int K, void* w_t_packed, void* stream);
int octic_linear_d8_pack_weights_scaled(const float* wA1, const float* wA2, const float* wB1, const float* wB2,
                                        const float* wE, const float* gamma, int Din, int Dout, void* w1d_t, void* wE_t,
                                        void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * D8 GELU (octic_vits/d8_gelu.py:103-196 fwd, :209-331 bwd, :456-482 autograd wrapper; maths
 * octic_vits/d8_utils.py:276-344): y = R2I(gelu(I2R(x))) over the 8 irrep components of each channel.
 * x, y: [T, 8C] packed rows of dtype OCTIC_F32 or OCTIC_BF16; ld* = row strides in elements.
 * colsum (optional, fp32 [8C], pre-zeroed) receives sum_t gin[t, :] (bias gradient of the preceding LinearD8).
 * --------------------------------------------------------------------------------------------------------- */
int octic_gelu_d8_fwd(const void* x, long ldx, void* y, long ldy, long T, int C, int dtype, void* stream);
int octic_gelu_d8_bwd(const void* g, long ldg, const void* x, long ldx, void* gin, long ldgin, long T, int C,
                      int dtype, float* colsum, void* stream);

/* Plain GELU backward for the dense half (nn.GELU, deit/vit.py:68): gin = g * gelu'(x). */
int octic_gelu_bwd(const void* g, const void* x, void* gin, long n_rows, int n_cols, float* colsum, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * LayerNormD8 + AffineD8 (octic_vits/d8_layers.py:161-186, 132-158).  x fp32 [T, D]; alpha fp32 [D] in packed
 * column order (alpha_E repeated for both E rows); beta fp32 [C] or NULL; y bf16 or fp32 [T, D];
 * stats fp32 [T, 8] = (mean A1,A2,B1,B2,E0,E1, rstd, unused) or NULL.
 * bwd: dx_out = dx_in (or 0 if NULL) + LN^T(dy); dalpha[D], dbeta[C] accumulate (pre-zeroed by the caller).
 * Optional by-products for the residual branch that produced x (NULL = off): dx_bf16 [T, D] (row stride lddx) =
 * bf16(dx_out), dx_colsum fp32 [D] += sum_t dx_out (pre-zeroed).
 * --------------------------------------------------------------------------------------------------------- */
int octic_layernorm_d8_fwd(const float* x, long ldx, const float* alpha, const float* beta, float eps, void* y,
                           long ldy, int y_dtype, float* stats, long T, int D, void* stream);
int octic_layernorm_d8_bwd(const void* dy, long lddy, int dy_dtype, const float* x, long ldx, const float* stats,
                           const float* alpha, const float* dx_in, float* dx_out, long lddx, float* dalpha,
                           float* dbeta, long T, int D, void* dx_bf16, float* dx_colsum, void* stream);

/* nn.LayerNorm(eps) of the dense half (octic_vits/model.py:95,140; deit/vit.py:110,124). stats fp32 [T,2]. */
int octic_layernorm_fwd(const float* x, long ldx, const float* w, const float* b, float eps, void* y, long ldy,
                        int y_dtype, float* stats, long T, int D, void* stream);
int octic_layernorm_bwd(const void* dy, long lddy, int dy_dtype, const float* x, long ldx, const float* stats,
                        const float* w, const float* dx_in, float* dx_out, long lddx, float* dw, float* db, long T,
                        int D, void* dx_bf16, float* dx_colsum, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Layer-scale + DropPath + residual, backward half (forward is the EPI_RESID GEMM epilogue).
 * LayerScaleD8 / AffineD8(bias=False) as gamma_1/2 (octic_vits/d8_layers.py:189-212, 698-707), DropPathD8
 * (:249-282).  dy_bf16 = gamma * s * dres; dgamma += sum_t dres * s * branch; colsum += sum_t dy.
 * --------------------------------------------------------------------------------------------------------- */
int octic_layerscale_bwd(const float* dres, long lddres, const void* branch, long ldbr, const float* gamma,
                         const float* row_scale, int rows_per_sample, void* dy, long lddy, float* dgamma,
                         float* colsum, long T, int D, void* stream);

/* Gamma-folded variant without DropPath (the branch output is NOT saved in forward).  With g = bf16(dres) and
 * cs = colsum(dres) (by-products of the layer-norm backward above):  dx = g (diag(gamma) W)  [dgrad with the *_scaled
 * packs],  dW_raw = g^T x  [ordinary wgrad into a zeroed buffer], and this call finishes, per weight row n:
 *   dgamma[n] += <W[n,:], dW_raw[n,:]> + bias[n] cs[n]   (= sum_t dres[t,n] branch[t,n], the autograd gradient of
 *   gamma_1/2 in octic_vits/d8_layers.py:698-707),   dW[n,:] = gamma[n] dW_raw[n,:] (in place),   dbias[n] = gamma[n] cs[n].
 * Up to 8 weight matrices (segments) per call: the five irrep weights of a LinearD8, or one nn.Linear. */
typedef struct {
  float* dw; const float* w; int N; int K;   /* fp32 [N, K], contiguous                         */
  const float* gamma;                        /* fp32 [N]                                        */
  const float* bias; const float* cs;        /* fp32 [N] or NULL                                */
  float* dgamma; float* dbias;               /* fp32 [N] or NULL; dgamma accumulates            */
  float* dw_acc;                             /* optional fp32 [N, K]: dw_acc += gamma dW_raw (the parameter's .grad), dw untouched */
} octic_lsfin_seg;
int octic_layerscale_wgrad_finalize(const octic_lsfin_seg* segs, int nseg, void* stream);

/* column sums of a bf16 matrix: out[c] += sum_t x[t, c] (bias gradients). */
int octic_colsum_bf16(const void* x, long ldx, long T, int n_cols, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Attention (AttentionD8, octic_vits/d8_layers.py:623-656; dense Attention, deit/vit.py:36-56).
 * qkv bf16 [B*N, 3D], o bf16 [B*N, D], lse fp32 [B, H, N] (natural log); softmax scale = hd^-1/2 (the SDPA default;
 * AttentionD8.scale is dead code in the reference).  `layout` selects how head vectors sit in the rows:
 *   OCTIC_ATTN_DENSE            qkv = [3][H][hd], o = [H][hd]                       (deit/vit.py:36-50)
 *   OCTIC_ATTN_OCTIC_PACKED     qkv = packed LinearD8 output (per irrep [3][H][c_h]), o = packed octic row: the head
 *                               vector [A1|A2|B1|B2|E0|E1] of d8_layers.py:632-641 is gathered on load and the output
 *                               scattered back into the row of d8_layers.py:650-656 (mma.sync kernels)
 *   OCTIC_ATTN_OCTIC_HEADMAJOR  qkv (and d_o in backward) = [3][H][hd] / [H][hd] with the head vector in the order
 *                               [A1|A2|B1|B2|E0|E1] -- what octic_linear_d8_fwd / _dgrad write with head_remap set --
 *                               while o and dqkv are packed octic rows.  tcgen05 kernels fed by TMA; the shape must
 *                               satisfy octic_attention_headmajor_supported().
 * In every case the reference's cat / permute / contiguous copies never exist.
 * --------------------------------------------------------------------------------------------------------- */
#define OCTIC_ATTN_DENSE 0
#define OCTIC_ATTN_OCTIC_PACKED 1
#define OCTIC_ATTN_OCTIC_HEADMAJOR 2
/* 1 when the tcgen05 kernels serve the head-major layouts at (N, hd) for the given direction.  Two families do:
 *   resident  the whole K / V (and Q / dO) of one (image, head) in one CTA's shared memory: N up to ~300 in backward
 *             and 512 in forward;
 *   streamed  one CTA per 128-row tile of one (image, head), the other side streamed in 64-row chunks.  Admitted only
 *             where neither the resident kernels nor the mma.sync backward of the dense layout fit (hd 64: N > 784,
 *             hd 80: N > 640), and for hd in {32, 64, 80, 96, 128} up to N = 8192 at least.  So every (N, hd) that
 *             trains on the other kernels keeps its kernel; forward-only calls just below the mma.sync forward limit
 *             (hd 64: N 785..800, hd 80: N 641..656) move here, since a layer uses one layout for both passes.
 * Returns 0 otherwise: the packed layout (mma.sync) remains the only one there. */
int octic_attention_headmajor_supported(int N, int hd, int backward);
int octic_attention_fwd(const void* qkv, void* o, float* lse, int B, int N, int H, int hd, int layout,
                        void* stream);
/* delta_ws: caller-provided fp32 workspace [B, H, N] (receives rowsum(dO * O)). */
int octic_attention_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, float* delta_ws,
                        void* dqkv, int B, int N, int H, int hd, int layout, void* stream);
/* Same backward with a caller-provided scratch for the staged dQ path of the tcgen05 kernel (the autograd of
 * F.scaled_dot_product_attention at octic_vits/d8_layers.py:645-648 / deit/vit.py:44-48): the key-major pass writes
 * dS^T (bf16) into an L2-resident slot per resident CTA and dQ = dS K is one MMA chain per 128-query tile instead of a
 * second pass that recomputes S, dP and the exponentials.  ws: octic_attention_bwd_workspace_bytes(N, hd) bytes,
 * 256-byte aligned, its first 4096 bytes zeroed once by the caller (slot flags; every launch leaves them zero); it
 * may be shared by all launches on ONE stream.  ws = NULL (or a shape the staged path does not cover: the size
 * query returns 0) runs the two-pass kernel; both produce the same gradients up to bf16 rounding of dS.
 * The streamed kernels need no workspace: dQ comes from a query-major pass that recomputes S and dP, so for their
 * shapes (and without a device) the size query returns 0 and ws is ignored. */
size_t octic_attention_bwd_workspace_bytes(int N, int hd);
int octic_attention_bwd_ws(const void* qkv, const void* o, const void* d_o, const float* lse, float* delta_ws,
                           void* dqkv, int B, int N, int H, int hd, int layout, void* ws, size_t ws_bytes,
                           void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * PowerSpectrumInvariant (octic_vits/d8_invariantization.py:49-64): [T, 8C] fp32 -> [T, 6C] bf16
 *   (A1, |A2|, |B1|, |B2|, sqrt(E0^2 + E1^2)); bwd gives fp32 [T, 8C] with the norm subgradient 0 at 0.
 * Hybrid bridge (octic_vits/model.py:200, octic_vits/d8_utils.py:370-385): packed row -> 8-tuple concat order
 * (swaps the column blocks [5C,6C) and [6C,7C)); it is an involution, so backward = the same call.
 * --------------------------------------------------------------------------------------------------------- */
int octic_power_spectrum_fwd(const float* x, long ldx, void* y, long ldy, long T, int C, void* stream);
int octic_power_spectrum_bwd(const void* dy, long lddy, int dy_dtype, const float* x, long ldx, float* dx,
                             long lddx, long T, int C, void* stream);
int octic_bridge_permute(const float* x, long ldx, float* y, long ldy, long T, int C, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Front end (PatchEmbedD8 / LiftD8, octic_vits/d8_layers.py:375-486): non-overlapping patches of an fp32 image
 * [B, Cin, H, W] -> bf16 rows [B*gh*gw, roundup64(Cin*p*p)] in (c, i, j) order (the conv-as-GEMM operand).
 * --------------------------------------------------------------------------------------------------------- */
int octic_im2col_patches(const float* img, int B, int Cin, int Himg, int Wimg, int p, void* out, long ldo,
                         void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Symmetric parameter expansion: the D8-symmetric lifting filters (LiftIrrepD8Conv2d.get_weight,
 * octic_vits/d8_layers.py:329-373, 475-484) and the unfolded positional embedding (isotypic_dim_interpolation,
 * octic_vits/d8_utils.py:388-451) are sparse linear maps of the stored half-size parameters; idx / coef are
 * [n_out, K] device tables built by the caller from the reference formula (K <= 16, unused slots: coef 0).
 *   rowmap: out[r, o] (+)= sum_k coef[o, k] * in[r, idx[o, k]]      rows r, fp32, row strides in elements
 *   posmap: out[o, c] (+)= sum_k coef[o, k] * in[idx[o, k], c]      cols c contiguous
 * The transposed tables give the backward of either (accumulate = 1 adds into out).
 * --------------------------------------------------------------------------------------------------------- */
int octic_sparse_rowmap(const float* in, long ld_in, float* out, long ld_out, long rows, int n_out, int K, const int* idx,
                        const float* coef, int accumulate, void* stream);
int octic_sparse_posmap(const float* in, long ld_in, float* out, long ld_out, int n_out, int cols, int K, const int* idx,
                        const float* coef, int accumulate, void* stream);

/* fp32 <-> bf16 casts of [rows, cols] matrices (row strides in elements). */
int octic_cast_f32_to_bf16(const float* x, long ldx, void* y, long ldy, long rows, int cols, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Parameter update of the training step (SURVEY section 8 f3), one or two streaming kernels over ALL parameters:
 *   LAMB   -- the DeiT-III recipe's optimizer (experiments/train_deit.py:42 `args.opt = "fusedlamb"`, created by
 *             timm.optim.create_optimizer at deit/main.py:365 -> apex.optimizers.FusedLAMB, apex pinned at commit
 *             2386a912164 in DEIT_ENV.md:5-14; neither timm nor apex is vendored in the reference);
 *   AdamW  -- the DINOv2 recipe's optimizer (dinov2/train/train.py:67-68 torch.optim.AdamW);
 *   EMA    -- teacher / model-EMA update fused into the parameter write (dinov2/train/ssl_meta_arch.py:370-379
 *             `_foreach_mul_` + `_foreach_add_`; deit/engine.py:81-82 ModelEma.update).
 * Gradients and both moments live in flat fp32 buffers (the .grad views of parallel.FlatGrads); parameters (and EMA
 * targets) stay where the framework allocated them and are reached through a chunk table: chunk i covers `len`
 * elements (<= 8192) of one parameter tensor `p` (EMA copy `ema`, may be NULL) whose gradient/moments start at flat
 * element `off`; `seg` indexes the per-tensor hyper-parameters.
 *
 *   stage 1   g' = g * min(1, max_grad_norm / sqrt(*gnorm_sq))                 (gnorm_sq == NULL: no clipping)
 *             m = beta1*m + beta3*g';  v = beta2*v + (1-beta2)*g'^2
 *             u = (m/bc1) / (sqrt(v/bc2) + eps) + weight_decay[seg]*p
 *             apply != 0 (AdamW):  p -= lr*lr_scale[seg]*u  [; ema = mom*ema + (1-mom)*p]
 *             apply == 0 (LAMB):   g <- u (in place), chunk_norms[chunk] = (|p|^2, |u|^2) of the chunk
 *   stage 2   (LAMB) per-tensor norms = fixed-order sums of the chunk partials (into seg_norms[nsegs][2]), then
 *             p -= lr*lr_scale[seg]*trust*u,  trust = |p|/|u| when (use_nvlamb or weight_decay[seg] != 0) and
 *             both norms are non-zero, else 1  [; ema update as above]
 * All reductions are deterministic (no float atomics): replicas holding identical all-reduced gradients stay
 * bit-identical.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
  float* p;     /* parameter tensor + element offset of this chunk                         */
  float* ema;   /* EMA copy of the same elements, or NULL                                  */
  long off;     /* first element in the flat gradient / moment buffers                     */
  int len;      /* elements in this chunk                                                  */
  int seg;      /* parameter tensor index (hyper-parameters, norms)                        */
} octic_optim_chunk;

typedef struct {
  float weight_decay;
  float lr_scale;
  int first_chunk;   /* chunks of one tensor are contiguous in the table                   */
  int num_chunks;
} octic_optim_seg;

#define OCTIC_OPTIM_SQNORM_PARTIALS 1184   /* floats of workspace octic_optim_sqnorm needs (148 SMs x 8) */

/* out[0] = sum_i x[i]^2 (two launches: per-CTA partials, fixed-order final sum) */
int octic_optim_sqnorm(const float* x, long n, float* partials, float* out, void* stream);
int octic_optim_stage1(const octic_optim_chunk* chunks, int nchunks, const octic_optim_seg* segs, float* g, float* m,
                       float* v, float* chunk_norms, const float* gnorm_sq, float max_grad_norm, float beta1,
                       float beta2, float beta3, float eps, float bc1, float bc2, float lr, int apply,
                       float ema_momentum, void* stream);
int octic_optim_lamb_stage2(const octic_optim_chunk* chunks, int nchunks, const octic_optim_seg* segs, int nsegs,
                            const float* u, const float* chunk_norms, float* seg_norms, float lr, int use_nvlamb,
                            float ema_momentum, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OCTIC_B200_H_ */
