"""Tensor-level wrappers over the C ABI (no autograd here; see functional.py for the differentiable ops).

Conventions: activations are packed octic rows (see include/octic_b200.h) stored as 2-D tensors [T, D]
(T = B*N tokens).  bf16 for GEMM operands, fp32 for the residual stream and parameters.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import BF16, EPI_BF16, EPI_F32, EPI_GELU_BF16, EPI_GELU_BWD, EPI_RESID, F32, GemmDesc, WgradDesc, call


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype: torch.dtype, name: str, ndim: int = 2) -> None:
    if not t.is_cuda:
        raise _lib.OcticError(f"{name}: expected a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise _lib.OcticError(f"{name}: expected {dtype}, got {t.dtype}")
    if ndim and t.dim() != ndim:
        raise _lib.OcticError(f"{name}: expected {ndim}-D, got shape {tuple(t.shape)}")
    if t.dim() >= 1 and t.stride(-1) != 1:
        raise _lib.OcticError(f"{name}: last dimension must be contiguous")


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise _lib.OcticError(f"unsupported dtype {t.dtype}")


def roundup64(x: int) -> int:
    return (x + 63) // 64 * 64


# ----------------------------------------------------------------------------------------------------------------
# zeroed fp32 scratch (targets of red.add accumulation: weight-gradient temporaries, LayerNorm / bias column sums).
# A training step asks for ~330 of them; inside a step bracketed by begin_step() they are slices of ONE buffer that is
# zero-filled once (its size is the previous step's demand), instead of one fill kernel each.
# ----------------------------------------------------------------------------------------------------------------
class _ZeroPool:
    def __init__(self):
        self.active, self.buf, self.off, self.demand, self.last_demand = False, None, 0, 0, 0

    def begin_step(self) -> None:
        self.active = True
        if self.demand > 0:
            self.last_demand = self.demand          # what the previous step asked for
        self.demand, self.off, self.buf = 0, 0, None

    def end(self) -> None:
        self.active, self.buf = False, None

    def take(self, n: int, device) -> torch.Tensor:
        n_al = (n + 63) // 64 * 64                       # slices stay 256-byte aligned
        self.demand += n_al
        if not self.active or self.last_demand == 0:
            return torch.zeros(n, dtype=torch.float32, device=device)
        if self.buf is None:
            self.buf = torch.zeros(self.last_demand, dtype=torch.float32, device=device)
            self.off = 0
        if self.buf.device != torch.device(device) or self.off + n_al > self.buf.numel():
            return torch.zeros(n, dtype=torch.float32, device=device)
        out = self.buf[self.off:self.off + n]
        self.off += n_al
        return out


ZERO_POOL = _ZeroPool()


def begin_step() -> None:
    """Call at the start of every training step (parallel.GraphedTrainStep does): see _ZeroPool."""
    ZERO_POOL.begin_step()


def reset_zero_pool() -> None:
    """Drop the step's pool buffer (after a failed CUDA-graph capture its zero fill was recorded, not executed)."""
    ZERO_POOL.end()


def zeros_f32(n: int, device) -> torch.Tensor:
    return ZERO_POOL.take(int(n), device)


# ----------------------------------------------------------------------------------------------------------------
# weights
# ----------------------------------------------------------------------------------------------------------------
@dataclass
class PackedD8:
    """bf16 GEMM operands of one LinearD8 (reference octic_vits/d8_layers.py:117-122)."""
    w1d: torch.Tensor      # [4*Co, roundup64(Ci)]
    wE: torch.Tensor       # [2*Co, roundup64(2*Ci)]
    w1d_t: torch.Tensor    # [4*Ci, roundup64(Co)]
    wE_t: torch.Tensor     # [2*Ci, roundup64(2*Co)]
    din: int
    dout: int


def pack_linear_d8(wA1, wA2, wB1, wB2, wE, need_t: bool = True) -> PackedD8:
    co, ci = wA1.shape
    for w in (wA1, wA2, wB1, wB2):
        _req(w, torch.float32, "LinearD8 weight")
        if tuple(w.shape) != (co, ci) or not w.is_contiguous():
            raise _lib.OcticError("LinearD8 1-D irrep weights must be contiguous [Dout/8, Din/8]")
    _req(wE, torch.float32, "LinearD8 lin_E weight")
    if tuple(wE.shape) != (2 * co, 2 * ci) or not wE.is_contiguous():
        raise _lib.OcticError("LinearD8 lin_E weight must be contiguous [Dout/4, Din/4]")
    dev = wA1.device
    w1d = torch.empty(4 * co, roundup64(ci), dtype=torch.bfloat16, device=dev)
    wEp = torch.empty(2 * co, roundup64(2 * ci), dtype=torch.bfloat16, device=dev)
    w1d_t = torch.empty(4 * ci, roundup64(co), dtype=torch.bfloat16, device=dev) if need_t else None
    wE_t = torch.empty(2 * ci, roundup64(2 * co), dtype=torch.bfloat16, device=dev) if need_t else None
    call("octic_linear_d8_pack_weights", wA1.data_ptr(), wA2.data_ptr(), wB1.data_ptr(), wB2.data_ptr(),
         wE.data_ptr(), 8 * ci, 8 * co, w1d.data_ptr(), wEp.data_ptr(), _ptr(w1d_t), _ptr(wE_t), _stream())
    return PackedD8(w1d, wEp, w1d_t, wE_t, 8 * ci, 8 * co)


def pack_linear_d8_scaled_t(wA1, wA2, wB1, wB2, wE, gamma: torch.Tensor) -> PackedD8:
    """Transposed packs of diag(gamma) W only (gamma = packed [Dout] vector): dgrad operand of the gamma-folded
    layer-scale backward.  The forward fields of the result are None."""
    co, ci = wA1.shape
    dev = wA1.device
    w1d_t = torch.empty(4 * ci, roundup64(co), dtype=torch.bfloat16, device=dev)
    wE_t = torch.empty(2 * ci, roundup64(2 * co), dtype=torch.bfloat16, device=dev)
    call("octic_linear_d8_pack_weights_scaled", wA1.data_ptr(), wA2.data_ptr(), wB1.data_ptr(), wB2.data_ptr(),
         wE.data_ptr(), gamma.data_ptr(), 8 * ci, 8 * co, w1d_t.data_ptr(), wE_t.data_ptr(), _stream())
    return PackedD8(None, None, w1d_t, wE_t, 8 * ci, 8 * co)


def pack_linear_scaled_t(w: torch.Tensor, gamma: torch.Tensor) -> torch.Tensor:
    n, k = w.shape
    wt = torch.empty(k, roundup64(n), dtype=torch.bfloat16, device=w.device)
    call("octic_linear_pack_weights_scaled", w.data_ptr(), gamma.data_ptr(), n, k, wt.data_ptr(), _stream())
    return wt


@dataclass
class PackedDense:
    w: torch.Tensor        # [N, roundup64(K)]
    w_t: Optional[torch.Tensor]  # [K, roundup64(N)]
    n: int
    k: int


def pack_linear(w: torch.Tensor, need_t: bool = True) -> PackedDense:
    _req(w, torch.float32, "Linear weight")
    if not w.is_contiguous():
        raise _lib.OcticError("Linear weight must be contiguous")
    n, k = w.shape
    wp = torch.empty(n, roundup64(k), dtype=torch.bfloat16, device=w.device)
    wt = torch.empty(k, roundup64(n), dtype=torch.bfloat16, device=w.device) if need_t else None
    call("octic_linear_pack_weights", w.data_ptr(), n, k, wp.data_ptr(), _ptr(wt), _stream())
    return PackedDense(wp, wt, n, k)


# ----------------------------------------------------------------------------------------------------------------
# GEMM front ends
# ----------------------------------------------------------------------------------------------------------------
def _epilogue_desc(mode: int, out=None, gamma=None, resid_in=None, resid_out=None, row_scale=None,
                   rows_per_sample: int = 1, branch_out=None, remap=(0, 0, 0), head=(0, 0), gelu_pre=None,
                   colsum=None) -> GemmDesc:
    d = GemmDesc()
    d.mode = mode
    if out is not None:
        d.out = out.data_ptr()
        d.ldo = out.stride(0)
    d.gamma = _ptr(gamma)
    d.resid_in = _ptr(resid_in)
    if resid_out is not None:
        d.resid_out = resid_out.data_ptr()
        d.ldr = resid_out.stride(0)
        if resid_in is not None and resid_in.stride(0) != resid_out.stride(0):
            raise _lib.OcticError("resid_in / resid_out must share a row stride")
    d.row_scale = _ptr(row_scale)
    d.rows_per_sample = rows_per_sample
    if branch_out is not None:
        d.branch_out = branch_out.data_ptr()
        d.ldb = branch_out.stride(0)
    d.remap_group, d.remap_extra, d.remap_off = remap
    d.head_H, d.head_S = head      # (heads, S): EPI_BF16 output rows head-major [S][H][hd] (see octic_b200.h)
    if mode == EPI_GELU_BWD:
        if gelu_pre is None or out is None or gelu_pre.stride(0) != out.stride(0) or gelu_pre.dtype != torch.bfloat16:
            raise _lib.OcticError("EPI_GELU_BWD needs a bf16 pre-activation with the row stride of out")
        d.gelu_pre = gelu_pre.data_ptr()
        d.colsum = _ptr(colsum)
    return d


def _pick_block_n(ns: Sequence[int]) -> int:
    for bn in range(256, 15, -16):
        if bn >= 32 and all(n % bn == 0 for n in ns):
            return bn
    return min(256, (max(ns) + 15) // 16 * 16)


def linear_d8(x: torch.Tensor, pk: PackedD8, bias: Optional[torch.Tensor], mode: int = EPI_BF16, **epi) -> None:
    """LinearD8.forward on packed rows; the result goes wherever the epilogue arguments point."""
    _req(x, torch.bfloat16, "x")
    if x.shape[1] != pk.din or x.stride(0) != pk.din:
        raise _lib.OcticError(f"x must be a dense [T, {pk.din}] bf16 matrix, got {tuple(x.shape)}")
    if bias is not None:
        _req(bias, torch.float32, "bias", ndim=1)
    d = _epilogue_desc(mode, **epi)
    call("octic_linear_d8_fwd", x.data_ptr(), x.shape[0], pk.din, pk.dout, pk.w1d.data_ptr(), pk.wE.data_ptr(),
         _ptr(bias), C.byref(d), _stream(), flops=2.0 * x.shape[0] * pk.din * pk.dout * 3 / 16)


def linear_d8_dgrad(dy: torch.Tensor, pk: PackedD8, head_H: int = 0) -> torch.Tensor:
    """dx = LinearD8^T(dy); head_H > 0 writes dx rows head-major (the d_o operand of the tcgen05 attention backward)."""
    _req(dy, torch.bfloat16, "dy")
    if dy.shape[1] != pk.dout or dy.stride(0) != pk.dout:
        raise _lib.OcticError("dy must be a dense [T, Dout] bf16 matrix")
    dx = torch.empty(dy.shape[0], pk.din, dtype=torch.bfloat16, device=dy.device)
    call("octic_linear_d8_dgrad", dy.data_ptr(), dy.shape[0], pk.din, pk.dout, pk.w1d_t.data_ptr(),
         pk.wE_t.data_ptr(), dx.data_ptr(), int(head_H), _stream(),
         flops=2.0 * dy.shape[0] * pk.din * pk.dout * 3 / 16)
    return dx


def linear_d8_wgrad(dy: torch.Tensor, x: torch.Tensor, din: int, dout: int, targets=None):
    """dW_* (+)= dy^T x per irrep.  targets: five fp32 tensors to accumulate into (the parameters' .grad) instead of a
    fresh zeroed buffer."""
    _req(dy, torch.bfloat16, "dy")
    _req(x, torch.bfloat16, "x")
    ci, co = din // 8, dout // 8
    if targets is not None:
        dws, dwE = list(targets[:4]), targets[4]
    else:
        flat = zeros_f32(8 * co * ci, x.device)      # one fill for all five gradients
        dws = [flat[i * co * ci:(i + 1) * co * ci].view(co, ci) for i in range(4)]
        dwE = flat[4 * co * ci:].view(2 * co, 2 * ci)
    call("octic_linear_d8_wgrad", dy.data_ptr(), x.data_ptr(), x.shape[0], din, dout, dws[0].data_ptr(),
         dws[1].data_ptr(), dws[2].data_ptr(), dws[3].data_ptr(), dwE.data_ptr(), _stream(),
         flops=2.0 * x.shape[0] * din * dout * 3 / 16)
    return (*dws, dwE)


def linear_dense(x: torch.Tensor, w: torch.Tensor, n: int, k: int, bias: Optional[torch.Tensor],
                 mode: int = EPI_BF16, **epi) -> None:
    """out = x[:, :k] @ w[:n, :k]^T (+ epilogue).  w is a packed bf16 matrix whose K extent is zero padded."""
    _req(x, torch.bfloat16, "x")
    _req(w, torch.bfloat16, "w")
    d = _epilogue_desc(mode, **epi)
    d.a, d.lda, d.a_cols, d.M = x.data_ptr(), x.stride(0), x.shape[1], x.shape[0]
    d.b0, d.b0_rows, d.b0_cols, d.b0_ld = w.data_ptr(), w.shape[0], w.shape[1], w.stride(0)
    d.b1 = None
    d.num_groups = 1
    g = d.groups[0]
    g.a_col, g.k, g.b_map, g.b_row, g.n, g.c_col = 0, k, 0, 0, n, 0
    g.bias_off = 0 if bias is not None else -1
    d.bias = _ptr(bias)
    d.block_n = _pick_block_n([n])
    call("octic_gemm_bf16", C.byref(d), _stream(), flops=2.0 * x.shape[0] * n * k)


def linear_dense_wgrad(dy: torch.Tensor, x: torch.Tensor, n: int, k: int, dw: Optional[torch.Tensor] = None,
                       splits: int = 0) -> torch.Tensor:
    """dw[n, k] += dy[:, :n]^T @ x[:, :k]."""
    _req(dy, torch.bfloat16, "dy")
    _req(x, torch.bfloat16, "x")
    if dw is None:
        dw = zeros_f32(n * k, x.device).view(n, k)
    d = WgradDesc()
    d.dy, d.ld_dy, d.dy_cols = dy.data_ptr(), dy.stride(0), dy.shape[1]
    d.x, d.ld_x, d.x_cols = x.data_ptr(), x.stride(0), x.shape[1]
    d.T = x.shape[0]
    d.num_groups = 1
    g = d.groups[0]
    g.dy_col, g.x_col, g.n_out, g.k_in, g.dw, g.ldw = 0, 0, n, k, dw.data_ptr(), dw.stride(0)
    d.block_n = min(256, roundup64(k))
    d.splits = splits
    call("octic_gemm_wgrad_bf16", C.byref(d), _stream(), flops=2.0 * x.shape[0] * n * k)
    return dw


def last_gemm_plan() -> dict:
    """Launch plan of the last GEMM this host thread launched (see octic_gemm_plan in include/octic_b200.h), as a dict
    of its fields.  Raises OcticError before the first GEMM launch."""
    plan = _lib.GemmPlan()
    _lib.check(_lib.load().octic_gemm_last_plan(C.byref(plan)), "octic_gemm_last_plan")
    return {name: getattr(plan, name) for name, _ in plan._fields_}


# ----------------------------------------------------------------------------------------------------------------
# pointwise
# ----------------------------------------------------------------------------------------------------------------
def gelu_d8_fwd(x: torch.Tensor) -> torch.Tensor:
    _req(x, x.dtype, "x")
    y = torch.empty_like(x)
    call("octic_gelu_d8_fwd", x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), x.shape[0], x.shape[1] // 8,
         _dt(x), _stream())
    return y


def gelu_d8_bwd(g: torch.Tensor, x: torch.Tensor, colsum: Optional[torch.Tensor] = None) -> torch.Tensor:
    _req(x, x.dtype, "x")
    _req(g, x.dtype, "g")
    gin = torch.empty_like(x)
    call("octic_gelu_d8_bwd", g.data_ptr(), g.stride(0), x.data_ptr(), x.stride(0), gin.data_ptr(), gin.stride(0),
         x.shape[0], x.shape[1] // 8, _dt(x), _ptr(colsum), _stream(), extra_kernels=int(colsum is not None))
    return gin


def gelu_bwd(g: torch.Tensor, x: torch.Tensor, colsum: Optional[torch.Tensor] = None) -> torch.Tensor:
    _req(x, torch.bfloat16, "x")
    _req(g, torch.bfloat16, "g")
    if not (x.is_contiguous() and g.is_contiguous()):
        raise _lib.OcticError("gelu_bwd expects contiguous matrices")
    gin = torch.empty_like(x)
    call("octic_gelu_bwd", g.data_ptr(), x.data_ptr(), gin.data_ptr(), x.shape[0], x.shape[1], _ptr(colsum), _stream(),
         extra_kernels=int(colsum is not None))
    return gin


def layernorm_fwd(x: torch.Tensor, alpha: torch.Tensor, beta: Optional[torch.Tensor], eps: float, d8: bool,
                  out_dtype=torch.bfloat16, want_stats: bool = True):
    _req(x, torch.float32, "x")
    T, D = x.shape
    y = torch.empty(T, D, dtype=out_dtype, device=x.device)
    stats = torch.empty(T, 8 if d8 else 2, dtype=torch.float32, device=x.device) if want_stats else None
    call("octic_layernorm_d8_fwd" if d8 else "octic_layernorm_fwd", x.data_ptr(), x.stride(0), alpha.data_ptr(),
         _ptr(beta), float(eps), y.data_ptr(), y.stride(0), _dt(y), _ptr(stats), T, D, _stream())
    return y, stats


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, stats: torch.Tensor, alpha: torch.Tensor, d8: bool,
                  dx_in: Optional[torch.Tensor] = None, want_aux: bool = False):
    """returns (dx [= dx_in + LN^T dy], dalpha [D], dbeta [C or D]) and, with want_aux, (bf16(dx), colsum(dx) [D])"""
    T, D = x.shape
    dx = torch.empty(T, D, dtype=torch.float32, device=x.device)
    nb = D // 8 if d8 else D
    flat = zeros_f32(D + nb + (D if want_aux else 0), x.device)
    dalpha, dbeta = flat[:D], flat[D:D + nb]
    dxb = torch.empty(T, D, dtype=torch.bfloat16, device=x.device) if want_aux else None
    dxs = flat[D + nb:] if want_aux else None
    call("octic_layernorm_d8_bwd" if d8 else "octic_layernorm_bwd", dy.data_ptr(), dy.stride(0), _dt(dy),
         x.data_ptr(), x.stride(0), stats.data_ptr(), alpha.data_ptr(), _ptr(dx_in), dx.data_ptr(), dx.stride(0),
         dalpha.data_ptr(), dbeta.data_ptr(), T, D, _ptr(dxb), _ptr(dxs), _stream())
    if want_aux:
        return dx, dalpha, dbeta, dxb, dxs
    return dx, dalpha, dbeta


def layerscale_wgrad_finalize(segs) -> None:
    """segs: list of (dw, w, gamma, bias, cs, dgamma, dbias, dw_acc) -- see octic_layerscale_wgrad_finalize in octic_b200.h."""
    arr = (_lib.LsFinSeg * len(segs))()
    for a, (dw, w, gamma, bias, cs, dgamma, dbias, dw_acc) in zip(arr, segs):
        a.dw_acc = _ptr(dw_acc)
        if not (dw.is_contiguous() and w.is_contiguous() and dw.shape == w.shape):
            raise _lib.OcticError("finalize: dw / w must be contiguous and of equal shape")
        a.dw, a.w, a.N, a.K = dw.data_ptr(), w.data_ptr(), w.shape[0], w.shape[1]
        a.gamma, a.bias, a.cs, a.dgamma, a.dbias = gamma.data_ptr(), _ptr(bias), _ptr(cs), _ptr(dgamma), _ptr(dbias)
    call("octic_layerscale_wgrad_finalize", arr, len(segs), _stream())


def layerscale_bwd(dres: torch.Tensor, branch: Optional[torch.Tensor], gamma: Optional[torch.Tensor],
                   row_scale: Optional[torch.Tensor], rows_per_sample: int, want_colsum: bool = True):
    """returns (dy bf16, dgamma [D] or None, colsum [D] or None)"""
    _req(dres, torch.float32, "dres")
    T, D = dres.shape
    dy = torch.empty(T, D, dtype=torch.bfloat16, device=dres.device)
    flat = zeros_f32(2 * D, dres.device)
    dgamma = flat[:D] if branch is not None else None
    colsum = flat[D:] if want_colsum else None
    call("octic_layerscale_bwd", dres.data_ptr(), dres.stride(0), _ptr(branch),
         branch.stride(0) if branch is not None else 0, _ptr(gamma), _ptr(row_scale), rows_per_sample,
         dy.data_ptr(), dy.stride(0), _ptr(dgamma), _ptr(colsum), T, D, _stream())
    return dy, dgamma, colsum


def colsum_bf16(x: torch.Tensor, n_cols: Optional[int] = None) -> torch.Tensor:
    _req(x, torch.bfloat16, "x")
    n_cols = x.shape[1] if n_cols is None else n_cols
    out = zeros_f32(n_cols, x.device)
    call("octic_colsum_bf16", x.data_ptr(), x.stride(0), x.shape[0], n_cols, out.data_ptr(), _stream())
    return out


# ----------------------------------------------------------------------------------------------------------------
# attention
# ----------------------------------------------------------------------------------------------------------------
ATTN_DENSE, ATTN_OCTIC_PACKED, ATTN_OCTIC_HEADMAJOR = 0, 1, 2


def attention_headmajor_ok(N: int, hd: int, backward: bool = True) -> bool:
    """True when the tcgen05 attention kernels (head-major q, k, v by TMA) cover this sequence length / head dim."""
    return bool(_lib.load().octic_attention_headmajor_supported(int(N), int(hd), int(backward)))


def attention_fwd(qkv: torch.Tensor, B: int, N: int, H: int, hd: int, layout: int, want_lse: bool = True,
                  out: Optional[torch.Tensor] = None):
    """`out`: optional preallocated contiguous bf16 [B*N, D] (e.g. a row slice of a larger matrix: the segments of a
    crop list write into one token matrix)."""
    _req(qkv, torch.bfloat16, "qkv")
    D = H * hd
    if tuple(qkv.shape) != (B * N, 3 * D) or not qkv.is_contiguous():
        raise _lib.OcticError(f"qkv must be contiguous [B*N, 3*D] = [{B * N}, {3 * D}], got {tuple(qkv.shape)}")
    if out is None:
        o = torch.empty(B * N, D, dtype=torch.bfloat16, device=qkv.device)
    else:
        o = out
        _req(o, torch.bfloat16, "out")
        if tuple(o.shape) != (B * N, D) or not o.is_contiguous():
            raise _lib.OcticError(f"out must be contiguous [B*N, D] = [{B * N}, {D}], got {tuple(o.shape)}")
    lse = torch.empty(B, H, N, dtype=torch.float32, device=qkv.device) if want_lse else None
    call("octic_attention_fwd", qkv.data_ptr(), o.data_ptr(), _ptr(lse), B, N, H, hd, int(layout), _stream(),
         flops=4.0 * B * H * N * N * hd)
    return o, lse


def attention_bwd(qkv, o, d_o, lse, B: int, N: int, H: int, hd: int, layout: int,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    for t, nm in ((qkv, "qkv"), (o, "o"), (d_o, "d_o")):
        _req(t, torch.bfloat16, nm)
        if not t.is_contiguous():
            raise _lib.OcticError(f"{nm} must be contiguous")
    if out is None:
        dqkv = torch.empty_like(qkv)
    else:
        dqkv = out
        _req(dqkv, torch.bfloat16, "out")
        if dqkv.shape != qkv.shape or not dqkv.is_contiguous():
            raise _lib.OcticError("out must be contiguous and shaped like qkv")
    delta = torch.empty(B, H, N, dtype=torch.float32, device=qkv.device)
    ws = _attention_bwd_workspace(N, hd, qkv.device) if layout != 1 else None
    call("octic_attention_bwd_ws", qkv.data_ptr(), o.data_ptr(), d_o.data_ptr(), lse.data_ptr(), delta.data_ptr(),
         dqkv.data_ptr(), B, N, H, hd, int(layout), _ptr(ws), 0 if ws is None else ws.numel(), _stream(),
         flops=10.0 * B * H * N * N * hd, stat="octic_attention_bwd")
    return dqkv


# staged-dQ scratch of the tcgen05 attention backward: one buffer per (device, stream), grown on demand, slot flags
# (first 4096 bytes) zeroed at allocation and left zero by every launch.  Launches on one stream are ordered, so they
# share it; OCTIC_ATTN_STAGED_DQ=0 selects the two-pass kernel (A/B timing, tests).
_attn_ws: dict = {}


def _attention_bwd_workspace(N: int, hd: int, device) -> Optional[torch.Tensor]:
    if os.environ.get("OCTIC_ATTN_STAGED_DQ", "1") == "0":
        return None
    need = int(_lib.load().octic_attention_bwd_workspace_bytes(int(N), int(hd)))
    if need == 0:
        return None
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    ws = _attn_ws.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(need, dtype=torch.uint8, device=device)
        _attn_ws[key] = ws
    return ws


# ----------------------------------------------------------------------------------------------------------------
# invariant / bridge / front end
# ----------------------------------------------------------------------------------------------------------------
def power_spectrum_fwd(x: torch.Tensor) -> torch.Tensor:
    _req(x, torch.float32, "x")
    T, D = x.shape
    y = torch.empty(T, 6 * D // 8, dtype=torch.bfloat16, device=x.device)
    call("octic_power_spectrum_fwd", x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), T, D // 8, _stream())
    return y


def power_spectrum_bwd(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    T, D = x.shape
    dx = torch.empty(T, D, dtype=torch.float32, device=x.device)
    call("octic_power_spectrum_bwd", dy.data_ptr(), dy.stride(0), _dt(dy), x.data_ptr(), x.stride(0),
         dx.data_ptr(), dx.stride(0), T, D // 8, _stream())
    return dx


def bridge_permute(x: torch.Tensor) -> torch.Tensor:
    _req(x, torch.float32, "x")
    y = torch.empty_like(x)
    call("octic_bridge_permute", x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), x.shape[0], x.shape[1] // 8,
         _stream())
    return y


def im2col_patches(img: torch.Tensor, p: int) -> torch.Tensor:
    _req(img, torch.float32, "img", ndim=4)
    if not img.is_contiguous():
        raise _lib.OcticError("img must be contiguous NCHW")
    B, Cin, H, W = img.shape
    kp = roundup64(Cin * p * p)
    out = torch.empty(B * (H // p) * (W // p), kp, dtype=torch.bfloat16, device=img.device)
    call("octic_im2col_patches", img.data_ptr(), B, Cin, H, W, p, out.data_ptr(), out.stride(0), _stream())
    return out


# ----------------------------------------------------------------------------------------------------------------
# symmetric parameter expansion (lifting filters, positional embedding): sparse linear maps applied by one kernel
# ----------------------------------------------------------------------------------------------------------------
@dataclass
class SparseMap:
    """out = S in for a sparse S [n_out, n_in] with at most K entries per row, and its transpose (backward)."""
    n_in: int
    n_out: int
    k_fwd: int
    idx_fwd: torch.Tensor      # int32 [n_out, k_fwd]
    coef_fwd: torch.Tensor     # fp32  [n_out, k_fwd]
    k_bwd: int
    idx_bwd: torch.Tensor      # int32 [n_in, k_bwd]
    coef_bwd: torch.Tensor


def _tables(dense: torch.Tensor):
    nz = dense != 0
    k = max(1, int(nz.sum(1).max()))
    if k > 16:
        raise _lib.OcticError("sparse map with more than 16 entries per row")
    idx = torch.zeros(dense.shape[0], k, dtype=torch.int32)
    coef = torch.zeros(dense.shape[0], k, dtype=torch.float32)
    for o in range(dense.shape[0]):
        cols = torch.nonzero(nz[o]).flatten()
        idx[o, :cols.numel()] = cols.to(torch.int32)
        coef[o, :cols.numel()] = dense[o, cols]
    return k, idx, coef


def build_sparse_map(dense: torch.Tensor, device) -> SparseMap:
    """dense: fp32 [n_out, n_in] on the CPU (obtained by pushing a one-hot basis through the reference formula)."""
    dense = dense.detach().to("cpu", torch.float32)
    kf, idf, cf = _tables(dense)
    kb, idb, cb = _tables(dense.t().contiguous())
    return SparseMap(dense.shape[1], dense.shape[0], kf, idf.to(device), cf.to(device), kb, idb.to(device), cb.to(device))


def sparse_rowmap(inp: torch.Tensor, out: torch.Tensor, m: SparseMap, transpose: bool = False, accumulate: bool = False) -> None:
    """out[r, :] (+)= S in[r, :] (or S^T with transpose=True); inp / out: fp32 2-D with unit inner stride."""
    _req(inp, torch.float32, "inp")
    _req(out, torch.float32, "out")
    n_in, n_out = (m.n_out, m.n_in) if transpose else (m.n_in, m.n_out)
    if inp.shape[1] != n_in or out.shape != (inp.shape[0], n_out) or inp.stride(1) != 1 or out.stride(1) != 1:
        raise _lib.OcticError(f"sparse_rowmap: shapes {tuple(inp.shape)} -> {tuple(out.shape)} do not match the map")
    k, idx, coef = (m.k_bwd, m.idx_bwd, m.coef_bwd) if transpose else (m.k_fwd, m.idx_fwd, m.coef_fwd)
    call("octic_sparse_rowmap", inp.data_ptr(), inp.stride(0), out.data_ptr(), out.stride(0), inp.shape[0], n_out, k,
         idx.data_ptr(), coef.data_ptr(), int(accumulate), _stream())


def sparse_posmap(inp: torch.Tensor, out: torch.Tensor, m: SparseMap, transpose: bool = False, accumulate: bool = False) -> None:
    """out[o, :] (+)= sum_i S[o, i] in[i, :] (or S^T); inp [n_in, cols], out [n_out, cols], unit inner stride."""
    _req(inp, torch.float32, "inp")
    _req(out, torch.float32, "out")
    n_in, n_out = (m.n_out, m.n_in) if transpose else (m.n_in, m.n_out)
    if inp.shape[0] != n_in or out.shape != (n_out, inp.shape[1]) or inp.stride(1) != 1 or out.stride(1) != 1:
        raise _lib.OcticError(f"sparse_posmap: shapes {tuple(inp.shape)} -> {tuple(out.shape)} do not match the map")
    k, idx, coef = (m.k_bwd, m.idx_bwd, m.coef_bwd) if transpose else (m.k_fwd, m.idx_fwd, m.coef_fwd)
    call("octic_sparse_posmap", inp.data_ptr(), inp.stride(0), out.data_ptr(), out.stride(0), n_out, inp.shape[1], k,
         idx.data_ptr(), coef.data_ptr(), int(accumulate), _stream())


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    _req(x, torch.float32, "x")
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    call("octic_cast_f32_to_bf16", x.data_ptr(), x.stride(0), y.data_ptr(), y.stride(0), x.shape[0], x.shape[1],
         _stream())
    return y
