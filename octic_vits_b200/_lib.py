"""ctypes binding of liboctic_b200.so (the C ABI declared in include/octic_b200.h).

PyTorch is used for device memory and streams only: every call passes raw `data_ptr()`s and the current CUDA
stream handle.  There is no fallback: if the shared library is missing, or a call returns an error code, an
exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "liboctic_b200.so"

OCTIC_MAX_GROUPS = 8
F32, BF16 = 0, 1
EPI_BF16, EPI_RESID, EPI_F32, EPI_GELU_BF16, EPI_GELU_BWD = 0, 1, 2, 3, 4


class OcticError(RuntimeError):
    pass


class GemmGroup(C.Structure):
    _fields_ = [("a_col", C.c_int), ("k", C.c_int), ("b_map", C.c_int), ("b_row", C.c_int), ("n", C.c_int),
                ("c_col", C.c_int), ("bias_off", C.c_int)]


class GemmDesc(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("lda", C.c_long), ("a_cols", C.c_long), ("M", C.c_int),
        ("b0", C.c_void_p), ("b0_rows", C.c_long), ("b0_cols", C.c_long), ("b0_ld", C.c_long),
        ("b1", C.c_void_p), ("b1_rows", C.c_long), ("b1_cols", C.c_long), ("b1_ld", C.c_long),
        ("num_groups", C.c_int), ("groups", GemmGroup * OCTIC_MAX_GROUPS),
        ("block_n", C.c_int), ("mode", C.c_int),
        ("out", C.c_void_p), ("ldo", C.c_long),
        ("bias", C.c_void_p), ("gamma", C.c_void_p),
        ("resid_in", C.c_void_p), ("resid_out", C.c_void_p), ("ldr", C.c_long),
        ("row_scale", C.c_void_p), ("rows_per_sample", C.c_int),
        ("branch_out", C.c_void_p), ("ldb", C.c_long),
        ("remap_group", C.c_int), ("remap_extra", C.c_int), ("remap_off", C.c_int),
        ("head_H", C.c_int), ("head_S", C.c_int), ("head_D", C.c_int), ("head_off", C.c_int * OCTIC_MAX_GROUPS),
        ("gelu_pre", C.c_void_p), ("colsum", C.c_void_p),
    ]


class WgradGroup(C.Structure):
    _fields_ = [("dy_col", C.c_int), ("x_col", C.c_int), ("n_out", C.c_int), ("k_in", C.c_int),
                ("dw", C.c_void_p), ("ldw", C.c_long)]


class WgradDesc(C.Structure):
    _fields_ = [
        ("dy", C.c_void_p), ("ld_dy", C.c_long), ("dy_cols", C.c_long),
        ("x", C.c_void_p), ("ld_x", C.c_long), ("x_cols", C.c_long),
        ("T", C.c_int), ("num_groups", C.c_int), ("groups", WgradGroup * OCTIC_MAX_GROUPS),
        ("block_n", C.c_int), ("splits", C.c_int),
    ]


GEMM_PLAN_TN, GEMM_PLAN_WGRAD = 0, 1


class GemmPlan(C.Structure):
    """Launch plan of the last GEMM on this host thread (octic_gemm_last_plan)."""
    _fields_ = [(name, C.c_int) for name in (
        "kind", "mode", "ncta", "num_stages", "ws", "block_n", "grid", "num_m_blocks", "total_tiles", "kb_total",
        "full_rounds", "rem_tiles", "rem_splits", "splits", "packed", "direct", "roles_low")]


class LsFinSeg(C.Structure):
    _fields_ = [("dw", C.c_void_p), ("w", C.c_void_p), ("N", C.c_int), ("K", C.c_int), ("gamma", C.c_void_p),
                ("bias", C.c_void_p), ("cs", C.c_void_p), ("dgamma", C.c_void_p), ("dbias", C.c_void_p),
                ("dw_acc", C.c_void_p)]


class OptimChunk(C.Structure):
    _fields_ = [("p", C.c_void_p), ("ema", C.c_void_p), ("off", C.c_long), ("len", C.c_int), ("seg", C.c_int)]


class OptimSeg(C.Structure):
    _fields_ = [("weight_decay", C.c_float), ("lr_scale", C.c_float), ("first_chunk", C.c_int), ("num_chunks", C.c_int)]


_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_long, C.c_float

# name -> argtypes; every function returns int.  Keep in sync with include/octic_b200.h (tests check that every
# prototype in the header is exported by the library and listed here).
SIGNATURES = {
    "octic_gemm_bf16": [C.POINTER(GemmDesc), _P],
    "octic_gemm_wgrad_bf16": [C.POINTER(WgradDesc), _P],
    "octic_gemm_last_plan": [C.POINTER(GemmPlan)],
    "octic_linear_d8_pack_weights": [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P],
    "octic_linear_d8_fwd": [_P, _I, _I, _I, _P, _P, _P, C.POINTER(GemmDesc), _P],
    "octic_linear_d8_dgrad": [_P, _I, _I, _I, _P, _P, _P, _I, _P],
    "octic_linear_d8_wgrad": [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P],
    "octic_linear_pack_weights": [_P, _I, _I, _P, _P, _P],
    "octic_linear_pack_weights_scaled": [_P, _P, _I, _I, _P, _P],
    "octic_linear_d8_pack_weights_scaled": [_P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P],
    "octic_layerscale_wgrad_finalize": [C.POINTER(LsFinSeg), _I, _P],
    "octic_gelu_d8_fwd": [_P, _L, _P, _L, _L, _I, _I, _P],
    "octic_gelu_d8_bwd": [_P, _L, _P, _L, _P, _L, _L, _I, _I, _P, _P],
    "octic_gelu_bwd": [_P, _P, _P, _L, _I, _P, _P],
    "octic_layernorm_d8_fwd": [_P, _L, _P, _P, _F, _P, _L, _I, _P, _L, _I, _P],
    "octic_layernorm_d8_bwd": [_P, _L, _I, _P, _L, _P, _P, _P, _P, _L, _P, _P, _L, _I, _P, _P, _P],
    "octic_layernorm_fwd": [_P, _L, _P, _P, _F, _P, _L, _I, _P, _L, _I, _P],
    "octic_layernorm_bwd": [_P, _L, _I, _P, _L, _P, _P, _P, _P, _L, _P, _P, _L, _I, _P, _P, _P],
    "octic_layerscale_bwd": [_P, _L, _P, _L, _P, _P, _I, _P, _L, _P, _P, _L, _I, _P],
    "octic_colsum_bf16": [_P, _L, _L, _I, _P, _P],
    "octic_attention_fwd": [_P, _P, _P, _I, _I, _I, _I, _I, _P],
    "octic_attention_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "octic_attention_bwd_ws": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, C.c_size_t, _P],
    "octic_power_spectrum_fwd": [_P, _L, _P, _L, _L, _I, _P],
    "octic_power_spectrum_bwd": [_P, _L, _I, _P, _L, _P, _L, _L, _I, _P],
    "octic_bridge_permute": [_P, _L, _P, _L, _L, _I, _P],
    "octic_im2col_patches": [_P, _I, _I, _I, _I, _I, _P, _L, _P],
    "octic_cast_f32_to_bf16": [_P, _L, _P, _L, _L, _I, _P],
    "octic_sparse_rowmap": [_P, _L, _P, _L, _L, _I, _I, _P, _P, _I, _P],
    "octic_sparse_posmap": [_P, _L, _P, _L, _I, _I, _I, _P, _P, _I, _P],
    "octic_optim_sqnorm": [_P, _L, _P, _P, _P],
    "octic_optim_stage1": [_P, _I, _P, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _F, _F, _F, _I, _F, _P],
    "octic_optim_lamb_stage2": [_P, _I, _P, _I, _P, _P, _P, _F, _I, _F, _P],
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library once; fail loudly if it has not been built (python __graft_entry__.py / build.sh)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise OcticError(
            f"{LIB_PATH} not found: build it with ./build.sh (nvcc, sm_100a). There is no CPU or PyTorch fallback.")
    lib = C.CDLL(os.fspath(LIB_PATH))
    lib.octic_strerror.restype = C.c_char_p
    lib.octic_strerror.argtypes = [C.c_int]
    lib.octic_version.restype = C.c_int
    lib.octic_device_ok.restype = C.c_int
    lib.octic_attention_headmajor_supported.restype = C.c_int
    lib.octic_attention_headmajor_supported.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.octic_attention_bwd_workspace_bytes.restype = C.c_size_t
    lib.octic_attention_bwd_workspace_bytes.argtypes = [C.c_int, C.c_int]
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().octic_strerror(rc).decode()
        raise OcticError(f"{what} failed: {msg} (code {rc})")


# kernels launched by one call of each entry point (for bench.py's gpu_launches claim)
KERNELS_PER_CALL = {"octic_linear_d8_pack_weights": 5, "octic_linear_d8_pack_weights_scaled": 5, "octic_attention_bwd": 2, "octic_attention_bwd_ws": 2,
                    "octic_optim_sqnorm": 2, "octic_optim_lamb_stage2": 2}   # bwd: delta + main (legacy: +1)


class _Stats:
    """Launch counter + optional CUDA-event timing of selected entry points (used by bench.py only)."""

    def __init__(self):
        self.profile_prefixes = ()
        self.reset()

    def reset(self):
        self.kernel_launches = 0
        self.calls = {}
        self._events = []

    def collect(self):
        """(total ms, total algorithmic FLOPs, number of timed calls) of the profiled entry points; synchronises."""
        per = self.collect_by_name()
        return (sum(v[0] for v in per.values()), sum(v[1] for v in per.values()), sum(v[2] for v in per.values()))

    def collect_by_name(self):
        """{entry point: (ms, algorithmic FLOPs, calls)} of the profiled entry points; synchronises."""
        import torch
        torch.cuda.synchronize()
        per = {}
        for name, a, b, f in self._events:
            ms0, f0, n0 = per.get(name, (0.0, 0.0, 0))
            per[name] = (ms0 + a.elapsed_time(b), f0 + f, n0 + 1)
        self._events = []
        return per


STATS = _Stats()


def call(name: str, *args, flops: float = 0.0, extra_kernels: int = 0, stat: str = "") -> None:
    """`stat`: the name the call is counted / timed under when it differs from the entry point (e.g. the `_ws` flavour
    of an op keeps the op's name in event tables)."""
    fn = getattr(load(), name)
    STATS.kernel_launches += KERNELS_PER_CALL.get(name, 1) + extra_kernels
    name = stat or name
    STATS.calls[name] = STATS.calls.get(name, 0) + 1
    if STATS.profile_prefixes and name in STATS.profile_prefixes:
        import torch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = fn(*args)
        b.record()
        STATS._events.append((name, a, b, flops))
    else:
        rc = fn(*args)
    check(rc, name)
