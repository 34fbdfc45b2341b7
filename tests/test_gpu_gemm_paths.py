"""Every dispatch path of the tcgen05 GEMM engine (gemm_sm100.cu) against an fp64 reference of the same operation.

Each case names the code path it guards and asserts the launch plan the engine recorded for it
(ops.last_gemm_plan()): when a re-tune of the launch policy moves a shape off its path, the case fails and the shape
has to be chosen again.  Expected values derive from the device's SM count, never from a hard-coded 148.

Reference and bound.  The reference is fp64 on the bf16 operands the kernel consumes, with the epilogue applied at
the kernel's rounding points (bias, bf16 rounding, then gamma, the DropPath factor, the residual, GELU).  Every element
must satisfy

    |got - ref| <= EPS_OUT * |ref| + EPS_ACC * (|A| |B|^T)      (scaled by the epilogue factors that follow the GEMM)

with EPS_OUT = 2^-7 for bf16-valued outputs (bf16's unit roundoff is 2^-8: one rounding, plus a rounding point the
kernel may take one ulp the other way) and a few fp32 ulps for fp32 outputs.  Each case also shows that its bound
has teeth: references with one 64-wide k-block dropped, with the last tile's columns shifted by one and (with a
DropPath factor) with two samples' factors swapped must FAIL the same bound on the same data.

Canaries.  Every destination is a view inside a larger buffer filled with a NaN bit pattern (rows above and below,
columns left and right, a leading dimension wider than the view); after the call everything outside the elements the
launch owns must be bit-identical.  Stray writes are caught in bounds, without provoking a fault.

The OCTIC_GEMM_* / OCTIC_BLOCK_N switches are cached in function-local statics of the library, so the `core` cases
are re-run in a child process per switch (test_switch_configuration), where they also assert that the switch took
effect through the plan.
"""
import math
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from octic_vits_b200 import ops
    from octic_vits_b200._lib import EPI_BF16, EPI_F32, EPI_GELU_BF16, EPI_GELU_BWD, EPI_RESID
from octic_vits_b200 import _lib
from octic_vits_b200._lib import OcticError

DEV = "cuda"
ROOT = Path(__file__).resolve().parents[1]

EPS_BF16 = 2.0 ** -7          # one bf16 ulp: a rounding (unit roundoff 2^-8) plus a 1-ulp different rounding point
EPS_F32 = 2.0 ** -22          # the fp32 adds after the accumulator (bias, residual, red.add of partial sums)
# fp32 accumulation error per unit of |A| |B|^T.  The ratio a case needs is printed per case ("eps_acc needed"); on a
# B200 (1000 W power limit) the largest over the file was 5.2e-7 = 2^-20.9 (wgrad_full_rounds_only, T = 4099; the tn
# cases stay below 2^-23.8).  EPS_ACC is 2^2.9 = ~7.5x that largest ratio.
EPS_ACC = 2.0 ** -18
GELU_LIP = 1.13               # max |gelu'|: how far a 1-ulp different bf16 pre-activation moves gelu
EPS_GELU = 2.0 ** -20         # A&S 7.1.26 erf (|err| <= 1.5e-7) and fp32 cancellation of x + |x| erf, per unit (1 + |x|)

PAT16 = 0x7FA5                # bf16 NaN with a payload no kernel computes
PAT32 = 0x7FA5A5A5            # fp32 NaN, likewise

SWITCH_ENV = ("OCTIC_GEMM_NCTA", "OCTIC_GEMM_WS", "OCTIC_GEMM_PACKED", "OCTIC_GEMM_DIRECT", "OCTIC_GEMM_STAGES",
              "OCTIC_GEMM_ROLES_HIGH", "OCTIC_BLOCK_N")
SWITCH = {k: os.environ[k] for k in SWITCH_ENV if k in os.environ}

# gemm_sm100.cu constants the expected ring depths derive from
K_MAX_DYN_SMEM, K_A_STAGE, K_MAX_STAGES = 232448, 128 * 64 * 2, 8


def setup_module(module):
    torch.backends.cuda.matmul.allow_tf32 = False


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def tn_max_stages(block_n, ncta):
    fixed = 1024 + 16 * 32 * 36 * 4 + (2 * K_MAX_STAGES + 4) * 8 + 16 + 16
    return min(K_MAX_STAGES, (K_MAX_DYN_SMEM - fixed) // (K_A_STAGE + block_n // ncta * 64 * 2))


def gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def bf_randn(shape, seed, scale=1.0):
    return (torch.randn(*shape, generator=gen(seed)) * scale).to(torch.bfloat16).to(DEV)


# ------------------------------------------------------------------------------------------------------------------
# canaries
# ------------------------------------------------------------------------------------------------------------------
class Canvas:
    """A [rows, cols] destination view inside a larger buffer whose every element starts as a NaN bit pattern: `top`
    rows above, `bottom` below, `left` columns before, and a row stride `ld` > left + cols (the right margin)."""

    def __init__(self, rows, cols, dtype, top=2, bottom=3, left=8, right=24, ld=None):
        self.dtype, self.top, self.left, self.rows, self.cols = dtype, top, left, rows, cols
        self.ld = ld if ld is not None else (left + cols + right + 7) // 8 * 8
        assert self.ld >= left + cols
        self.buf = torch.empty(top + rows + bottom, self.ld, dtype=dtype, device=DEV)
        self.bits().fill_(PAT16 if dtype == torch.bfloat16 else PAT32)
        self.view = self.buf[top:top + rows, left:left + cols]

    def bits(self):
        return self.buf.view(torch.int16 if self.dtype == torch.bfloat16 else torch.int32)

    def assert_untouched_outside(self, rows=None, cols=None, what="out"):
        """Everything but view[rows][:, cols] (default: the whole view) still holds the pattern, bit for bit."""
        mask = torch.zeros(self.buf.shape, dtype=torch.bool, device=DEV)
        r = torch.arange(self.rows, device=DEV) if rows is None else rows
        c = torch.arange(self.cols, device=DEV) if cols is None else cols
        mask[(self.top + r)[:, None], (self.left + c)[None, :]] = True
        pat = PAT16 if self.dtype == torch.bfloat16 else PAT32
        bad = (self.bits() != pat) & ~mask
        n = int(bad.sum())
        if n:
            idx = bad.nonzero()[:4].tolist()
            raise AssertionError(f"{what}: {n} elements written outside the destination, e.g. buffer [row, col] {idx} "
                                 f"(view starts at [{self.top}, {self.left}], {self.rows} x {self.cols})")


# ------------------------------------------------------------------------------------------------------------------
# fp64 references and the bound
# ------------------------------------------------------------------------------------------------------------------
class Grp:
    """One GEMM group as the reference sees it: out[:, c_col + j] = sum_k a[:, a_col + k] * w[j, k] (+ bias[j])."""

    def __init__(self, a_col, k, w, c_col, bias=None):
        self.a_col, self.k, self.w, self.c_col, self.bias = a_col, k, w, c_col, bias
        self.n = w.shape[0]


def ref_acc(a, groups, width, drop_kblock=False):
    """acc = a @ w^T per group (fp64) and |a| @ |w|^T, [M, width]; drop_kblock: group 0 loses its first 64 columns."""
    M = a.shape[0]
    acc = torch.zeros(M, width, dtype=torch.float64, device=DEV)
    mag = torch.zeros_like(acc)
    for i, g in enumerate(groups):
        ag = a[:, g.a_col:g.a_col + g.k].double()
        if drop_kblock and i == 0:
            ag = ag.clone()
            ag[:, :64] = 0
        w = g.w.double()
        acc[:, g.c_col:g.c_col + g.n] = ag @ w.T
        mag[:, g.c_col:g.c_col + g.n] = ag.abs() @ w.abs().T
    return acc, mag


def bias_row(groups, width):
    b = torch.zeros(width, dtype=torch.float64, device=DEV)
    for g in groups:
        if g.bias is not None:
            b[g.c_col:g.c_col + g.n] = g.bias.double()
    return b


def shift_cols(t, cols):
    """t with columns `cols` (one tile) replaced by their left neighbours: a tile written one column off."""
    t = t.clone()
    t[:, cols] = t[:, cols - 1] if int(cols[0]) > 0 else t[:, cols.roll(1)]
    return t


def last_tile_cols(groups, block_n):
    g = max(groups, key=lambda g: g.c_col)
    n0 = (g.n - 1) // block_n * block_n
    return torch.arange(g.c_col + n0, g.c_col + g.n, device=DEV)


class Stats:
    """Largest |got - ref| / bound and the EPS_ACC a case needs beyond its rounding term, printed once per case."""

    def __init__(self):
        self.ratio, self.eps_acc = 0.0, 0.0

    def report(self, name):
        print(f"\n[{name}] worst |err|/bound {self.ratio:.3e}   eps_acc needed {self.eps_acc:.3e} "
              f"(= 2^{math.log2(self.eps_acc) if self.eps_acc > 0 else float('-inf'):.1f}, bound uses 2^{math.log2(EPS_ACC):.0f})")


def within(got, ref, rnd, acc_unit):
    """Element-wise |got - ref| <= rnd + EPS_ACC * acc_unit (NaN fails).  Returns (ok, ratio, eps_acc needed)."""
    err = (got.double() - ref).abs()
    bound = rnd + EPS_ACC * acc_unit
    ok = bool((err <= bound).all())
    ratio = float((err / bound.clamp_min(1e-300)).nan_to_num(float("inf")).max()) if err.numel() else 0.0
    need = float(((err - rnd).clamp_min(0) / acc_unit.clamp_min(1e-300)).nan_to_num(float("inf")).max()) if err.numel() else 0.0
    return ok, ratio, need


def verify(name, outputs_for, perturbations):
    """outputs_for(**perturbation) -> [(label, got, ref, rnd, acc_unit)].  The true reference must pass every output;
    every perturbed one must fail at least one."""
    st = Stats()
    for label, got, ref, rnd, unit in outputs_for():
        ok, ratio, need = within(got, ref, rnd, unit)
        st.ratio, st.eps_acc = max(st.ratio, ratio), max(st.eps_acc, need)
        if not ok:
            err = (got.double() - ref).abs() - (rnd + EPS_ACC * unit)
            i = int(err.nan_to_num(float("inf")).argmax())
            idx = [int(v) for v in torch.unravel_index(torch.tensor(i), err.shape)] if err.dim() > 0 else []
            raise AssertionError(f"{name}/{label}: outside the bound at {idx}: got {float(got.reshape(-1)[i])} "
                                 f"want {float(ref.reshape(-1)[i])} (worst |err|/bound {ratio:.3g})")
    for pname, kw in perturbations:
        caught = any(not within(got, ref, rnd, unit)[0] for _, got, ref, rnd, unit in outputs_for(**kw))
        assert caught, f"{name}: the bound does not reject the perturbed reference '{pname}'"
    st.report(name)
    return st


def teeth(groups, block_n, row_scale=None):
    p = [("k-block dropped", {"drop": True}), ("last tile shifted", {"shift": last_tile_cols(groups, block_n)})]
    if row_scale is not None:
        rs = row_scale.clone()
        j = int((rs != rs[0]).nonzero()[0])
        rs[0], rs[j] = row_scale[j], row_scale[0]
        p.append(("row_scale swapped", {"rs": rs}))
    return p


# ------------------------------------------------------------------------------------------------------------------
# plans
# ------------------------------------------------------------------------------------------------------------------
def plan():
    return ops.last_gemm_plan()


def expect(pl, **want):
    """The default-policy path of a case.  Under a switch the launch is on the switch's path instead (check_switch)."""
    if SWITCH:
        return
    got = {k: pl[k] for k in want}
    assert got == want, f"launch plan moved off the path this case guards: {got} != {want} (full plan {pl})"


def check_switch(pl, grouped_small_k=False, pairs_possible=False, d8=False):
    """Inside a switch configuration: assert that the switch reached this launch."""
    e = SWITCH
    if e.get("OCTIC_GEMM_NCTA") == "1":
        assert pl["ncta"] == 1, pl
    if e.get("OCTIC_GEMM_NCTA") == "2" and pl["kind"] == _lib.GEMM_PLAN_TN and pairs_possible:
        assert pl["ncta"] == 2, pl
    if e.get("OCTIC_GEMM_WS") == "1" and pl["kind"] == _lib.GEMM_PLAN_TN and grouped_small_k and pairs_possible:
        assert pl["ws"] == 1 and pl["ncta"] == 2, pl
    if e.get("OCTIC_GEMM_PACKED") == "0" and pl["kind"] == _lib.GEMM_PLAN_TN:
        assert pl["packed"] == 0, pl
    if "OCTIC_GEMM_DIRECT" in e and pl["kind"] == _lib.GEMM_PLAN_TN:
        assert pl["direct"] == (int(e["OCTIC_GEMM_DIRECT"]) >> pl["mode"]) & 1, pl
    if "OCTIC_GEMM_STAGES" in e and pl["kind"] == _lib.GEMM_PLAN_TN:
        assert pl["num_stages"] <= int(e["OCTIC_GEMM_STAGES"]), pl
    if e.get("OCTIC_GEMM_ROLES_HIGH") == "1":
        assert pl["roles_low"] == 0, pl
    if "OCTIC_BLOCK_N" in e and d8:
        assert pl["block_n"] == int(e["OCTIC_BLOCK_N"]), pl


# ------------------------------------------------------------------------------------------------------------------
# tn GEMM: launch + outputs
# ------------------------------------------------------------------------------------------------------------------
def d8_weights(ci, co, seed, bias=True):
    g = gen(seed)
    w1 = [torch.randn(co, ci, generator=g) / math.sqrt(ci) for _ in range(4)]
    wE = torch.randn(2 * co, 2 * ci, generator=g) / math.sqrt(2 * ci)
    b = torch.randn(co, generator=g).to(DEV) if bias else None
    pk = ops.pack_linear_d8(*(w.to(DEV).contiguous() for w in w1 + [wE]))
    w1 = [w.to(torch.bfloat16).to(DEV) for w in w1]
    wE = wE.to(torch.bfloat16).to(DEV)
    # LinearD8 as the header defines it: five block-diagonal linears over [A1 | A2 | B1 | B2 | E0 | E1]
    groups = [Grp(i * ci, ci, w1[i], i * co, b if i == 0 else None) for i in range(4)]
    groups += [Grp(4 * ci + r * 2 * ci, 2 * ci, wE, 4 * co + r * 2 * co) for r in range(2)]
    return pk, groups


def dense_weights(n, k, seed, bias=True):
    g = gen(seed)
    w = torch.randn(n, k, generator=g) / math.sqrt(k)
    b = torch.randn(n, generator=g).to(DEV) if bias else None
    pk = ops.pack_linear(w.to(DEV).contiguous())
    return pk, [Grp(0, k, w.to(torch.bfloat16).to(DEV), 0, b)]


def head_perm(width, S, H):
    """logical (packed) column -> head-major column of a LinearD8 forward with head remap: feature [s][h][j] of the
    irrep group with c_g = Co/(S*H) columns per head goes to s*D/S... (see octic_gemm_desc.head_*)."""
    co = width // 8
    ch = co // (S * H)
    hd_s = width // S                       # head_D: columns per S slice
    offs = [0, ch, 2 * ch, 3 * ch, 4 * ch, 6 * ch]
    ns = [co] * 4 + [2 * co] * 2
    ccol = [0, co, 2 * co, 3 * co, 4 * co, 6 * co]
    perm = torch.empty(width, dtype=torch.long)
    for g in range(6):
        cg_all = ns[g] // S
        cg = cg_all // H
        for n in range(ns[g]):
            s_, rem = divmod(n, cg_all)
            h_, j_ = divmod(rem, cg)
            perm[ccol[g] + n] = s_ * hd_s + h_ * (hd_s // H) + offs[g] + j_
    return perm.to(DEV)


def run_tn(name, *, a, groups, width, mode, launch, block_n_hint, M=None, bias_rows=None, gamma=None, resid=None,
           row_scale=None, rps=1, branch=False, in_place=False, colsum=False, gelu_pre=None, col_perm=None,
           remap=(0, 0, 0), out_rows=None, left=8):
    """Allocate canvases, launch, then check every output against the fp64 reference and its perturbations.
    launch(**epi) runs the GEMM with the epilogue keyword arguments of ops._epilogue_desc; returns the plan."""
    M = a.shape[0] if M is None else M
    rows_out = M if out_rows is None else out_rows
    # row r of the GEMM lands on out row mo(r) (patch-embed remap)
    m = torch.arange(M, device=DEV)
    mo = m + (m // remap[0]) * remap[1] + remap[2] if remap[0] else m
    cols_phys = torch.arange(width, device=DEV) if col_perm is None else col_perm
    epi = {"remap": remap} if remap[0] else {}
    canv = {}
    if mode == EPI_RESID:
        base = torch.randn(rows_out, width, generator=gen(99)).to(DEV)
        canv["resid_out"] = Canvas(rows_out, width, torch.float32, left=left)
        if in_place:
            canv["resid_out"].view.copy_(base)
            epi["resid_in"] = canv["resid_out"].view
        elif resid:
            rin = torch.empty_like(canv["resid_out"].buf).normal_()     # same row stride (the descriptor has one ldr)
            rin_view = rin[canv["resid_out"].top:canv["resid_out"].top + rows_out, left:left + width]
            rin_view.copy_(base)
            epi["resid_in"] = rin_view
        else:
            base = torch.zeros_like(base)
        epi["resid_out"] = canv["resid_out"].view
        if gamma is not None:
            epi["gamma"] = gamma
        if row_scale is not None:
            epi["row_scale"], epi["rows_per_sample"] = row_scale, rps
        if branch:
            canv["branch_out"] = Canvas(rows_out, width, torch.bfloat16, top=1, bottom=2, left=left, right=40)
            epi["branch_out"] = canv["branch_out"].view
    else:
        dt = torch.float32 if mode == EPI_F32 else torch.bfloat16
        canv["out"] = Canvas(rows_out, width, dt, left=left)
        epi["out"] = canv["out"].view
        if mode == EPI_GELU_BF16 and branch:
            canv["branch_out"] = Canvas(rows_out, width, torch.bfloat16, left=left, ld=canv["out"].ld)
            epi["branch_out"] = canv["branch_out"].view
        if mode == EPI_GELU_BWD:
            pre_buf = torch.zeros_like(canv["out"].buf)
            pre_view = pre_buf[canv["out"].top:canv["out"].top + rows_out, left:left + width]
            pre_view.copy_(gelu_pre)
            epi["gelu_pre"] = pre_view
            if colsum:
                cs = Canvas(1, width, torch.float32, top=0, bottom=1, left=8, right=24)
                cs.view.zero_()
                canv["colsum"] = cs
                epi["colsum"] = cs.view[0]
    pl = launch(**epi)
    torch.cuda.synchronize()

    for key, c in canv.items():
        if key == "colsum":
            c.assert_untouched_outside(torch.tensor([0], device=DEV), cols_phys, what=key)
        else:
            c.assert_untouched_outside(mo, cols_phys, what=key)

    def got_of(key):
        v = canv[key].view if key != "colsum" else canv[key].view[0]
        if key == "colsum":
            return v[cols_phys]
        return v[mo][:, cols_phys]

    bias = bias_row(groups, width)

    def outputs_for(drop=False, shift=None, rs=None):
        acc, mag = ref_acc(a, groups, width, drop_kblock=drop)
        y = acc + bias
        if shift is not None:
            y, mag = shift_cols(y, shift), shift_cols(mag, shift)
        outs = []
        if mode == EPI_BF16:
            outs.append(("out", got_of("out"), y, EPS_BF16 * y.abs(), mag))
        elif mode == EPI_F32:
            outs.append(("out", got_of("out"), y, EPS_F32 * y.abs(), mag))
        elif mode == EPI_GELU_BF16:
            pre = y.to(torch.bfloat16).double()            # the kernel's rounding point (1 ulp either way is in the bound)
            g = torch.nn.functional.gelu(pre)
            outs.append(("out", got_of("out"), g,
                         EPS_BF16 * g.abs() + GELU_LIP * EPS_BF16 * y.abs() + EPS_GELU * (1 + y.abs()), GELU_LIP * mag))
            if branch:
                outs.append(("branch_out", got_of("branch_out"), y, EPS_BF16 * y.abs(), mag))
        elif mode == EPI_GELU_BWD:
            p = gelu_pre.double()
            cdf = 0.5 * (1 + torch.erf(p / math.sqrt(2)))
            gp = cdf + p * torch.exp(-0.5 * p * p) / math.sqrt(2 * math.pi)
            d = y * gp
            unit = mag * (gp.abs() + EPS_GELU / EPS_ACC)
            outs.append(("out", got_of("out"), d, EPS_BF16 * d.abs(), unit))
            if colsum:
                outs.append(("colsum", got_of("colsum"), d.sum(0), EPS_F32 * M * d.abs().sum(0), unit.sum(0)))
        else:
            r = row_scale if rs is None else rs
            sc = torch.ones(M, dtype=torch.float64, device=DEV) if r is None else r.double()[mo // rps]
            gm = torch.ones(width, dtype=torch.float64, device=DEV) if gamma is None else gamma.double()
            f = (sc[:, None] * gm[None, :]).abs()
            yb = y.to(torch.bfloat16).double()               # the Linear emits bf16 (1 ulp either way is in the bound)
            want = base.double()[mo] + sc[:, None] * gm[None, :] * yb
            rnd = f * EPS_BF16 * y.abs() + EPS_F32 * (want.abs() + base.double()[mo].abs())
            outs.append(("resid_out", got_of("resid_out"), want, rnd, f * mag))
            if branch:
                outs.append(("branch_out", got_of("branch_out"), y, EPS_BF16 * y.abs(), mag))
        return outs

    verify(name, outputs_for, teeth(groups, block_n_hint(pl), row_scale))
    return pl


def d8_launch(x, pk, bias, mode):
    def launch(**epi):
        ops.linear_d8(x, pk, bias, mode, **epi)
        return plan()
    return launch


def dense_launch(x, pk, n, k, bias, mode):
    def launch(**epi):
        ops.linear_dense(x, pk.w, n, k, bias, mode, **epi)
        return plan()
    return launch


def gp(pl):
    return pl["block_n"]


# LinearD8 forward cases: (name, T, Ci, Co, mode, options, expected plan given sms)
def _d8_case(name, T, ci, co, mode, expected, head=None, rps=None, in_place=False, seed=0):
    x = bf_randn((T, 8 * ci), seed)
    pk, groups = d8_weights(ci, co, seed + 1)
    bias = groups[0].bias
    width = 8 * co
    kw = {}
    col_perm = None
    if mode == EPI_RESID:
        kw.update(gamma=torch.randn(width, generator=gen(seed + 2)).to(DEV), resid=True, branch=not in_place,
                  in_place=in_place)
        if rps is not None:
            nsmp = (T + rps - 1) // rps
            rs = torch.where(torch.rand(nsmp, generator=gen(seed + 3)) < 0.3, 0.0, 1.0 / 0.7)
            rs[0], rs[-1] = 0.0, 1.0 / 0.7
            kw.update(row_scale=rs.to(DEV), rps=rps)
    launch = d8_launch(x, pk, bias, mode)
    if head is not None:
        S, H = head
        col_perm = head_perm(width, S, H)
        inner = launch

        def launch(**epi):
            return inner(head=(H, S), **epi)
    pl = run_tn(name, a=x, groups=groups, width=width, mode=mode, launch=launch, block_n_hint=gp, col_perm=col_perm, **kw)
    kmax = 2 * ci
    check_switch(pl, grouped_small_k=kmax <= 320, pairs_possible=T > 128 and pl["block_n"] >= 32, d8=True)
    expect(pl, **expected)
    return pl


@pytest.mark.parametrize("name", [
    "d8_exact_bn144", "d8_exact_bn128_k40", "core_d8_wide_ragged_co480", "d8_wide_ragged_co640", "d8_kmax512_pairs",
    "d8_resid_grouped_k640_4stages", "d8_head_major_bn128", "core_d8_head_major_exact", "core_d8_unaligned_co132",
    "d8_m1_bf16_single"])
def test_linear_d8_paths(name):
    if name == "d8_exact_bn144":           # exact block_n 144, ragged-free, single CTA, deepest ring
        _d8_case(name, 300, 48, 144, EPI_BF16, dict(ncta=1, block_n=144, num_stages=tn_max_stages(144, 1), ws=0))
    elif name == "d8_exact_bn128_k40":     # exact block_n 128, K = 40 / 80 (not multiples of 64)
        _d8_case(name, 255, 40, 128, EPI_BF16, dict(ncta=1, block_n=128, num_stages=tn_max_stages(128, 1)))
    elif name == "core_d8_wide_ragged_co480":   # wide_small_k pairs, 256-column tiles with a ragged last tile (480 = 256 + 224)
        _d8_case(name, 514, 160, 480, EPI_BF16, dict(ncta=2, block_n=256, num_stages=tn_max_stages(256, 2)))
    elif name == "d8_wide_ragged_co640":   # 640 = 2 * 256 + 128
        _d8_case(name, 300, 160, 640, EPI_BF16, dict(ncta=2, block_n=256, num_stages=tn_max_stages(256, 2)))
    elif name == "d8_kmax512_pairs":       # kmax >= 512 takes pairs (block_n 160 exact)
        _d8_case(name, 257, 256, 160, EPI_BF16, dict(ncta=2, block_n=160, num_stages=tn_max_stages(160, 2)))
    elif name == "d8_resid_grouped_k640_4stages":   # fc2 + residual: grouped EPI_RESID, K = 640, pairs, ring capped at 4
        _d8_case(name, 2 * 257, 320, 160, EPI_RESID, dict(ncta=2, block_n=160, num_stages=4), rps=257)
    elif name == "d8_head_major_bn128":    # qkv head-major: 128-column tile rule, pairs, 3-stage ring
        _d8_case(name, 2 * 197, 160, 480, EPI_BF16, dict(ncta=2, block_n=128, num_stages=3), head=(3, 16))
    elif name == "core_d8_head_major_exact":    # head-major with the exact tile rule (block_n 192)
        _d8_case(name, 257, 64, 192, EPI_BF16, dict(ncta=2, block_n=192, num_stages=3), head=(3, 4))
    elif name == "core_d8_unaligned_co132":    # Co % 8 != 0: unaligned c_col, n % 32 != 0, K = 32 / 64: staged path
        _d8_case(name, 129, 32, 132, EPI_BF16, dict(ncta=2, block_n=256))
    elif name == "d8_m1_bf16_single":      # M = 1: pairs impossible
        _d8_case(name, 1, 160, 160, EPI_BF16, dict(ncta=1, num_m_blocks=1, total_tiles=8))


@pytest.mark.parametrize("rps", [1, 7, 31, 32, 33, 257])
def test_core_d8_residual_row_scale(rps):
    """Octic proj + residual: grouped EPI_RESID with K = 320 on single CTAs and a 2-stage ring; the DropPath factor
    per sample of rps rows, zeros among the factors (rps = 1 is the DINOv2 concatenated-crop form)."""
    _d8_case(f"core_d8_resid_k320_rps{rps}", 3 * 257 + 5, 160, 160, EPI_RESID, dict(ncta=1, block_n=160, num_stages=2),
             rps=rps)


def test_core_d8_residual_in_place():
    """resid_in is resid_out (the inference form)."""
    _d8_case("core_d8_resid_in_place", 600, 40, 160, EPI_RESID, dict(ncta=1, num_stages=2), in_place=True)


def test_misaligned_operand_columns_are_refused():
    """The TMA box of a group starts at its first A column (dY / X columns for the weight gradient): it must sit on a
    16-byte boundary, so Din / 8 = 20 (a_col = 20, 40, ...) is refused instead of launching a load that never lands."""
    x = bf_randn((129, 160), 0)
    pk, _ = d8_weights(20, 9, 1)
    out = torch.empty(129, 72, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(OcticError, match="16-byte"):
        ops.linear_d8(x, pk, None, EPI_BF16, out=out)
    dy = bf_randn((129, 72), 2)
    with pytest.raises(OcticError, match="16-byte"):
        ops.linear_d8_wgrad(dy, x, 160, 72)


def test_linear_d8_head_major_refused_shapes():
    """c_h = Co / (S * H) must be even: the C ABI refuses instead of writing a wrong layout."""
    x = bf_randn((64, 8 * 48), 0)
    pk, _ = d8_weights(48, 48, 1)
    out = torch.empty(64, 8 * 48, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(OcticError):
        ops.linear_d8(x, pk, None, EPI_BF16, out=out, head=(16, 3))       # c_h = 1


# dense (one group): pairs whenever M > 128
@pytest.mark.parametrize("name", ["dense_resid_rps7_m1000", "dense_resid_m257", "dense_gelu_m255", "core_dense_gelu_bwd_m1000",
                                  "dense_f32_m129_k200", "dense_bf16_m257", "m1_bf16", "m31_resid_rps1", "core_m33_f32",
                                  "m127_gelu", "m128_gelu_bwd"])
def test_dense_paths(name):
    spec = {
        # name: (M, K, N, mode, extra)
        "dense_resid_rps7_m1000": (1000, 384, 320, EPI_RESID, dict(rps=7)),
        "dense_resid_m257": (257, 640, 160, EPI_RESID, dict(rps=32)),
        "dense_gelu_m255": (255, 256, 512, EPI_GELU_BF16, {}),
        "core_dense_gelu_bwd_m1000": (1000, 320, 1000, EPI_GELU_BWD, {}),
        "dense_f32_m129_k200": (129, 200, 96, EPI_F32, {}),
        "dense_bf16_m257": (257, 64, 48, EPI_BF16, {}),
        "m1_bf16": (1, 192, 160, EPI_BF16, {}),
        "m31_resid_rps1": (31, 128, 96, EPI_RESID, dict(rps=1)),
        "core_m33_f32": (33, 104, 40, EPI_F32, {}),
        "m127_gelu": (127, 320, 200, EPI_GELU_BF16, {}),
        "m128_gelu_bwd": (128, 96, 72, EPI_GELU_BWD, {}),
    }[name]
    M, K, N, mode, extra = spec
    seed = M + K + N
    x = bf_randn((M, K), seed)
    bias_on = mode != EPI_GELU_BWD
    pk, groups = dense_weights(N, K, seed + 1, bias=bias_on)
    kw = {}
    if mode == EPI_RESID:
        kw.update(gamma=torch.randn(N, generator=gen(seed + 2)).to(DEV), resid=True, branch=True)
        rps = extra["rps"]
        nsmp = (M + rps - 1) // rps
        rs = torch.where(torch.rand(nsmp, generator=gen(seed + 3)) < 0.3, 0.0, 1.25)
        rs[0], rs[-1] = 0.0, 1.25
        kw.update(row_scale=rs.to(DEV), rps=rps)
    if mode == EPI_GELU_BF16:
        kw.update(branch=True)
    if mode == EPI_GELU_BWD:
        pre = (torch.rand(M, N, generator=gen(seed + 4)) * 12 - 6).to(torch.bfloat16).to(DEV)   # spans +-6
        kw.update(gelu_pre=pre, colsum=True)
    if mode == EPI_RESID and M == 31:
        # the single-sample swap of teeth() needs two distinct factors among the samples that exist
        kw["row_scale"] = torch.tensor([0.0 if i % 2 else 1.25 for i in range(M)], device=DEV)
    pl = run_tn(name, a=x, groups=groups, width=N, mode=mode, launch=dense_launch(x, pk, N, K, groups[0].bias, mode),
                block_n_hint=gp, **kw)
    pairs_possible = M > 128 and pl["block_n"] >= 32
    check_switch(pl, pairs_possible=pairs_possible)
    ncta = 2 if pairs_possible else 1
    # the residual epilogue with K <= 320 runs a 2-stage ring (epilogue-paced); everything else the deepest one
    stages = 2 if mode == EPI_RESID and K <= 320 else tn_max_stages(pl["block_n"], ncta)
    expect(pl, ncta=ncta, num_stages=stages, mode=mode)


def test_gelu_branch_with_its_own_stride_is_refused():
    """EPI_GELU_BF16 stores its pre-activation copy with the row stride of out: a different ldb is refused."""
    x = bf_randn((200, 64), 0)
    pk, groups = dense_weights(64, 64, 1)
    out = torch.empty(200, 64, dtype=torch.bfloat16, device=DEV)
    pre = torch.empty(200, 72, dtype=torch.bfloat16, device=DEV)[:, :64]
    with pytest.raises(OcticError):
        ops.linear_dense(x, pk.w, 64, 64, groups[0].bias, EPI_GELU_BF16, out=out, branch_out=pre)


@pytest.mark.parametrize("mode_name", ["resid", "f32"])
@pytest.mark.parametrize("lead", [1, 5])
def test_core_patch_embed_row_remap(mode_name, lead):
    """Patch embedding: GEMM row m of image b lands on token row b * (npatch + lead) + lead + m % npatch; the lead
    (cls / register) rows of every image stay untouched.  x comes from im2col, wider than K with zero pad columns."""
    B, p, npatch = 3, 14, 49
    img = torch.randn(B, 3, 7 * p, 7 * p, generator=gen(lead)).to(DEV)
    x = ops.im2col_patches(img, p)                                  # [B * 49, 640], K = 588
    K, N = 3 * p * p, 160
    assert x.shape[1] == 640 and bool((x[:, K:] == 0).all())
    pk, groups = dense_weights(N, K, 7 + lead)
    mode = EPI_RESID if mode_name == "resid" else EPI_F32
    kw = dict(resid=True, gamma=torch.randn(N, generator=gen(3)).to(DEV), branch=True) if mode == EPI_RESID else {}
    pl = run_tn(f"core_patch_embed_{mode_name}_lead{lead}", a=x, groups=groups, width=N, mode=mode,
                launch=dense_launch(x, pk, N, K, groups[0].bias, mode), block_n_hint=gp,
                remap=(npatch, lead, lead), out_rows=B * (npatch + lead), **kw)
    check_switch(pl, pairs_possible=True)
    expect(pl, ncta=2, mode=mode)


# ------------------------------------------------------------------------------------------------------------------
# weight gradient
# ------------------------------------------------------------------------------------------------------------------
def wgrad_raw(dy, x, groups, block_n, splits=0):
    """octic_gemm_wgrad_bf16 with explicit groups: [(dy_col, x_col, n_out, k_in, dw view)]."""
    d = _lib.WgradDesc()
    d.dy, d.ld_dy, d.dy_cols = dy.data_ptr(), dy.stride(0), dy.shape[1]
    d.x, d.ld_x, d.x_cols = x.data_ptr(), x.stride(0), x.shape[1]
    d.T = x.shape[0]
    d.num_groups = len(groups)
    for i, (dc, xc, n, k, dw) in enumerate(groups):
        g = d.groups[i]
        g.dy_col, g.x_col, g.n_out, g.k_in, g.dw, g.ldw = dc, xc, n, k, dw.data_ptr(), dw.stride(0)
    d.block_n, d.splits = block_n, splits
    _lib.call("octic_gemm_wgrad_bf16", _lib.C.byref(d), ops._stream())


def wgrad_plan_expected(tiles, T, ncta, splits):
    """The work split the wgrad launch documents (gemm_wgrad_kernel): CTA (pair) count, full rounds, remainder."""
    kb = (T + 63) // 64
    ncl = sms() // ncta
    if splits > 0 and tiles * splits < ncl:
        ncl = tiles * splits
    ncl = max(1, min(ncl, (tiles * kb + 3) // 4))
    return kb, ncl, tiles // ncl, tiles % ncl


def verify_wgrad(name, dy, x, parts, preload, canvases, block_n):
    """parts: [(dy_col, x_col, n_out, k_in, target index)]; targets accumulate (two E-row groups share one)."""
    torch.cuda.synchronize()
    for c, rows, cols in canvases:
        c.assert_untouched_outside(rows, cols, what="dw")

    def outputs_for(drop=False, shift=None, rs=None):
        outs = []
        for t, (pre, got) in enumerate(preload):
            acc = pre.double().clone()
            mag = torch.zeros_like(acc)
            for dc, xc, n, k, ti in parts:
                if ti != t:
                    continue
                dyp = dy[:, dc:dc + n].double()
                xp = x[:, xc:xc + k].double()
                if drop:
                    dyp = dyp.clone()
                    dyp[:64] = 0
                acc += dyp.T @ xp
                mag += dyp.abs().T @ xp.abs()
            if shift is not None:
                k = acc.shape[1]
                cols = torch.arange((k - 1) // block_n * block_n, k, device=DEV)
                acc, mag = shift_cols(acc, cols), shift_cols(mag, cols)
            outs.append((f"dw{t}", got, acc, EPS_F32 * (acc.abs() + pre.double().abs()), mag))
        return outs

    verify(name, outputs_for, [("k-block dropped", {"drop": True}), ("last tile shifted", {"shift": True})])


def _wgrad_dense_case(name, T, n, k, block_n, splits=0, ld_extra=8, via_ops=False, seed=0):
    dy = bf_randn((T, n + 8), seed)                      # row strides wider than the columns used
    x = bf_randn((T, (k + 7) // 8 * 8 + 8), seed + 1)
    c = Canvas(n, k, torch.float32, left=4, right=ld_extra, ld=4 + k + ld_extra)
    pre = torch.randn(n, k, generator=gen(seed + 2)).to(DEV)
    c.view.copy_(pre)
    if via_ops:
        assert block_n == min(256, (k + 63) // 64 * 64)
        ops.linear_dense_wgrad(dy, x, n, k, dw=c.view, splits=splits)
    else:
        wgrad_raw(dy, x, [(0, 0, n, k, c.view)], block_n, splits)
    pl = plan()
    verify_wgrad(name, dy, x, [(0, 0, n, k, 0)], [(pre, c.view)], [(c, None, None)], block_n)
    return pl


def test_wgrad_full_rounds_only():
    """splits = 1: one whole tile per CTA pair over the full token range, nothing left over."""
    pl = _wgrad_dense_case("wgrad_full_rounds_only", 4099, 256, 512, 256, splits=1, via_ops=True)
    check_switch(pl)
    expect(pl, ncta=2, full_rounds=1, rem_tiles=0, splits=1, grid=4)


def test_wgrad_full_rounds_and_rem_splits():
    """More tiles than CTAs; the sms // 2 left over are each cut into token ranges (rem_splits > 0)."""
    n = sms()
    tiles = n + n // 2
    s_al = n // (n // 2)
    T = 64 * (8 * s_al) + 1
    pl = _wgrad_dense_case("wgrad_full_rounds_rem_splits", T, 128, 64 * tiles, 64)
    check_switch(pl)
    kb, ncl, fr, rem = wgrad_plan_expected(tiles, T, 1, 0)
    assert fr >= 1 and rem == n // 2
    expect(pl, ncta=1, full_rounds=fr, rem_tiles=rem, rem_splits=s_al, grid=ncl)


def test_wgrad_full_rounds_and_stream_k_line():
    """sms + 1 tiles over a short token range: one full round, then one stream-K line over the last tile."""
    n = sms()
    T = 200
    pl = _wgrad_dense_case("wgrad_full_rounds_stream_k", T, 128, 64 * (n + 1), 64)
    check_switch(pl)
    expect(pl, ncta=1, full_rounds=1, rem_tiles=1, rem_splits=0, grid=n)


def test_wgrad_pure_stream_k_line():
    """One tile over 4099 tokens: no full round; the k-blocks form one stream-K line over a few CTAs."""
    pl = _wgrad_dense_case("wgrad_pure_stream_k", 4099, 128, 64, 64, ld_extra=1)
    check_switch(pl)
    kb, ncl, fr, rem = wgrad_plan_expected(1, 4099, 1, 0)
    expect(pl, ncta=1, full_rounds=0, rem_tiles=1, rem_splits=0, grid=ncl, kb_total=kb)


@pytest.mark.parametrize("splits", [1, 2, 3, 7])
def test_wgrad_explicit_splits(splits):
    """CTA pairs (n_out = 160 > 128, 256-column tile), an explicit token-range split count."""
    pl = _wgrad_dense_case(f"wgrad_splits{splits}", 2000, 160, 256, 256, splits=splits, via_ops=True)
    check_switch(pl)
    kb, ncl, fr, rem = wgrad_plan_expected(1, 2000, 2, splits)
    expect(pl, ncta=2, splits=splits, grid=2 * ncl, full_rounds=fr, rem_tiles=rem, rem_splits=0)


@pytest.mark.parametrize("T", [1, 63, 64, 65, 4099])
def test_core_wgrad_token_counts_scalar_tails(T):
    """Token counts around the 64-token k-block; k_in = 100 and ldw = 101: scalar-atomic tails (no red.v4)."""
    pl = _wgrad_dense_case(f"core_wgrad_T{T}", T, 96, 100, 128, ld_extra=1)
    check_switch(pl)
    expect(pl, ncta=1, block_n=128)


@pytest.mark.parametrize("ci,co,want_ncta", [(128, 160, 2), (24, 16, 1)])
def test_core_linear_d8_wgrad(ci, co, want_ncta):
    """LinearD8 weight gradient: four irrep groups plus the two E-row groups accumulating into one dW_E, into pre-loaded
    targets that sit in one flat buffer with canaries between them."""
    T = 600
    din, dout = 8 * ci, 8 * co
    dy = bf_randn((T, dout), ci + co)
    x = bf_randn((T, din), ci + co + 1)
    shapes = [(co, ci)] * 4 + [(2 * co, 2 * ci)]
    gap = 8
    total = sum(a * b for a, b in shapes) + gap * 6
    flat = Canvas(1, total, torch.float32, top=0, bottom=0, left=0, right=0, ld=total)
    views, pres, spans, off = [], [], [], gap
    for i, (a, b) in enumerate(shapes):
        v = flat.buf[0, off:off + a * b].view(a, b)
        p = torch.randn(a, b, generator=gen(i)).to(DEV)
        v.copy_(p)
        views.append(v)
        pres.append(p)
        spans.append(torch.arange(off, off + a * b, device=DEV))
        off += a * b + gap
    ops.linear_d8_wgrad(dy, x, din, dout, targets=views)
    pl = plan()
    parts = [(g * co, g * ci, co, ci, g) for g in range(4)]
    parts += [(4 * co + r * 2 * co, 4 * ci + r * 2 * ci, 2 * co, 2 * ci, 4) for r in range(2)]
    verify_wgrad(f"core_d8_wgrad_ci{ci}_co{co}", dy, x, parts, list(zip(pres, views)),
                 [(flat, torch.tensor([0], device=DEV), torch.cat(spans))], min(256, (ci + 63) // 64 * 64))
    check_switch(pl)
    expect(pl, ncta=want_ncta, kind=_lib.GEMM_PLAN_WGRAD)


# ------------------------------------------------------------------------------------------------------------------
# switch configurations (fresh process each: the switches are read once per process)
# ------------------------------------------------------------------------------------------------------------------
SWITCHES = [{"OCTIC_GEMM_NCTA": "1"}, {"OCTIC_GEMM_NCTA": "2"}, {"OCTIC_GEMM_WS": "1"}, {"OCTIC_GEMM_PACKED": "0"},
            {"OCTIC_GEMM_DIRECT": "31"}, {"OCTIC_GEMM_STAGES": "2"}, {"OCTIC_GEMM_ROLES_HIGH": "1"},
            {"OCTIC_BLOCK_N": "64"}, {"OCTIC_BLOCK_N": "96"}]


@pytest.mark.skipif(bool(SWITCH), reason="already inside a switch configuration")
@pytest.mark.parametrize("env", SWITCHES, ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()))
def test_switch_configuration(env):
    child_env = {k: v for k, v in os.environ.items() if k not in SWITCH_ENV}
    child_env.update(env)
    r = subprocess.run([sys.executable, "-m", "pytest", __file__, "-q", "-m", "gpu", "-k", "core", "-p", "no:cacheprovider",
                        "-s"], cwd=ROOT, env=child_env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=900)
    tail = "\n".join(r.stdout.splitlines()[-60:])
    print(tail)
    assert r.returncode == 0, f"core cases under {env} failed:\n{tail}"
    assert " passed" in tail and " failed" not in tail
