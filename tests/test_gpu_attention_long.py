"""Streamed tcgen05 attention (attention_tc.cu, attn_stream_tc_kernel): head-major sequences too long for the resident
tcgen05 kernels and for the mma.sync backward.

Kernel results are compared with an fp32 attention (and its autograd) on the same bf16 inputs, with the bounds of
test_gpu_kernels.py::test_attention; each case also shows that the bound rejects the result of a reference that
dropped one 64-key chunk.  Outputs are written into NaN-filled buffers through the C ABI, and nothing outside the
launch's own rows may change.
"""
import ctypes as C

import pytest
import torch

from octic_vits_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda"
ATTN_DENSE, ATTN_OCTIC_PACKED, ATTN_OCTIC_HEADMAJOR = 0, 1, 2     # include/octic_b200.h OCTIC_ATTN_*
PAD = 7                                                           # NaN guard rows around every output

# last N the mma.sync backward of the dense layout fits (2 Npad (hd + 8) 2 + 8 Npad + 6 hd <= 227 KiB)
LEGACY_BWD_LAST = {64: 784, 80: 640}
# last N octic_attention_headmajor_supported(N, hd, backward) returned 1 for before the streamed kernels existed
# (the resident envelope): {hd: (forward, backward)}
RESIDENT_LAST = {32: (512, 512), 64: (512, 352), 80: (512, 272), 96: (512, 208), 128: (368, 144)}


def setup_module(module):
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


def _lib_():
    return _lib.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _supported(N, hd, backward):
    return bool(_lib_().octic_attention_headmajor_supported(int(N), int(hd), int(backward)))


# ---------------------------------------------------------------------------------------------------------------------
# layouts: the kernels read head-major q, k, v, dO; OCTIC_HEADMAJOR writes o and dqkv as packed octic rows
# ---------------------------------------------------------------------------------------------------------------------
def _octic_perms(H, hd):
    """(o_perm, qkv_perm): packed column c of an o row / qkv row holds head-major column perm[c]."""
    from oracle import octic_oracle as O
    idx = torch.arange(H * hd, dtype=torch.float32).reshape(1, H, 1, hd)
    o_perm = O.pack_rows(O.attention_unpack_d8(idx)).reshape(-1).long()
    D = H * hd
    rows = torch.arange(3 * D, dtype=torch.float32).reshape(1, 1, 3 * D)
    q, k, v = O.attention_heads_d8(O.unpack_rows(rows), H)
    hm_of = torch.stack((q, k, v), 0).permute(1, 3, 0, 2, 4).reshape(3 * D).long()   # head-major j <- packed hm_of[j]
    qkv_perm = torch.empty_like(hm_of)
    qkv_perm[hm_of] = torch.arange(3 * D)
    return o_perm, qkv_perm


def _reference(qkv_hm, d_o_hm, B, N, H, hd, drop_chunk=None):
    """fp32 attention on head-major bf16 rows: (o_hm [B*N, D], lse [B, H, N], dqkv_hm [B*N, 3D]).
    drop_chunk: key chunk index whose 64 keys are left out (the error the bounds must detect)."""
    D = H * hd
    x = qkv_hm.float().clone().requires_grad_(True)
    t = x.reshape(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    q, k, v = t[0], t[1], t[2]
    s = q @ k.transpose(-1, -2) / hd ** 0.5
    if drop_chunk is not None:
        s = s.clone()
        s[..., drop_chunk * 64:(drop_chunk + 1) * 64] = float("-inf")
    lse = torch.logsumexp(s, dim=-1)
    o = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B * N, D)
    (o * d_o_hm.float()).sum().backward()
    return o.detach(), lse.detach(), x.grad


def _to_layout(o_hm, dqkv_hm, layout, H, hd):
    if layout == ATTN_DENSE:
        return o_hm, dqkv_hm
    o_perm, qkv_perm = _octic_perms(H, hd)
    return o_hm[:, o_perm.to(o_hm.device)], dqkv_hm[:, qkv_perm.to(dqkv_hm.device)]


def _nan_buffer(rows, cols, dtype):
    return torch.full((rows + 2 * PAD, cols), float("nan"), dtype=dtype, device=DEV)


def _guards_intact(buf):
    return bool(torch.isnan(buf[:PAD].float()).all()) and bool(torch.isnan(buf[-PAD:].float()).all())


def _run(qkv_hm, d_o_hm, B, N, H, hd, layout):
    """forward + backward through the C ABI, every output inside a NaN-filled buffer"""
    D = H * hd
    L = _lib_()
    o_buf = _nan_buffer(B * N, D, torch.bfloat16)
    lse_buf = _nan_buffer(B * H, N, torch.float32)
    o, lse = o_buf[PAD:PAD + B * N], lse_buf[PAD:PAD + B * H]
    rc = L.octic_attention_fwd(qkv_hm.data_ptr(), o.data_ptr(), lse.data_ptr(), B, N, H, hd, layout, _stream())
    assert rc == 0, _lib.OcticError(rc)
    assert L.octic_attention_bwd_workspace_bytes(N, hd) == 0
    dq_buf = _nan_buffer(B * N, 3 * D, torch.bfloat16)
    dqkv = dq_buf[PAD:PAD + B * N]
    delta = torch.full((B, H, N), float("nan"), dtype=torch.float32, device=DEV)
    rc = L.octic_attention_bwd_ws(qkv_hm.data_ptr(), o.data_ptr(), d_o_hm.data_ptr(), lse.data_ptr(), delta.data_ptr(),
                                  dqkv.data_ptr(), B, N, H, hd, layout, None, 0, _stream())
    assert rc == 0, rc
    torch.cuda.synchronize()
    for buf, core in ((o_buf, o), (lse_buf, lse), (dq_buf, dqkv)):
        assert _guards_intact(buf), "a launch wrote outside its rows"
        assert torch.isfinite(core.float()).all(), "an output row was not written (or is not finite)"
    return o, lse.reshape(B, H, N), dqkv


def _inputs(B, N, H, hd, seed, scale=1.5):
    g = torch.Generator().manual_seed(seed)
    D = H * hd
    qkv = (torch.randn(B * N, 3 * D, generator=g) * scale).to(torch.bfloat16).to(DEV)
    d_o = torch.randn(B * N, D, generator=g).to(torch.bfloat16).to(DEV)
    return qkv, d_o


def _close(got, want, rtol, atol):
    return bool(torch.isclose(got.float(), want.float(), rtol=rtol, atol=atol).all())


# ---------------------------------------------------------------------------------------------------------------------
# 1. kernels against the fp32 reference
# ---------------------------------------------------------------------------------------------------------------------
LONG_SHAPES = [
    (1, 785, 2, 64),     # first streamed N for hd 64
    (1, 641, 2, 80),     # first streamed N for hd 80
    (2, 1025, 2, 80),
    (1, 1370, 3, 64),
    (1, 1370, 2, 80),
    (1, 2049, 2, 64),
    (1, 4096, 1, 80),
    (1, 1001, 2, 80),    # neither a multiple of 16 nor of 128
    (1, 1500, 2, 32),
    (1, 1111, 2, 96),
    (1, 900, 2, 128),
]


@pytest.mark.parametrize("layout", [ATTN_DENSE, ATTN_OCTIC_HEADMAJOR])
@pytest.mark.parametrize("B,N,H,hd", LONG_SHAPES)
def test_streamed_attention_matches_fp32(B, N, H, hd, layout):
    assert _supported(N, hd, True) and _supported(N, hd, False)
    qkv, d_o = _inputs(B, N, H, hd, seed=N * 3 + hd + layout)
    # the kernels read dO head-major; the reference's o / dO live in the same head-major space
    o, lse, dqkv = _run(qkv, d_o, B, N, H, hd, layout)
    want_o, want_lse, want_dqkv = _reference(qkv, d_o, B, N, H, hd)
    want_o, want_dqkv = _to_layout(want_o, want_dqkv, layout, H, hd)
    assert _close(o, want_o, 2e-2, 2e-2), float((o.float() - want_o).abs().max())
    assert _close(lse, want_lse, 1e-3, 1e-3), float((lse - want_lse).abs().max())
    assert _close(dqkv, want_dqkv, 3e-2, 3e-2), float((dqkv.float() - want_dqkv).abs().max())
    # the bounds see one dropped key chunk (in the forward output and in the gradients)
    bad_o, _, bad_dqkv = _reference(qkv, d_o, B, N, H, hd, drop_chunk=N // 128)
    bad_o, bad_dqkv = _to_layout(bad_o, bad_dqkv, layout, H, hd)
    assert not _close(o, bad_o, 2e-2, 2e-2)
    assert not _close(dqkv, bad_dqkv, 3e-2, 3e-2)


def test_streamed_backward_is_deterministic():
    """dQ is recomputed per query tile, not reduced with atomics: two launches give the same bits"""
    B, N, H, hd = 1, 1025, 4, 80
    qkv, d_o = _inputs(B, N, H, hd, seed=11)
    a = _run(qkv, d_o, B, N, H, hd, ATTN_DENSE)
    b = _run(qkv, d_o, B, N, H, hd, ATTN_DENSE)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------------------------
# 2. extreme score ranges (test_gpu_kernels.py::test_attention_extreme_score_ranges at long N)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("growth", [6.0, -6.0])
@pytest.mark.parametrize("B,N,H,hd", [(1, 1370, 2, 80), (1, 2049, 2, 64)])
def test_streamed_attention_extreme_score_ranges(B, N, H, hd, growth):
    """keys whose scale grows (growth > 0: the row maximum first appears in the last key chunks, so the forward's lazy
    rescale runs again and again) or shrinks with the token index; o, lse and the gradients stay finite and right"""
    D = H * hd
    g = torch.Generator().manual_seed(N * 7 + hd)
    x = torch.randn(B, N, 3, H, hd, generator=g) * 1.5
    ramp = torch.linspace(0.0, 1.0, N).view(1, N, 1, 1)
    x[:, :, 1] *= torch.exp2(ramp * growth) if growth > 0 else torch.exp2((1.0 - ramp) * -growth)
    qkv = x.reshape(B * N, 3 * D).to(torch.bfloat16).to(DEV)
    d_o = torch.randn(B * N, D, generator=g).to(torch.bfloat16).to(DEV)
    o, lse, dqkv = _run(qkv, d_o, B, N, H, hd, ATTN_DENSE)
    want_o, want_lse, want_dqkv = _reference(qkv, d_o, B, N, H, hd)
    if growth > 0:
        s = (qkv.float().reshape(B, N, 3, H, hd)[:, :, 0].transpose(1, 2)
             @ qkv.float().reshape(B, N, 3, H, hd)[:, :, 1].permute(0, 2, 3, 1))
        assert float((s.argmax(-1) >= N - 128).float().mean()) > 0.5     # row maxima in the last two key chunks
    assert _close(o, want_o, 2e-2, 2e-2)
    assert _close(lse, want_lse, 1e-3, 2e-3)
    got, ref = dqkv.float(), want_dqkv
    assert float((got - ref).norm() / ref.norm()) < 3e-2
    assert float((got - ref).abs().max() / ref.abs().max()) < 3e-2


# ---------------------------------------------------------------------------------------------------------------------
# 3. boundary: which shapes the streamed kernels take
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hd", [64, 80])
def test_streamed_admission_boundary(hd):
    last = LEGACY_BWD_LAST[hd]
    for bw in (0, 1):
        assert not _supported(last, hd, bw)
        assert _supported(last + 1, hd, bw)
        assert _supported(4096, hd, bw)


@pytest.mark.parametrize("hd", [32, 64, 80, 96, 128])
def test_shapes_that_run_today_keep_their_kernel(hd):
    """up to the mma.sync backward limit, octic_attention_headmajor_supported answers as before the streamed kernels"""
    Npad_max = (227 * 1024 - 6 * hd) // (2 * (hd + 8) * 2 + 8)
    legacy_last = Npad_max // 16 * 16
    if hd in LEGACY_BWD_LAST:
        assert legacy_last == LEGACY_BWD_LAST[hd]
    fwd_last, bwd_last = RESIDENT_LAST[hd]
    for N in range(1, legacy_last + 1):
        assert _supported(N, hd, 0) == (N <= fwd_last), (N, hd)
        assert _supported(N, hd, 1) == (N <= bwd_last), (N, hd)
    assert _supported(legacy_last + 1, hd, 1)


@pytest.mark.parametrize("N,hd", [(641, 80), (656, 80), (785, 64), (800, 64)])
def test_band_forward_agrees_with_mma_sync_forward(N, hd):
    """forward-only calls where only the mma.sync backward fails moved to the streamed kernel: it agrees with the
    mma.sync forward of the packed layout on the same q, k, v"""
    B, H = 2, 2
    D = H * hd
    qkv_hm, _ = _inputs(B, N, H, hd, seed=N + hd)
    o_perm, qkv_perm = _octic_perms(H, hd)
    qkv_packed = qkv_hm[:, qkv_perm.to(DEV)].contiguous()
    L = _lib_()
    o1 = torch.empty(B * N, D, dtype=torch.bfloat16, device=DEV)
    o2 = torch.empty_like(o1)
    l1 = torch.empty(B, H, N, dtype=torch.float32, device=DEV)
    l2 = torch.empty_like(l1)
    assert L.octic_attention_fwd(qkv_hm.data_ptr(), o1.data_ptr(), l1.data_ptr(), B, N, H, hd, ATTN_OCTIC_HEADMAJOR,
                                 _stream()) == 0
    assert L.octic_attention_fwd(qkv_packed.data_ptr(), o2.data_ptr(), l2.data_ptr(), B, N, H, hd, ATTN_OCTIC_PACKED,
                                 _stream()) == 0
    torch.cuda.synchronize()
    assert _close(o1, o2, 1e-2, 1e-2)
    assert _close(l1, l2, 1e-4, 1e-4)
    want_o, _, _ = _reference(qkv_hm, torch.zeros(B * N, D, device=DEV), B, N, H, hd)
    assert _close(o1, want_o[:, o_perm.to(DEV)], 2e-2, 2e-2)


def test_packed_layout_keeps_refusing_long_sequences():
    B, N, H, hd = 1, 1025, 2, 80
    qkv = torch.zeros(B * N, 3 * H * hd, dtype=torch.bfloat16, device=DEV)
    o = torch.empty(B * N, H * hd, dtype=torch.bfloat16, device=DEV)
    assert _lib_().octic_attention_fwd(qkv.data_ptr(), o.data_ptr(), None, B, N, H, hd, ATTN_OCTIC_PACKED,
                                       _stream()) != 0


# ---------------------------------------------------------------------------------------------------------------------
# 4. models above the old limit: nothing in layers.py / model.py / dinov2_models.py branches on it
# ---------------------------------------------------------------------------------------------------------------------
def _rel(got, want):
    got, want = got.float().cpu(), want.float().cpu()
    return float((got - want).norm() / want.norm().clamp_min(1e-12))


def _check(got, want, rel, mx, what):
    got, want = got.float().cpu(), want.float().cpu()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    r = _rel(got, want)
    m = float((got - want).abs().max() / want.abs().max().clamp_min(1e-12))
    assert r < rel and m < mx, f"{what}: rel L2 {r:.3e} (< {rel}), max-abs/max {m:.3e} (< {mx})"


def _hybrid_364(depth=2):
    """hybrid octic ViT, head dim 80 (embed 640, 8 heads), patch 14 at 364 px: N = 26^2 + 1 = 677 tokens (the
    symmetric pos-embed is a quarter table unfolded by reflection, so the patch grid must be even)"""
    from octic_vits_b200.model import OcticVisionTransformer
    from tests.test_gpu_model import _randomize
    torch.manual_seed(0)
    model = OcticVisionTransformer(img_size=364, patch_size=14, embed_dim=640, depth=depth, num_heads=8, num_classes=10,
                                   qkv_bias=True).to(DEV)
    _randomize(model, seed=1)
    return model


HYBRID_364_KEYS = ["patch_embed.lift8.conv_A1.weight", "pos_embed.0", "cls_token.0", "blocks.0.norm1.scaling.alpha_E",
                   "blocks.0.attn.qkv.lin_A1.weight", "blocks.0.attn.qkv.lin_E.weight", "blocks.0.attn.qkv.lin_A1.bias",
                   "blocks.0.attn.proj.lin_E.weight", "blocks.0.ls1.alpha_A2", "blocks.0.mlp.fc1.lin_E.weight",
                   "blocks.0.mlp.fc2.lin_A1.weight", "blocks.1.attn.qkv.weight", "blocks.1.attn.qkv.bias",
                   "blocks.1.attn.proj.weight", "blocks.1.ls1.gamma", "blocks.1.mlp.fc1.weight", "blocks.1.mlp.fc2.weight",
                   "norm.weight", "head.weight", "head.bias"]


def test_hybrid_vit_hd80_364px_within_reference_bf16_budget():
    """logits and a spread of parameter gradients through both blocks (streamed attention forward and backward in the
    octic head-major and the dense layout) against the fp32 CPU oracle (BlockD8: layer scale ls1 / ls2, the oracle's
    'dinov2' block style), held to the bound of test_gpu_parity_budget.py:
    err(ours vs fp32) <= 1.25 x err(oracle under bf16 autocast vs fp32) + 2e-3, and the logits also to the flat
    5e-2 relative L2 of test_gpu_model.py::test_config1_vit_s16_against_oracle."""
    from oracle import octic_oracle as O
    budget, floor = 1.25, 2e-3
    assert _supported(677, 80, True) and _supported(677, 80, False)
    model = _hybrid_364().train()
    gen = torch.Generator().manual_seed(2)
    img = torch.randn(2, 3, 364, 364, generator=gen)
    gout = torch.randn(2, 10, generator=gen)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    keys = [k for k in HYBRID_364_KEYS if k in sd]
    assert len(keys) == len(HYBRID_364_KEYS), sorted(set(HYBRID_364_KEYS) - set(sd))

    def oracle(bf16):
        params = {k: v.clone().requires_grad_(k in keys) for k, v in sd.items()}
        with torch.autocast("cpu", dtype=torch.bfloat16, enabled=bf16):
            out = O.octic_vit_forward(img, params, patch=14, depth=2, num_heads=8, style="dinov2")
        (out.float() * gout).sum().backward()
        return out.detach().float(), {k: params[k].grad.float() for k in keys}

    want, gwant = oracle(False)
    ref16, gref16 = oracle(True)
    logits = model(img.to(DEV))
    (logits.float() * gout.to(DEV)).sum().backward()
    params = dict(model.named_parameters())
    _check(logits.detach(), want, 5e-2, 1.5e-1, "logits at N = 677")
    rows = {"logits": (_rel(logits.detach(), want), _rel(ref16, want))}
    for k in keys:
        assert params[k].grad is not None, k
        rows[k] = (_rel(params[k].grad, gwant[k]), _rel(gref16[k], gwant[k]))
    for k, (ours, ref) in rows.items():
        print(f"  {k:42s} ours {ours:.3e} | reference bf16 {ref:.3e} | ratio {ours / max(ref, 1e-12):.2f}")
    bad = {k: v for k, v in rows.items() if not v[0] <= budget * v[1] + floor}
    assert not bad, f"error above {budget} x the reference's own bf16 error at N = 677: {bad}"


def test_graphed_train_step_at_streamed_size():
    """parallel.GraphedTrainStep at N = 677 (streamed attention forward and backward inside the graph): replay equals
    the eager step"""
    from octic_vits_b200.parallel import FlatGrads, GraphedTrainStep
    model = _hybrid_364().train()
    fg = FlatGrads(model.parameters())
    img = torch.randn(2, 3, 364, 364, device=DEV)
    tgt = torch.randint(0, 10, (2,), device=DEV)
    step = GraphedTrainStep(model, fg, img.shape, warmup=2)
    assert step.graphed, getattr(step, "capture_error", "")
    loss_g = float(step(img, tgt))
    grads_g = fg.flat.clone()
    eager = GraphedTrainStep(model, fg, img.shape, use_graph=False)
    loss_e = float(eager(img, tgt))
    assert abs(loss_g - loss_e) <= 1e-5 * max(1.0, abs(loss_e))
    assert _rel(grads_g, fg.flat) < 1e-4
    assert float(grads_g.abs().max()) > 0


def test_hybrid_trunk_equivariance_at_364px():
    """D8 equivariance of the octic trunk at N = 677, held to the bound test_headline_model_equivariance_report uses
    at 224 px (2e-2 relative L2)"""
    from octic_vits_b200 import layers as L
    from oracle import octic_oracle as O
    model = _hybrid_364(depth=4).eval()
    img = torch.randn(2, 3, 364, 364, device=DEV)
    worst = 0.0
    with torch.no_grad():
        base = tuple(t.float() for t in L.OF.unpack_five(model.forward_trunk_packed(img)))
        assert base[0].shape[1] == 677
        for g in O.GROUP:
            moved = L.OF.unpack_five(model.forward_trunk_packed(O.image_action(g, img).contiguous()))
            want = O.token_action(g, base, has_cls=True)
            worst = max([worst] + [_rel(a, b) for a, b in zip(moved, want)])
    print(f"trunk equivariance at 364 px (N = 677): worst relative L2 over D8 = {worst:.3e}")
    assert worst < 2e-2


def test_dinov2_hd64_448px_dynamic_img_size_crop_list():
    """DINOv2 octic backbone, head dim 64, dynamic_img_size=True: 448 px global crops (N = 28^2 + 1 + 2 registers =
    787, pos-embed unfolded from the 14 x 14 table) and 96 px local crops in one list through the concatenated-segment
    path.  Outputs against the oracle crop by crop; gradients of the segment path against the crop-by-crop path."""
    from octic_vits_b200 import dinov2_models as DM
    from oracle import octic_oracle as O
    torch.manual_seed(3)
    model = DM.OcticDinoVisionTransformer(img_size=224, patch_size=16, embed_dim=256, depth=2, num_heads=4,
                                          num_register_tokens=2, init_values=0.5, dynamic_img_size=True).to(DEV).train()
    with torch.no_grad():
        for p in model.parameters():
            if p.requires_grad and p.dim() >= 2:
                p.mul_(3.0)
    big, small = torch.randn(2, 3, 448, 448), torch.randn(3, 3, 96, 96)
    assert _supported(787, 64, True) and _supported(39, 64, True)
    segs = ((2, 787), (3, 39))
    assert all(b.supports_segments(segs) for b in model.blocks[:model.octic_equi_break_layer])
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    keys = ("x_norm_clstoken", "x_norm_regtokens", "x_norm_patchtokens", "x_prenorm")

    def run(concat):
        model.concat_crops = concat
        for p in model.parameters():
            p.grad = None
        outs = model([big.to(DEV), small.to(DEV)], is_training=True)
        loss = sum((o["x_norm_clstoken"].float() ** 2).mean() + (o["x_norm_patchtokens"].float() ** 2).mean()
                   for o in outs)
        loss.backward()
        return outs, {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}

    outs, grads = run(True)
    for o, im in zip(outs, (big, small)):
        with torch.no_grad():
            want = O.octic_dino_forward_features(im, sd, patch=16, depth=2, num_heads=4)
        assert o["x_norm_patchtokens"].shape[1] == (im.shape[-1] // 16) ** 2
        for k in keys:
            _check(o[k].detach(), want[k], 3e-2, 8e-2, f"{im.shape[-1]} px {k}")
    outs_b, grads_b = run(False)
    for oa, ob in zip(outs, outs_b):
        for k in keys:
            _check(oa[k].detach(), ob[k].detach(), 1e-6, 1e-5, f"concat vs crop-by-crop {k}")
    assert set(grads) == set(grads_b) and len(grads) > 0
    for n in grads:
        assert torch.isfinite(grads[n]).all()
        _check(grads[n], grads_b[n], 2e-3, 2e-2, f"grad {n}")
