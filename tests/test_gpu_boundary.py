"""Boundary contract on the GPU (SURVEY.md section 8b): torch.compile around the modules, the autocast policy, and the
INTEGRATION.md recipe that keeps the REFERENCE's OcticVisionTransformer class and swaps only the blocks."""
import pytest
import torch

from oracle import octic_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from octic_vits_b200 import functional as OF, layers as L
    from octic_vits_b200._lib import OcticError
    from octic_vits_b200.model import OcticVisionTransformer

DEV = "cuda"


def rel(a, b):
    a, b = a.detach().float(), b.detach().float()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def small_model(seed=0):
    torch.manual_seed(seed)
    m = OcticVisionTransformer(img_size=64, patch_size=8, embed_dim=128, depth=4, num_heads=2, num_classes=10, qkv_bias=True,
                               init_scale=0.5, standard_block_layers=L.Layer_scale_init_Block,
                               octic_block_layers=L.Layer_scale_init_BlockD8).to(DEV).train()
    return m


def test_torch_compile_wraps_the_model_and_its_blocks():
    """deit/main.py:341-342 wraps the whole model in torch.compile.  The kernels sit behind a C ABI that Dynamo cannot
    trace; the module forwards are marked torch.compiler.disable, so compile() is a supported call: same logits, same
    gradients, no exception from inside ctypes.  backend='eager' keeps Inductor code generation out of the test."""
    model = small_model()
    img = torch.randn(3, 3, 64, 64, device=DEV)
    w = torch.randn(3, 10, device=DEV)
    want = model(img)
    (want * w).sum().backward()
    g_want = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    for p in model.parameters():
        p.grad = None
    compiled = torch.compile(model, backend="eager")
    got = compiled(img)
    (got * w).sum().backward()
    assert torch.equal(got, want)
    for k, p in model.named_parameters():
        if k in g_want:
            assert rel(p.grad, g_want[k]) < 1e-4, k          # wgrad red.add order differs run to run

    # a user module that loops over OUR blocks the way the reference model does (5-tuples between blocks)
    class Trunk(torch.nn.Module):
        def __init__(self, blocks):
            super().__init__()
            self.blocks = blocks

        def forward(self, xs):
            for blk in self.blocks:
                xs = blk(xs)
            return tuple(2.0 * t for t in xs)

    trunk = Trunk(model.blocks[:2])
    t0 = torch.randn(2, 65, 128, device=DEV)
    xs = OF.unpack_five(t0)
    want5 = trunk(xs)
    got5 = torch.compile(trunk, backend="eager")(xs)
    for a, b in zip(got5, want5):
        assert torch.equal(a, b)


def test_strict_autocast_switch():
    """The arithmetic is always the reference's bf16-autocast arithmetic; strict mode turns a call outside such a
    context into an error instead of a silent precision change."""
    model = small_model(1).eval()
    img = torch.randn(2, 3, 64, 64, device=DEV)
    with torch.no_grad():
        base = model(img)
        OF.set_strict_autocast(True)
        try:
            with pytest.raises(OcticError, match="autocast"):
                model(img)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                inside = model(img)
            with torch.autocast("cuda", dtype=torch.float16), pytest.raises(OcticError, match="autocast"):
                model(img)
        finally:
            OF.set_strict_autocast(False)
    assert torch.equal(inside.float(), base.float())


def reference_class_forward(model, img):
    """The reference's OcticVisionTransformer.forward (octic_vits/model.py:170-227, global_pool=False, hybrid) as the
    oracle restates it -- pinned to the reference's own outputs by tests/test_oracle_golden.py::test_whole_model --
    with the submodules that its injection points octic_block_layers / standard_block_layers / Patch_layer
    (model.py:62-64) would hold called through the reference's interfaces: Patch_layer(img) -> 5-tuple, octic blocks
    on 5-tuples, dense blocks on [B, N, D].  Positional embedding, cls token, bridge, norm and head are the reference's
    fp32 torch ops, not this package's fused paths."""
    xs = model.patch_embed(img)
    pos = O.unfold_pos_embed(list(model.pos_embed))
    xs = tuple(x + p.flatten(0, 1) for x, p in zip(xs, pos))
    B = img.shape[0]
    xs = tuple(torch.cat((c.expand(B, *c.shape[1:]), x), dim=1) for c, x in zip(model.cls_token, xs))
    k = model.octic_equi_break_layer
    for blk in model.blocks[:k]:
        xs = blk(xs)
    x = O.hybrid_bridge(xs)
    for blk in model.blocks[k:]:
        x = blk(x)
    return model.head(model.norm(x)[:, 0])


def test_reference_model_class_with_our_blocks():
    """INTEGRATION.md section 1, second recipe: the reference's model-level code with this package's blocks plugged in
    through its injection points must give what our model class gives with the same parameters.  (The state-dict
    layout of the reference class is checked by test_cpu_host.py::test_reference_state_dict_loads_key_for_key.)"""
    torch.manual_seed(3)
    kw = dict(img_size=64, patch_size=8, embed_dim=128, depth=4, num_heads=2, num_classes=10, qkv_bias=True, init_scale=0.5)
    ours = OcticVisionTransformer(standard_block_layers=L.Layer_scale_init_Block,
                                  octic_block_layers=L.Layer_scale_init_BlockD8, **kw).to(DEV).eval()
    img = torch.randn(3, 3, 64, 64, device=DEV)
    with torch.no_grad():
        a, b = reference_class_forward(ours, img), ours(img)
    assert a.shape == b.shape
    # same kernels underneath; the reference class adds the positional embedding / concatenates in fp32 torch ops
    assert rel(a, b) < 5e-3, rel(a, b)
    # and it trains: gradients reach the octic parameters through the reference's tuple plumbing
    ours.train()
    reference_class_forward(ours, img).square().sum().backward()
    g = ours.blocks[0].attn.qkv.lin_E.weight.grad
    assert g is not None and float(g.abs().sum()) > 0
