"""CPU-only tests: the C-ABI library loads and exports every prototype of include/octic_b200.h, the host-side mirror
keeps the reference's constructor / state-dict / error contract, the product path refuses to run without a GPU, and
the batch-shard + flat-gradient all-reduce logic works at world_size 2 (gloo)."""
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def lib():
    from octic_vits_b200 import _lib
    if not _lib.LIB_PATH.exists():
        subprocess.run(["bash", str(ROOT / "build.sh")], check=True, cwd=ROOT)
    return _lib.load()


def header_prototypes():
    hdr = (ROOT / "include" / "octic_b200.h").read_text()
    return re.findall(r"^(?:int|size_t|const char\*)\s+(octic_\w+)\s*\(", hdr, flags=re.M)


def test_library_exports_every_header_symbol(lib):
    from octic_vits_b200 import _lib
    names = header_prototypes()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/octic_b200.h but not exported"
    bound = set(_lib.SIGNATURES) | {"octic_strerror", "octic_version", "octic_device_ok",
                                      "octic_attention_headmajor_supported", "octic_attention_bwd_workspace_bytes"}
    assert set(names) == bound, set(names) ^ bound
    assert lib.octic_version() >= 201
    if not torch.cuda.is_available():
        # size query of the staged-dQ scratch: no device -> "the staged path does not apply" (0), never a crash
        assert lib.octic_attention_bwd_workspace_bytes(257, 80) == 0
        # no GEMM launched on this thread yet: no launch plan to report
        import ctypes as C
        assert lib.octic_gemm_last_plan(C.byref(_lib.GemmPlan())) == -1
    assert lib.octic_strerror(-2).decode().startswith("pointer or leading dimension")


def test_no_cpu_fallback(lib):
    from octic_vits_b200 import layers as L
    from octic_vits_b200._lib import OcticError
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert lib.octic_device_ok() == 0
    xs = tuple(torch.randn(1, 3, 8) for _ in range(4)) + (torch.randn(1, 3, 2, 16),)
    for mod in (L.LinearD8(64, 64), L.LayerNormD8(64), L.TritonGeluD8(), L.AttentionD8(64, 2), L.MlpD8(64),
                L.Layer_scale_init_BlockD8(64, 2), L.BlockD8(64, 2), L.PowerSpectrumInvariant(64),
                L.IsotypicToPatchD8(64, 4, out_channels=4)):
        with pytest.raises(OcticError):
            mod(xs)


def test_constructor_contract_matches_reference():
    from octic_vits_b200 import layers as L
    for bad in (lambda: L.LinearD8(60, 64), lambda: L.LinearD8(64, 60), lambda: L.AffineD8(12),
                lambda: L.LayerScaleD8(12), lambda: L.LiftD8(3, 60, 8, 8, True), lambda: L.PatchEmbedD8(embed_dim=60)):
        with pytest.raises(ValueError):
            bad()
    with pytest.raises(NotImplementedError):
        L.AttentionD8(64, 2, rope=object())
    with pytest.raises(AssertionError):
        L.AttentionD8(60, 7)
    with pytest.raises(ValueError):
        L.LiftIrrepD8Conv2d(3, 8, 8, 8, bias=True, irrep="A2")
    with pytest.raises(ValueError):
        L.LiftIrrepD8Conv2d(3, 8, 2, 2, bias=False, irrep="B1")
    with pytest.raises(NotImplementedError):
        L.LiftIrrepD8Conv2d(3, 8, 7, 7, bias=False)
    blk = L.Layer_scale_init_BlockD8(64, 2, init_values=0.25)
    assert float(blk.gamma_1.alpha_E[0]) == 0.25 and blk.gamma_1.beta is None
    assert isinstance(L.BlockD8(64, 2).ls1, torch.nn.Identity)
    assert isinstance(L.BlockD8(64, 2, init_values=1e-5).ls1, L.LayerScaleD8)


@pytest.mark.parametrize("name", ["model_hybrid", "model_invariant", "model_timm_default"])
def test_reference_state_dict_loads_key_for_key(golden, name):
    from octic_vits_b200 import layers as L
    from octic_vits_b200.model import OcticVisionTransformer
    fx = golden(name)
    cfg = fx["cfg"]
    kw = dict(img_size=cfg["img_size"], patch_size=cfg["patch"], embed_dim=cfg["embed_dim"], depth=cfg["depth"],
              num_heads=cfg["num_heads"], num_classes=cfg["num_classes"])
    if name == "model_timm_default":
        model = OcticVisionTransformer(init_scale=0.7, **kw)
    else:
        model = OcticVisionTransformer(qkv_bias=True, invariant=cfg["invariant"],
                                       standard_block_layers=L.Layer_scale_init_Block,
                                       octic_block_layers=L.Layer_scale_init_BlockD8, **kw)
    assert list(model.state_dict().keys()) == list(fx["sd"].keys())
    for k, v in model.state_dict().items():
        assert v.shape == fx["sd"][k].shape, k
    model.load_state_dict(fx["sd"], strict=True)
    frozen = [n for n, p in model.named_parameters() if not p.requires_grad]
    assert frozen == [f"cls_token.{i}" for i in range(1, 5)]
    assert "cls_token.0" in model.no_weight_decay() and "pos_embed.5" in model.no_weight_decay()


def test_factories_and_param_counts():
    from octic_vits_b200.deit_models import create_model, list_models
    assert {"hybrid_deit_large_patch16", "hybrid_deit_huge_patch14", "d8_inv_early_deit_huge_patch14",
            "d8_inv_early_deit_large_patch16"} <= set(list_models())
    with pytest.raises(RuntimeError):
        create_model("no_such_model")
    m = create_model("hybrid_deit_small_patch16", num_classes=1000, drop_rate=0.0, drop_path_rate=0.1, drop_block_rate=None)
    assert sum(p.numel() for p in m.parameters()) == 12_439_432 or abs(sum(p.numel() for p in m.parameters()) / 1e6 - 12.44) < 0.01


@pytest.mark.parametrize("name", ["model_dinov2", "model_dinov2_inv"])
def test_dinov2_reference_state_dict_loads_key_for_key(golden, name):
    """OcticDinoVisionTransformer (reference dinov2_models.py:40-111): same keys, in the same order, same shapes."""
    from octic_vits_b200.dinov2_models import OcticDinoVisionTransformer
    fx = golden(name)
    model = OcticDinoVisionTransformer(**fx["cfg"])
    # the base class passes init_values=init_scale (1e-4) to every block, overriding a partial's 1e-5 (model.py:116-137)
    assert float(model.blocks[0].ls1.alpha_A1[0].detach()) == pytest.approx(1e-4)
    assert float(model.blocks[-1].ls1.gamma[0].detach()) == pytest.approx(1e-4)
    assert list(model.state_dict().keys()) == list(fx["sd"].keys())
    for k, v in model.state_dict().items():
        assert v.shape == fx["sd"][k].shape, k
    model.load_state_dict(fx["sd"], strict=True)
    frozen = sorted(n for n, p in model.named_parameters() if not p.requires_grad)
    want = [f"{g}.{i}" for g in ("cls_token", "mask_token") for i in range(1, 8)]
    if fx["cfg"]["num_register_tokens"]:
        want += [f"register_tokens.{i}" for i in range(1, 8)]
    assert frozen == sorted(want)
    assert isinstance(model.head, torch.nn.Identity)
    assert model.no_weight_decay() >= {"pos_embed.0", "cls_token.0", "_orig_mod.pos_embed.5"}


def test_dinov2_factories_and_contract():
    from octic_vits_b200 import dinov2_models as DM
    from octic_vits_b200.deit_models import create_model, list_models
    assert {"hybrid_dinov2_vit_large_patch16", "hybrid_dinov2_vit_huge_patch16", "d8_inv_early_dinov2_vit_large_patch16",
            "d8_inv_early_dinov2_vit_huge_patch16"} <= set(list_models())
    m = create_model("hybrid_dinov2_vit_large_patch16", num_register_tokens=4, drop_path_rate=0.3)
    assert m.depth == 24 and m.embed_dim == 1024 and m.register_tokens[0].shape == (1, 4, 128)
    assert isinstance(m.blocks[0], DM.NestedTensorBlockD8) and isinstance(m.blocks[12], DM.NestedTensorBlock)
    assert m.blocks[12].sample_drop_ratio == 0.3 and m.blocks[0].sample_drop_ratio == 0.3
    with pytest.raises(AssertionError):
        DM.OcticDinoVisionTransformer(img_size=32, patch_size=8, embed_dim=64, depth=3, num_heads=2)
    with pytest.raises(AssertionError):
        m.blocks[12]("not a tensor")
    with pytest.raises(AssertionError):
        m.blocks[0]("not a tuple")
    with pytest.raises(AssertionError):
        DM.MemEffAttention(64, 2)(torch.zeros(1, 4, 64), attn_bias=object())
    k3 = DM.OcticDinoVisionTransformer(img_size=32, patch_size=8, embed_dim=64, depth=4, num_heads=2, octic_equi_break_layer=3)
    assert [isinstance(b, DM.NestedTensorBlockD8) for b in k3.blocks] == [True, True, True, False]
    with pytest.raises(AssertionError):          # only dense-half blocks can be taken (reference :206)
        m.get_intermediate_layers(torch.zeros(1, 3, 224, 224), n=[3])
    if not torch.cuda.is_available():
        from octic_vits_b200._lib import OcticError
        with pytest.raises(OcticError):
            m(torch.zeros(1, 3, 224, 224))


def test_dinov2_subset_stochastic_depth_factor():
    """drop_add_residual_stochastic_depth (dinov2/layers/block.py:117-140) as a per-sample factor"""
    from octic_vits_b200.dinov2_models import Block, subset_drop_scale
    torch.manual_seed(0)
    s = subset_drop_scale(10, 0.35, "cpu")
    assert int((s > 0).sum()) == 6 and torch.allclose(s[s > 0], torch.tensor(10 / 6))
    assert float(s.sum()) == pytest.approx(10.0)
    assert int((subset_drop_scale(3, 0.99, "cpu") > 0).sum()) == 1
    blk = Block(64, 2, init_values=1e-5, drop_path=0.05).train()
    s1, s2 = blk._drop_scales(8, "cpu")                      # <= 0.1: Bernoulli mask / keep
    assert all(v == 0.0 or v == pytest.approx(1 / 0.95) for v in s1.tolist())
    s1, _ = blk._drop_scales(8, "cpu", nested=True)          # list input: always the subset rule
    assert int((s1 > 0).sum()) == 7
    assert blk.eval()._drop_scales(8, "cpu") == (None, None)


def test_pos_embed_unfold_matches_oracle(golden):
    from octic_vits_b200.model import unfold_pos_embed_packed
    from oracle import octic_oracle as O
    fx = golden("model_hybrid")
    ps = [fx["sd"][f"pos_embed.{i}"] for i in range(6)]
    want = O.pack_rows(tuple(t.flatten(0, 1) for t in O.unfold_pos_embed(ps)))
    assert torch.equal(unfold_pos_embed_packed(ps), want)


def test_lift_weight_expansion_matches_oracle(golden):
    from octic_vits_b200 import layers as L
    from oracle import octic_oracle as O
    fx = golden("model_hybrid")
    lift = L.LiftD8(3, 64, 16, 16, True)
    lift.load_state_dict({k[len("patch_embed.lift8."):]: v for k, v in fx["sd"].items() if k.startswith("patch_embed.lift8.")})
    for name in ("A1", "A2", "B1", "B2"):
        got = getattr(lift, f"conv_{name}").expand_weight()
        assert torch.allclose(got, O.expand_lift_weight(fx["sd"][f"patch_embed.lift8.conv_{name}.weight"], name), atol=1e-7)
    assert torch.allclose(lift.conv_E_left.expand_weight(),
                          O.expand_lift_weight(fx["sd"]["patch_embed.lift8.conv_E_left.weight"], "E"), atol=1e-7)
    w, b = lift.packed_weight_and_bias()
    assert w.shape == (64, 3 * 16 * 16) and b.shape == (64,) and torch.count_nonzero(b[8:]) == 0


def test_pack_unpack_views_are_zero_copy():
    from octic_vits_b200 import functional as OF
    x = torch.randn(2, 5, 64)
    xs = OF.unpack_five(x)
    assert [tuple(t.shape) for t in xs] == [(2, 5, 8)] * 4 + [(2, 5, 2, 16)]
    assert OF.pack_five(xs) is x                       # views of one packed tensor: no copy
    ys = tuple(t.clone() for t in xs)
    assert torch.equal(OF.pack_five(ys), x)            # foreign tensors: packed by concatenation
    with pytest.raises(AssertionError):
        OF.pack_five(xs[:4])


def test_shard_batch_covers_everything():
    from octic_vits_b200.parallel import shard_batch
    for gb, world in [(256, 8), (10, 4), (7, 8), (2048, 2)]:
        spans = [shard_batch(gb, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == gb
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from octic_vits_b200.parallel import FlatGrads, shard_batch
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
torch.manual_seed(0)                                   # same replica on both ranks
model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.GELU(), torch.nn.Linear(5, 3))
model[0].bias.requires_grad_(False)                    # a frozen parameter, like cls_token.1-4
fg = FlatGrads(model.parameters())
data = torch.randn(8, 6, generator=torch.Generator().manual_seed(1))
a, b = shard_batch(8, rank, 2)
fg.zero()
model(data[a:b]).square().sum().backward()
fg.all_reduce()
# reference: the whole batch on one replica; mean over ranks of per-shard sums = full sum / 2
ref = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.GELU(), torch.nn.Linear(5, 3))
ref.load_state_dict(model.state_dict())
ref(data).square().sum().backward()
for (n, p), q in zip(model.named_parameters(), ref.parameters()):
    if p.requires_grad:
        assert torch.allclose(p.grad, q.grad / 2, atol=1e-5), n
    else:
        assert p.grad is None
assert model[0].weight.grad.data_ptr() == fg.flat.data_ptr()
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
"""


def test_flat_grad_allreduce_world2_gloo(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    procs = [subprocess.Popen([sys.executable, str(script), str(ROOT), str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


_GLOO_EARLY_WORKER = r"""
import sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from octic_vits_b200.parallel import FlatGrads, install_early_allreduce, shard_batch
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()


class Toy(torch.nn.Module):
    # the hook point and parameter order of OcticVisionTransformer: front end | blocks[:k] | blocks[k:] | norm | head
    def __init__(self, late_param_last=False):
        super().__init__()
        self.embed = torch.nn.Linear(6, 8)
        self.blocks = torch.nn.ModuleList([torch.nn.Linear(8, 8) for _ in range(4)])
        self.norm = torch.nn.LayerNorm(8)
        self.head = torch.nn.Linear(8, 3)
        if late_param_last:
            self.mask_token = torch.nn.ParameterList([torch.nn.Parameter(torch.zeros(8))])   # registered last, used first (DINOv2)
        self.octic_equi_break_layer = 2
        self._bridge_grad_hook = None
        self.fired = 0

    def forward(self, x):
        t = self.embed(x) + (self.mask_token[0] if hasattr(self, "mask_token") else 0)
        for b in self.blocks[:2]:
            t = torch.tanh(b(t))
        if self._bridge_grad_hook is not None and t.requires_grad:
            t.register_hook(self._bridge_grad_hook)
        for b in self.blocks[2:]:
            t = torch.tanh(b(t))
        return self.head(self.norm(t))


torch.manual_seed(0)
model, ref = Toy(), Toy()
ref.load_state_dict(model.state_dict())
fg = FlatGrads(model.parameters(), fuse_accumulation=False)
assert install_early_allreduce(model, fg)
names = [n for n, _ in model.named_parameters()]
assert fg.split == fg.offsets[names.index("blocks.2.weight")] and 0 < fg.split < fg.flat.numel()
calls = []
orig = fg.all_reduce_early
fg.all_reduce_early = lambda *a, **k: (calls.append(fg._early_done), orig(*a, **k))
data = torch.randn(8, 6, generator=torch.Generator().manual_seed(1))
a, b = shard_batch(8, rank, 2)
for step in range(2):                                   # two steps: the per-step flag must reset
    fg.begin_step()
    model(data[a:b]).square().sum().backward()
    assert fg._early_done                               # the hook fired during backward and reduced flat[split:]
    fg.all_reduce()                                     # ... so this reduces only flat[:split]
    assert not fg._early_done
    ref.zero_grad()
    ref(data).square().sum().backward()
    for (n, p), q in zip(model.named_parameters(), ref.parameters()):
        assert torch.allclose(p.grad, q.grad / 2, atol=1e-5), (step, n)
assert calls == [False, False]
# a parameter of the octic side registered after the head: the overlap must refuse
m2 = Toy(late_param_last=True)
fg2 = FlatGrads(m2.parameters(), fuse_accumulation=False)
assert not install_early_allreduce(m2, fg2) and fg2.split == fg2.flat.numel() and m2._bridge_grad_hook is None
fg2.begin_step()
m2(data[a:b]).square().sum().backward()
fg2.all_reduce()
ref2 = Toy(late_param_last=True); ref2.load_state_dict(m2.state_dict())
ref2(data).square().sum().backward()
for (n, p), q in zip(m2.named_parameters(), ref2.parameters()):
    assert torch.allclose(p.grad, q.grad / 2, atol=1e-5), n


class ToyMulti(Toy):
    # OcticVisionTransformer also calls per-block hooks: several exchange buckets, issued back to front during backward
    def __init__(self):
        super().__init__()
        self._block_grad_hooks = {}

    def forward(self, x):
        t = self.embed(x)
        for i, b in enumerate(self.blocks):
            if i == 2 and self._bridge_grad_hook is not None and t.requires_grad:
                t.register_hook(self._bridge_grad_hook)
            elif i in self._block_grad_hooks and t.requires_grad:
                t.register_hook(self._block_grad_hooks[i])
            t = torch.tanh(b(t))
        return self.head(self.norm(t))


m3, ref3 = ToyMulti(), ToyMulti()
ref3.load_state_dict(m3.state_dict())
fg3 = FlatGrads(m3.parameters(), fuse_accumulation=False)
assert install_early_allreduce(m3, fg3, boundaries=[3, 2, 1])
n3 = [n for n, _ in m3.named_parameters()]
assert fg3.bounds == [fg3.offsets[n3.index(f"blocks.{i}.weight")] for i in (3, 2, 1)] and fg3.split == fg3.bounds[-1]
assert sorted(m3._block_grad_hooks) == [1, 3] and m3._bridge_grad_hook is not None
spans = []
orig3 = fg3._reduce
fg3._reduce = lambda t, avg: (spans.append((t.storage_offset(), t.numel())), orig3(t, avg))
for step in range(2):
    fg3.begin_step()
    m3(data[a:b]).square().sum().backward()
    assert fg3._early_n == 3
    fg3.all_reduce()
    assert fg3._early_n == 0
    ref3.zero_grad()
    ref3(data).square().sum().backward()
    for (n, p), q in zip(m3.named_parameters(), ref3.parameters()):
        assert torch.allclose(p.grad, q.grad / 2, atol=1e-5), (step, n)
# four disjoint spans per step that tile the buffer back to front: [b3, end), [b2, b3), [b1, b2), [0, b1)
b3, b2, b1 = fg3.bounds
want = [(b3, fg3.flat.numel() - b3), (b2, b3 - b2), (b1, b2 - b1), (0, b1)]
assert spans == want + want, spans
# a step in which backward stops early (only some hooks fire) still reduces every element exactly once
fg3.begin_step(); spans.clear()
fg3._early_n = 0
fg3.all_reduce_early()                  # bucket 0 only
fg3.all_reduce()
assert spans == [(b3, fg3.flat.numel() - b3), (0, b3)], spans
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
"""


def test_early_allreduce_overlap_world2_gloo(tmp_path):
    """parallel.install_early_allreduce: the dense half's gradients are exchanged from an autograd hook at the bridge,
    the rest after backward; the result equals the single all-reduce."""
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "worker_early.py"
    script.write_text(_GLOO_EARLY_WORKER)
    procs = [subprocess.Popen([sys.executable, str(script), str(ROOT), str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors in _lib.py have the size and the field offsets the C compiler gives the structs of
    include/octic_b200.h (a drift would corrupt every descriptor passed through the C ABI)."""
    import ctypes as C
    from octic_vits_b200 import _lib
    pairs = {"octic_gemm_group": _lib.GemmGroup, "octic_gemm_desc": _lib.GemmDesc, "octic_wgrad_group": _lib.WgradGroup,
             "octic_wgrad_desc": _lib.WgradDesc, "octic_lsfin_seg": _lib.LsFinSeg, "octic_optim_chunk": _lib.OptimChunk,
             "octic_optim_seg": _lib.OptimSeg, "octic_gemm_plan": _lib.GemmPlan}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{ROOT / "include" / "octic_b200.h"}"', 'int main(void) {']
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = {}
    for line in subprocess.run([str(exe)], check=True, stdout=subprocess.PIPE, text=True).stdout.splitlines():
        cname, field, val = line.split()
        got[(cname, field)] = int(val)
    for cname, cls in pairs.items():
        assert got[(cname, "size")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)


def test_optimizer_chunk_table_covers_every_parameter_once():
    from octic_vits_b200.optim import CHUNK, build_chunk_table, timm_no_decay
    from octic_vits_b200.deit_models import create_model
    from octic_vits_b200.parallel import FlatGrads
    model = create_model("hybrid_deit_small_patch16", num_classes=10)
    fg = FlatGrads(model.parameters(), fuse_accumulation=False)
    assert all(o % 4 == 0 for o in fg.offsets) and fg.flat.numel() >= sum(p.numel() for p in fg.params)
    numels = [p.numel() for p in fg.params]
    ptrs = [p.data_ptr() for p in fg.params]
    chunks, segs = build_chunk_table(numels, fg.offsets, ptrs, [0] * len(ptrs), [(0.05, 1.0)] * len(ptrs))
    assert len(segs) == len(fg.params)
    covered = torch.zeros(fg.flat.numel(), dtype=torch.int32)
    for i, (p, e, off, n, seg) in enumerate(chunks):
        assert 0 < n <= CHUNK and e == 0
        first, count = segs[seg][2], segs[seg][3]
        assert first <= i < first + count
        assert p == ptrs[seg] + 4 * (off - fg.offsets[seg])           # same element in the parameter and the flat buffer
        covered[off:off + n] += 1
    for o, n in zip(fg.offsets, numels):
        assert bool((covered[o:o + n] == 1).all())
    assert int(covered.sum()) == sum(numels)                           # padding elements are never touched
    assert sum(s[3] for s in segs) == len(chunks)
    from octic_vits_b200._lib import OptimChunk, OptimSeg
    ch = (OptimChunk * len(chunks))(*[OptimChunk(*c) for c in chunks])
    sg = (OptimSeg * len(segs))(*[OptimSeg(*t) for t in segs])
    last = chunks[-1]
    assert (ch[len(chunks) - 1].p, ch[len(chunks) - 1].off, ch[len(chunks) - 1].len, ch[len(chunks) - 1].seg) == (last[0], last[2], last[3], last[4])
    assert ch[0].ema is None and sg[3].first_chunk == segs[3][2] and sg[3].num_chunks == segs[3][3]
    assert abs(sg[0].weight_decay - 0.05) < 1e-7 and sg[0].lr_scale == 1.0
    nd = timm_no_decay(model)
    assert "cls_token.0" in nd and "pos_embed.3" in nd and "blocks.0.norm1.scaling.alpha_E" in nd
    assert "blocks.0.attn.qkv.lin_A1.bias" in nd and "blocks.0.attn.qkv.lin_E.weight" not in nd
    assert "blocks.7.gamma_1" in nd and "head.weight" not in nd and "cls_token.1" not in nd   # frozen: not a candidate
    # the product class refuses CPU parameters (after validating them and building the tables): no CPU path
    from octic_vits_b200.optim import FusedOptimizer
    from octic_vits_b200._lib import OcticError
    ema = create_model("hybrid_deit_small_patch16", num_classes=10)
    for kind in ("lamb", "adamw"):
        with pytest.raises(OcticError, match="no CPU path"):
            FusedOptimizer(model, fg, kind=kind, lr=1e-3, weight_decay=0.05, ema=(ema, 0.99), lr_scales={"head.weight": 0.5})
    with pytest.raises(ValueError):
        FusedOptimizer(model, fg, kind="sgd")
    with pytest.raises(ValueError):
        FusedOptimizer(ema, fg)                                        # fg's parameters are not this model's


def test_dinov2_subset_draw_is_uniform_and_segment_row_scales():
    """The graph-safe subset draw (rank of iid uniforms, no randperm / sort) selects every sample with probability
    keep / b; per-segment per-sample factors of a concatenated crop list expand to one factor per token ROW."""
    from octic_vits_b200.dinov2_models import subset_drop_scale
    from octic_vits_b200.layers import _seg_row_scale, _seg_rows
    torch.manual_seed(1)
    b, ratio, trials = 8, 0.5, 4000
    hits = torch.zeros(b)
    for _ in range(trials):
        s = subset_drop_scale(b, ratio, "cpu")
        assert int((s > 0).sum()) == 4 and float(s.max()) == pytest.approx(2.0)
        hits += (s > 0).float()
    assert torch.all((hits / trials - 0.5).abs() < 0.04), hits / trials
    segs = ((2, 3), (3, 2))
    assert _seg_rows(segs) == 12
    assert _seg_row_scale([None, None], segs, "cpu") is None
    rs = _seg_row_scale([torch.tensor([2.0, 0.0]), None], segs, "cpu")
    assert rs.tolist() == [2.0] * 3 + [0.0] * 3 + [1.0] * 6
    rs = _seg_row_scale([torch.tensor([2.0, 0.0]), torch.tensor([0.0, 3.0, 1.5])], segs, "cpu")
    assert rs.tolist() == [2.0] * 3 + [0.0] * 3 + [0.0] * 2 + [3.0] * 2 + [1.5] * 2
