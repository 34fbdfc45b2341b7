#!/usr/bin/env python
"""bench.py -- headline benchmark of the octic ViT hot path (contract: see the task brief / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference]
                    [--optimizer none|lamb|adamw] [--no-overlap] [--drop-path P] [--no-graph] [--no-cpu-baseline]
                    [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step handed its caller as DIR/<name>.npy (see dump_outputs); the inputs
and the initial weights are seeded, so two builds run with the same arguments can be compared output for output.

Metric (BASELINE.json): hybrid octic ViT-H/14 (DeiT-III: embed 1280, depth 32, heads 16, patch 14, 224 px) images/s,
forward + backward (+ NCCL gradient all-reduce when N > 1), bf16 compute / fp32 residual, synthetic images, random-init
weights.  One process per GPU (torchrun for N > 1); the batch is sharded over ranks (weak scaling: B images per GPU).

The step is the public-API parallel.GraphedTrainStep: bf16 weight re-pack + forward + loss + backward replayed from one
CUDA graph.  `--optimizer` adds the fused parameter update (optim.FusedOptimizer) to every step.  For N > 1 the all-reduce of the
dense half's gradients (88 % of the bytes) runs inside the graph, concurrent with the octic half's backward
(`--no-overlap`: one all-reduce after the replay).

`--impl reference` times the reference on the host CPU cores: the vendored, unmodified reference itself when
baseline/_ref exists (tools/vendor_reference.sh; it travels to the GPU box with the repo snapshot), else the oracle port
of the reference PyTorch path (oracle/octic_oracle.py).  The reference on the SAME B200 (eager and torch.compile) is
measured by tools/bench_reference_gpu.py -> profiles/r02_reference_gpu.json.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

MODEL = dict(name="hybrid_deit_huge_patch14", img=224, patch=14, dim=1280, depth=32, heads=16, classes=1000)


# ----------------------------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md section 8d): FLOP = 2 * MAC, backward = 2 x forward
# ----------------------------------------------------------------------------------------------------------------
def model_flops_per_image(fwd_bwd: bool = True) -> float:
    D, depth, p = MODEL["dim"], MODEL["depth"], MODEL["patch"]
    N = (MODEL["img"] // p) ** 2 + 1
    k = depth // 2
    lin_oct, lin_std, attn = 12 * D * D * 3 / 16, 12 * D * D, 2 * N * D
    mac = k * N * (lin_oct + attn) + (depth - k) * N * (lin_std + attn) + (N - 1) * 3 * p * p * D + D * MODEL["classes"]
    return 2 * mac * (3 if fwd_bwd else 1)


def load_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


# ----------------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference PyTorch path on the host cores
# ----------------------------------------------------------------------------------------------------------------
def vendored_reference_step_fn(batch: int):
    """The UNMODIFIED reference (baseline/_ref, vendored by tools/vendor_reference.sh; git-ignored, travels with gpurun)
    on the host cores: its own OcticVisionTransformer classes through its timm factory, bf16 autocast, fwd + bwd.  Two
    stand-ins are unavoidable on a CPU: tools/timm_shim (timm is not installed) and the reference's own PyTorch GeluD8
    in place of the CUDA-only Triton kernel, mapped exactly as octic_vits/d8_gelu.py:517-541 maps between them.
    Returns None when baseline/_ref is absent."""
    ref = ROOT / "baseline" / "_ref"
    if not (ref / "octic_vits" / "model.py").exists():
        return None
    for q in (str(ROOT / "tools" / "timm_shim"), str(ref)):
        if q not in sys.path:
            sys.path.insert(0, q)
    import octic_vits.deit_models  # noqa: F401  (registers the factories)
    from octic_vits import d8_layers, d8_utils
    from timm.models import create_model as ref_create

    class CpuGeluD8(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.inner = d8_layers.GeluD8()

        def forward(self, xs):
            return d8_utils.convert_8tuple_to_5tuple(self.inner(d8_utils.convert_5tuple_to_8tuple(xs)))

    def swap(mod):
        for name, child in mod.named_children():
            if isinstance(child, d8_layers.TritonGeluD8):
                setattr(mod, name, CpuGeluD8())
            else:
                swap(child)

    torch.manual_seed(0)
    model = ref_create(MODEL["name"], num_classes=MODEL["classes"]).train()
    swap(model)
    img = torch.randn(batch, 3, MODEL["img"], MODEL["img"])
    tgt = torch.randint(0, MODEL["classes"], (batch,))
    params = [q for q in model.parameters() if q.requires_grad]

    def step():
        for q in params:
            q.grad = None
        with torch.autocast("cpu", dtype=torch.bfloat16):
            logits = model(img)
        loss = torch.nn.functional.cross_entropy(logits.float(), tgt)
        loss.backward()
        return loss.item()
    return step


def cpu_reference_step_fn(batch: int):
    from oracle import octic_oracle as O
    from octic_vits_b200.deit_models import create_model
    torch.manual_seed(0)
    model = create_model(MODEL["name"], num_classes=MODEL["classes"])          # parameters only (CPU tensors)
    params = {k: v.detach().clone().requires_grad_(v.is_floating_point() and "cls_token" not in k or k == "cls_token.0")
              for k, v in model.state_dict().items()}
    del model
    img = torch.randn(batch, 3, MODEL["img"], MODEL["img"])
    tgt = torch.randint(0, MODEL["classes"], (batch,))

    def step():
        for p in params.values():
            p.grad = None
        with torch.autocast("cpu", dtype=torch.bfloat16):
            logits = O.octic_vit_forward(img, params, patch=MODEL["patch"], depth=MODEL["depth"], num_heads=MODEL["heads"])
        loss = torch.nn.functional.cross_entropy(logits.float(), tgt)
        loss.backward()
        return loss.item()
    return step


def time_cpu_reference(batch: int, steps: int, warmup: int):
    """(images/s, s/step, threads, kind): kind = "reference" when the vendored reference itself ran, "port" for the
    oracle restatement (baseline/_ref absent)."""
    torch.set_num_threads(os.cpu_count() or 1)
    kind = "reference"
    step = None
    try:
        step = vendored_reference_step_fn(batch)
    except Exception as e:  # noqa: BLE001  (a broken vendored copy must not take the bench line down)
        print(f"bench.py: vendored reference unusable ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
    if step is None:
        kind, step = "port", cpu_reference_step_fn(batch)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return batch / dt, dt, torch.get_num_threads(), kind


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = 4
    steps, warmup = max(1, min(args.steps, 3)), max(1, min(args.warmup, 1))
    ips, dt, cores, kind = time_cpu_reference(batch, steps, warmup)
    what = ("the unmodified reference (baseline/_ref: its own OcticVisionTransformer via its timm factory; PyTorch GeluD8 "
            "for the CUDA-only Triton kernel)" if kind == "reference" else "CPU oracle port of the reference PyTorch path")
    line = {
        "impl": "reference", "metric": "hybrid octic ViT-H/14 images/s fwd+bwd", "value": ips, "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"hybrid_deit_huge_patch14 fwd+bwd, 224px, {what}, bf16 autocast on the host cores, "
                               "bounded sample", "batch": batch},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": f"batch {batch}, {warmup} warm-up + {steps} timed fwd+bwd steps"},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# outputs of the timed step, for comparing two builds
# ----------------------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 22          # positions drawn per sample: at most 16 MB per array in fp32, ~33 MB in all
DUMP_SEED = 0


def dump_outputs(out_dir: str, loss: torch.Tensor, fg, updated_params: bool) -> None:
    """Writes the step's results as float32 / float64 .npy files:
        loss.npy          the loss, float32 [1]
        grad_norm.npy     L2 norm of every trainable parameter's gradient, float64, in model.parameters() order
        grad_sample.npy   the gradient at fixed positions over all trainable elements, float32, in position order:
                          DUMP_SAMPLE draws with seed DUMP_SEED, repeats removed (4,169,746 distinct positions for the
                          headline model)
    and, when the step also ran the optimizer, param_norm.npy / param_sample.npy: the updated parameters, same layout.
    The full gradient (1.4 GB for the headline model) is too large to keep; the per-parameter norms catch an error in
    any one tensor, the sample compares element by element.  The weight-gradient kernels reduce with atomic adds, so
    two runs of the same build differ in the last bits; profiles/r03_bench_dump_spread.txt records how much."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    params = fg.params
    numels = torch.tensor([p.numel() for p in params])
    ends = numels.cumsum(0)
    pick = torch.randint(int(ends[-1]), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(DUMP_SEED)).unique()
    owner = torch.searchsorted(ends, pick, right=True)
    local = pick - (ends - numels)[owner]
    bounds = torch.searchsorted(owner, torch.arange(len(params) + 1)).tolist()

    def sample_and_norms(tensors):
        vals = [t.detach().reshape(-1)[local[bounds[i]:bounds[i + 1]].to(t.device)] for i, t in enumerate(tensors)]
        norms = [torch.linalg.vector_norm(t.detach(), dtype=torch.float64) for t in tensors]
        return torch.cat(vals).float().cpu().numpy(), torch.stack(norms).cpu().numpy()

    arrays = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
    arrays["grad_sample"], arrays["grad_norm"] = sample_and_norms([p.grad for p in params])
    if updated_params:
        arrays["param_sample"], arrays["param_norm"] = sample_and_norms(params)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from octic_vits_b200 import _lib, functional as OF, ops
    from octic_vits_b200.deit_models import create_model

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if not _lib.load().octic_device_ok():
        raise SystemExit("bench.py: no sm_100 device -- the CUDA path is the only path")

    torch.manual_seed(1234 + rank)
    B = args.batch
    model = create_model(MODEL["name"], num_classes=MODEL["classes"], drop_path_rate=args.drop_path).to(dev).train()
    # one flat fp32 gradient buffer: .grad tensors are views, the all-reduce is a single NCCL call over NVLink
    from octic_vits_b200.parallel import FlatGrads, GraphedTrainStep
    fg = FlatGrads(model.parameters())
    flat = fg.flat
    opt = None
    if args.optimizer != "none":
        # fused parameter update (optim.FusedOptimizer: LAMB = the DeiT-III recipe, experiments/train_deit.py:42)
        from octic_vits_b200.optim import FusedOptimizer
        opt = FusedOptimizer(model, fg, kind=args.optimizer, lr=1e-3, weight_decay=0.05)

    img_dev = torch.randn(B, 3, MODEL["img"], MODEL["img"], device=dev)
    tgt_dev = torch.randint(0, MODEL["classes"], (B,), device=dev)
    img_host = torch.randn(B, 3, MODEL["img"], MODEL["img"]).pin_memory()
    tgt_host = torch.randint(0, MODEL["classes"], (B,)).pin_memory()

    def eager_step(img, tgt):
        ops.begin_step()
        flat.zero_()
        logits = model(img)
        loss = torch.nn.functional.cross_entropy(logits, tgt)
        loss.backward()
        fg.all_reduce()
        if opt is not None:
            opt.step()
        return loss

    # public-API step: fwd + loss + bwd captured in a CUDA graph (parallel.GraphedTrainStep), all-reduce after the replay
    overlap = False
    if world > 1 and not args.no_overlap:
        # the dense half's gradients (88 % of the bytes) are all-reduced from an autograd hook at the bridge, on a side
        # stream inside the captured graph, while the octic half is still in backward
        from octic_vits_b200.parallel import install_early_allreduce
        overlap = install_early_allreduce(model, fg)
    gstep = GraphedTrainStep(model, fg, img_dev.shape, warmup=args.warmup, use_graph=not args.no_graph, optimizer=opt)
    overlap = overlap and model._bridge_grad_hook is not None
    step = gstep if gstep.graphed else eager_step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps

    for _ in range(args.warmup):
        step(img_dev, tgt_dev)
    barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = {}

    def timed_step():
        last["loss"] = step(img_dev, tgt_dev)
    ms_dev = timed(timed_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before the untimed eager steps below overwrite the gradients (and, with an optimizer, the parameters)
        dump_outputs(args.dump_outputs, last["loss"], fg, updated_params=opt is not None)
    # launches of our kernels inside the timed region: counted on one eager step (a graph replay launches the same nodes)
    from octic_vits_b200 import functional as OF
    if gstep.graphed:
        OF.bump_param_epoch()         # the graphed step re-packs the bf16 weights every replay: count those launches too
    _lib.STATS.reset()
    eager_step(img_dev, tgt_dev)
    torch.cuda.synchronize()
    launches = _lib.STATS.kernel_launches * args.steps

    # Roofline evidence, measured live on this binary: every launch of the two kernel families that dominate the step is
    # timed with CUDA events on the launching stream during one extra eager step (untimed for the headline, so the headline
    # number carries no event overhead).
    #   dense family  (tensor bound): gemm_tn_kernel with one group + gemm_wgrad_kernel = every nn.Linear of the 16 dense
    #                 blocks, forward, dgrad and wgrad (82 % of the model FLOPs)
    #   octic family  (HBM bound, SURVEY.md section 8d): the four LinearD8 forward GEMMs of the 16 octic blocks
    _lib.STATS.reset()
    _lib.STATS.profile_prefixes = ("octic_gemm_bf16", "octic_gemm_wgrad_bf16", "octic_linear_d8_fwd", "octic_linear_d8_dgrad",
                                   "octic_linear_d8_wgrad", "octic_attention_fwd", "octic_attention_bwd")
    eager_step(img_dev, tgt_dev)
    torch.cuda.synchronize()
    fam = _lib.STATS.collect_by_name()
    _lib.STATS.profile_prefixes = ()
    z = (0.0, 0.0, 0)
    gemm_ms = fam.get("octic_gemm_bf16", z)[0] + fam.get("octic_gemm_wgrad_bf16", z)[0]
    gemm_flops = fam.get("octic_gemm_bf16", z)[1] + fam.get("octic_gemm_wgrad_bf16", z)[1]
    gemm_calls = fam.get("octic_gemm_bf16", z)[2] + fam.get("octic_gemm_wgrad_bf16", z)[2]
    oct_ms, oct_flops, oct_calls = fam.get("octic_linear_d8_fwd", z)
    # algorithmic bytes of the octic forward linears per token and block (fp32 residual, bf16 activations; weights are
    # L2 resident and excluded): qkv 2D+6D, proj+residual 2D+4D+4D, fc1 2D+8D, fc2+residual 8D+4D+4D = 44 D
    T_tokens = B * ((MODEL["img"] // MODEL["patch"]) ** 2 + 1)
    oct_bytes = 44.0 * MODEL["dim"] * T_tokens * (MODEL["depth"] // 2)

    if gstep.graphed:
        gstep.stage(img_host, tgt_host)

    def e2e_step():
        if gstep.graphed:
            # public-API input pipeline: the step consumes the staged batch, the H2D copy of the NEXT batch (every step
            # copies its own inputs from pinned host memory) runs on the copy stream meanwhile, then the loss is read back
            loss = gstep.run()
            gstep.stage(img_host, tgt_host)
            return loss.item()
        img = img_host.to(dev, non_blocking=True)
        tgt = tgt_host.to(dev, non_blocking=True)
        return eager_step(img, tgt).item()
    e2e_step()
    ms_e2e = timed(e2e_step, max(2, args.steps // 2))

    if rank == 0:
        peaks = load_peaks()
        ips = world * B / (ms_dev * 1e-3)
        flops_img = model_flops_per_image(True)
        achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
        cpu_ips, cpu_dt, cores, cpu_kind = (None, None, None, "port")
        if world == 1 and not args.no_cpu_baseline:
            cpu_ips, cpu_dt, cores, cpu_kind = time_cpu_reference(2, 2, 1)
        line = {
            "metric": "hybrid octic ViT-H/14 images/s fwd+bwd", "value": ips, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "hybrid_deit_huge_patch14 (embed 1280, depth 32: 16 octic + 16 dense, heads 16, patch 14) "
                                   "DeiT-III training step: fwd + bwd" + (" + NCCL grad all-reduce" if world > 1 else ""),
                       "img": MODEL["img"], "batch_per_gpu": B, "global_batch": world * B, "tokens_per_image": 257,
                       "batch_policy": "BASELINE configs[3] / SURVEY 8d: 64-256 images per GPU; default 192 (round 1 ran 128; "
                                       "same-box sweep in profiles/r02_bench_batch_sweep.txt)",
                       "drop_path": args.drop_path, "parallelism": f"dp{world}",
                       "optimizer_step": False if opt is None else f"fused {args.optimizer} (3 launches/step, weight "
                                                                    "re-pack inside the graph)",
                       "cuda_graph": bool(gstep.graphed), "allreduce_overlap": bool(overlap),
                       "weight_repack_in_step": True,   # fp32 -> bf16 weight packs run every step (as autocast re-casts)
                       "l2": "activations per step (>50 GB) exceed the 126 MB L2; no explicit flush"},
            "model_tflops": ips * flops_img / 1e12,
            "tc_util_vs_sustained_peak": ips * flops_img / 1e12 / (world * peaks["tf_sustained"]),
            "roofline": {"kernel": "gemm_tn_kernel<groups=1> + gemm_wgrad_kernel (tcgen05 bf16 GEMM, CTA pairs): every nn.Linear "
                                   "of the 16 dense blocks, forward + dgrad + wgrad",
                         "bound": "tensor", "achieved": achieved_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": (achieved_tf / peaks["tf_sustained"]) if achieved_tf else None,
                         # DRAM bytes per launch come from ncu --set full captures of single shapes, not from this run
                         "traffic": None, "traffic_source": "profiles/r02_ncu_*.md (per-shape dram__bytes vs algorithmic bytes)",
                         "peak_source": f"{peaks['src']} (bf16 sustained)", "launches_timed": gemm_calls,
                         "share_of_step": gemm_ms / ms_dev},
            "roofline_octic": {"kernel": "gemm_tn_kernel<groups=6> (LinearD8 forward: qkv, proj+residual, fc1, fc2+residual of "
                                         "the 16 octic blocks)",
                               "bound": "hbm", "achieved": (oct_bytes / (oct_ms * 1e-3) / 1e9) if oct_ms > 0 else None,
                               "peak": peaks["hbm"], "unit": "GB/s",
                               "frac": (oct_bytes / (oct_ms * 1e-3) / 1e9 / peaks["hbm"]) if oct_ms > 0 else None,
                               "traffic": None, "algorithmic_bytes_per_token_per_block": 44 * MODEL["dim"],
                               "peak_source": f"{peaks['src']} (copy bandwidth)", "launches_timed": oct_calls,
                               "share_of_step": oct_ms / ms_dev,
                               "tflops": (oct_flops / (oct_ms * 1e-3) / 1e12) if oct_ms > 0 else None},
            "step_breakdown_ms": {k: round(v[0], 3) for k, v in sorted(fam.items())},
            "cpu_baseline": {"value": cpu_ips, "unit": "images/s", "cores": cores, "kind": cpu_kind,
                             "sample": "batch 2, 1 warm-up + 2 timed fwd+bwd steps of the same model on the host cores, bf16 autocast ("
                                       + ("the vendored reference itself" if cpu_kind == "reference" else "oracle port") + ")"},
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "images/s",
                    "h2d_bytes_per_step": img_host.numel() * 4 + tgt_host.numel() * 8, "d2h_bytes_per_step": 4},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # A CUDA graph that captured NCCL kernels keeps the communicator alive: release it before tearing NCCL down (the
        # process otherwise hangs in destroy_process_group, observed at 2 GPUs in round 1).  The result line is already
        # printed; a watchdog ends the process if the teardown still does not return.
        sys.stdout.flush()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        gstep.close()
        del gstep
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=192,
                    help="images per GPU (SURVEY.md section 8d / BASELINE.json configs[3]: 64-256 per GPU; 192 measured "
                         "+3 %% images/s over 128 on the same box, profiles/r02_bench_batch_sweep.txt)")
    ap.add_argument("--drop-path", type=float, default=0.0)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run the eager step instead of the captured CUDA graph")
    ap.add_argument("--overlap", action="store_true", help="(default since round 2; kept for old command lines)")
    ap.add_argument("--no-overlap", action="store_true",
                    help="N > 1: one all-reduce after the graph replay instead of all-reducing the dense half's gradients "
                         "from inside the captured graph while the octic half is still in backward (DESIGN.md section 5)")
    ap.add_argument("--optimizer", default="none", choices=["none", "lamb", "adamw"],
                    help="also run the fused parameter update every step (the headline metric is fwd+bwd)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and the (sampled) gradients of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
