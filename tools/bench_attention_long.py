"""Long-sequence attention on the streamed tcgen05 kernels (attention_tc.cu, attn_stream_tc_kernel).

Reports, in one run on one GPU:
  * per-launch forward and backward time (CUDA events over many launches) at ViT-H/14 shapes (hd 80, 16 heads,
    N = 730 / 1025 / 1370) and ViT-L/16 shapes (hd 64, 16 heads, N = 785 / 1025), head-major octic layout, with TFLOP/s
    against the algorithmic FLOPs (forward 4 N^2 hd, backward 10 N^2 hd per (image, head));
  * images/s of a hybrid octic ViT-H/14 GraphedTrainStep at 448 px (N = 1025);
  * per-kernel counts of UTCHMMA / LDTM / UTMALDG / HMMA in the SASS of the streamed kernels (cuobjdump -sass);
  * the card's name and power limit, read in the same run.

    python tools/bench_attention_long.py [--out profiles/r04_attention_long.txt] [--iters 50] [--e2e-batch 16]
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

SHAPES = [("ViT-H/14", 16, 730, 80), ("ViT-H/14 448px", 16, 1025, 80), ("ViT-H/14", 16, 1370, 80),
          ("ViT-L/16 448px", 16, 785, 64), ("ViT-L/16 512px", 16, 1025, 64)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def time_ms(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def kernel_times(batch, iters):
    from octic_vits_b200 import ops
    rows = []
    for name, H, N, hd in SHAPES:
        assert ops.attention_headmajor_ok(N, hd, True), (N, hd)
        B = batch
        D = H * hd
        g = torch.Generator(device="cuda").manual_seed(N)
        qkv = torch.randn(B * N, 3 * D, device="cuda", generator=g).to(torch.bfloat16)
        d_o = torch.randn(B * N, D, device="cuda", generator=g).to(torch.bfloat16)
        o, lse = ops.attention_fwd(qkv, B, N, H, hd, ops.ATTN_OCTIC_HEADMAJOR)
        dqkv = torch.empty_like(qkv)
        t_f = time_ms(lambda: ops.attention_fwd(qkv, B, N, H, hd, ops.ATTN_OCTIC_HEADMAJOR, out=o), iters)
        t_b = time_ms(lambda: ops.attention_bwd(qkv, o, d_o, lse, B, N, H, hd, ops.ATTN_OCTIC_HEADMAJOR, out=dqkv), iters)
        f_fwd, f_bwd = 4.0 * B * H * N * N * hd, 10.0 * B * H * N * N * hd
        rows.append({"shape": name, "B": B, "H": H, "N": N, "hd": hd, "fwd_ms": t_f, "bwd_ms": t_b,
                     "fwd_tflops": f_fwd / t_f / 1e9, "bwd_tflops": f_bwd / t_b / 1e9})
    return rows


def e2e(batch, steps):
    from octic_vits_b200.deit_models import create_model
    from octic_vits_b200.parallel import FlatGrads, GraphedTrainStep
    torch.manual_seed(0)
    model = create_model("hybrid_deit_huge_patch14", img_size=448, num_classes=1000).cuda().train()
    fg = FlatGrads(model.parameters())
    img = torch.randn(batch, 3, 448, 448, device="cuda")
    tgt = torch.randint(0, 1000, (batch,), device="cuda")
    step = GraphedTrainStep(model, fg, img.shape, warmup=2)
    for _ in range(2):
        float(step(img, tgt))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step(img, tgt)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    return {"model": "hybrid_deit_huge_patch14", "img": 448, "N": 1025, "batch": batch, "graphed": bool(step.graphed),
            "step_ms": dt * 1e3, "images_per_s": batch / dt, "loss": float(loss),
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}


def sass_counts():
    from octic_vits_b200._lib import LIB_PATH
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([exe, "-sass", os.fspath(LIB_PATH)], capture_output=True, text=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if "attn_stream_tc_kernel" in m.group(1) else None
            if cur:
                counts[cur] = {k: 0 for k in ("UTCHMMA", "LDTM", "STTM", "UTMALDG", "HMMA")}
            continue
        if cur:
            for k in counts[cur]:
                if re.search(r"\b" + k + r"\b", line):
                    counts[cur][k] += 1
    return counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_attention_long.txt")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--batch", type=int, default=8, help="images per attention launch")
    ap.add_argument("--e2e-batch", type=int, default=16)
    ap.add_argument("--e2e-steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no CPU mode")
    res = {"card": card(), "kernels": kernel_times(args.batch, args.iters), "e2e": e2e(args.e2e_batch, args.e2e_steps),
           "sass": sass_counts()}
    lines = [f"# streamed tcgen05 attention -- {res['card']} (name, power limit, max SM clock)",
             f"# per-launch CUDA-event means over {args.iters} launches; head-major octic layout; TFLOP/s against "
             "4 N^2 hd (fwd) / 10 N^2 hd (bwd, incl. delta) per (image, head)",
             f"{'shape':<16} {'B':>3} {'H':>3} {'N':>5} {'hd':>3} {'fwd ms':>8} {'fwd TF/s':>9} {'bwd ms':>8} {'bwd TF/s':>9}"]
    for r in res["kernels"]:
        lines.append(f"{r['shape']:<16} {r['B']:>3} {r['H']:>3} {r['N']:>5} {r['hd']:>3} {r['fwd_ms']:>8.3f} "
                     f"{r['fwd_tflops']:>9.1f} {r['bwd_ms']:>8.3f} {r['bwd_tflops']:>9.1f}")
    e = res["e2e"]
    lines.append(f"# end to end: {e['model']} GraphedTrainStep at {e['img']} px (N = {e['N']}), batch {e['batch']}, "
                 f"graphed={e['graphed']}: {e['step_ms']:.1f} ms/step = {e['images_per_s']:.1f} images/s, "
                 f"peak memory {e['peak_mem_gb']:.1f} GiB")
    lines.append("# SASS of the streamed kernels (instruction counts per kernel):")
    for k, v in sorted(res["sass"].items()):
        lines.append(f"{k}: " + " ".join(f"{n}={c}" for n, c in v.items()))
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)
    with open(os.path.splitext(args.out)[0] + ".json", "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
