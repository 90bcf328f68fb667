"""Teacher attention capture without a CLS token: the reference-style hook (full softmax(q k^T * scale) map per layer, the
loss reading every map) against query_mean_attention (query-mean rows per layer, the loss reading those).

Per step and configuration it times, with CUDA events after warm-up,
  (a) softmax(q @ k^T * scale) per teacher layer (bf16, what src/models/teacher.py:27-39 builds) + BASDLoss fwd+bwd on the maps,
  (b) query_mean_attention(q, k) per teacher layer + BASDLoss fwd+bwd on the rows,
and the kernel alone per layer, its FLOP/s against the 2 * 2 * B * H * S^2 * dh it performs, and the bytes the rows save.
q and k are strided views of one fused qkv tensor per layer (timm layout); that working set exceeds the 126 MB L2.

    python tools/gpu_query_mean_attention.py --out profiles/qm_attention.txt
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = [dict(B=256, N=196, H=12, dh=64, Lt=12), dict(B=128, N=576, H=12, dh=64, Lt=12)]
DS, DT, P, STUDENT_DEPTH = 192, 768, 4, 12


def gpu_info() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                      # (the name still comes from torch)
        q = f"nvidia-smi unavailable: {e}"
    return f"{torch.cuda.get_device_name(0)} | nvidia-smi: {q}"


def time_ms(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps


def run(cfg, warmup, steps, log):
    import vit_bias_aware_structural_distillation_b200 as pkg
    dev = torch.device("cuda:0")
    B, N, H, dh, Lt = cfg["B"], cfg["N"], cfg["H"], cfg["dh"], cfg["Lt"]
    g = torch.Generator(device=dev).manual_seed(0)
    qkv = [torch.randn(B, N, 3, H, dh, device=dev, generator=g).bfloat16() for _ in range(Lt)]
    qk = [tuple(t.permute(2, 0, 3, 1, 4).unbind(0)[:2]) for t in qkv]
    def spiked(r):                                   # low-rank signal + noise (i.i.d. tokens have Marchenko-Pastur rank 0)
        basis = torch.linalg.qr(torch.randn(DT, r, device=dev, generator=g))[0]
        return ((torch.randn(B, N, r, device=dev, generator=g) * 4.0) @ basis.T + torch.randn(B, N, DT, device=dev, generator=g)).bfloat16()
    teacher = {j: spiked(16 + 4 * j) for j in range(Lt)}
    torch.manual_seed(0)
    m = pkg.BASDLoss(nn.CrossEntropyLoss(), DS, DT, STUDENT_DEPTH, N, config=argparse.Namespace(num_extraction_points=P),
                     teacher_has_cls_token=False).to(dev)
    basis = torch.linalg.qr(torch.randn(DS, DS, device=dev, generator=g))[0]
    spec = 3.0 * 0.985 ** torch.arange(DS, device=dev)
    student = {l: ((torch.randn(B, N, DS, device=dev, generator=g) * spec) @ basis.T).bfloat16().requires_grad_() for l in m.token_layers}
    logits = torch.randn(B, 1000, device=dev, generator=g).requires_grad_()
    targets = torch.randint(0, 1000, (B,), device=dev, generator=g)
    scale = dh ** -0.5

    def maps():
        return {j: torch.softmax((q @ k.transpose(-2, -1)) * scale, dim=-1) for j, (q, k) in enumerate(qk)}

    def rows():
        return {j: pkg.query_mean_attention(q, k, scale) for j, (q, k) in enumerate(qk)}

    def step(capture):
        loss = m(logits, targets, student, teacher, capture())
        loss.backward()
        return loss

    losses = {}
    for name, cap in (("a_full_maps", maps), ("b_query_mean_rows", rows)):
        for _ in range(warmup):
            losses[name] = step(cap).item()
    res = {"a_full_maps": [], "b_query_mean_rows": []}
    for _ in range(2):                               # alternate the two arms: the spread of a shared host shows up
        res["a_full_maps"].append(time_ms(lambda: step(maps), steps))
        res["b_query_mean_rows"].append(time_ms(lambda: step(rows), steps))
    q0, k0 = qk[0]
    for _ in range(warmup):
        pkg.query_mean_attention(q0, k0, scale)
    kern = [time_ms(lambda: [pkg.query_mean_attention(q, k, scale) for q, k in qk], steps) / Lt for _ in range(2)]
    hook = [time_ms(lambda: [torch.softmax((q @ k.transpose(-2, -1)) * scale, dim=-1) for q, k in qk], steps) / Lt for _ in range(2)]
    flop = 2 * 2 * B * H * N * N * dh
    map_bytes = Lt * B * H * N * N * 2               # bf16 maps: written by the hook, read by the loss
    row_bytes = Lt * B * H * N * 4                   # fp32 rows
    ref_rows = torch.softmax((q0.double() @ k0.double().transpose(-2, -1)) * scale, -1).mean(2, keepdim=True)
    err = ((pkg.query_mean_attention(q0, k0, scale).double() - ref_rows).norm() / ref_rows.norm()).item()
    log(f"config B={B} N={N} H={H} dh={dh} L_t={Lt} D_s={DS} D_t={DT} P={P} (teacher without CLS, bf16 q/k as fused-qkv views)")
    log(f"  step (a) full maps + loss fwd+bwd   : " + ", ".join(f"{t:.3f}" for t in res["a_full_maps"]) + " ms")
    log(f"  step (b) query-mean rows + loss     : " + ", ".join(f"{t:.3f}" for t in res["b_query_mean_rows"]) + " ms")
    log(f"  hook softmax(q k^T) per layer       : " + ", ".join(f"{t * 1e3:.1f}" for t in hook) + " us")
    log(f"  query_mean_attention per layer      : " + ", ".join(f"{t * 1e3:.1f}" for t in kern) + " us"
        f"  -> {flop / (min(kern) * 1e-3) / 1e12:.1f} TFLOP/s on {flop / 1e9:.2f} GFLOP (2*2*B*H*S^2*dh)")
    log(f"  attention bytes per step            : maps {map_bytes / 1e9:.2f} GB written + read; rows {row_bytes / 1e6:.1f} MB "
        f"({(map_bytes - row_bytes) / 1e9:.2f} GB not written, as much not read; the same not copied by HostStager)")
    log(f"  loss on maps {losses['a_full_maps']:.6f}, on rows {losses['b_query_mean_rows']:.6f} (maps rounded to bf16); "
        f"layer-0 rows vs fp64: {err:.2e} Frobenius-relative")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log(f"GPU: {gpu_info()}")
    for cfg in CONFIGS:
        run(cfg, args.warmup, args.steps, log)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
