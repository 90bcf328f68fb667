"""Cost of carrying fp32 tokens as split-bf16 pairs (BASDLoss.token_precision = "fp32") against rounding them to bf16 on entry
(the default), with fp32 student and teacher tokens.

Per configuration it times BASDLoss forward + backward per step with CUDA events after warm-up (the two modes alternate, twice),
then, in a separate pass with the library's event brackets on, the per-step time of each kernel group that the mode touches
(split_pack, project, gram, colsum, mix_teacher, polar_prep, wgrad_dots, student_grad) and of the whole bracketed path.  It also
reports how far the two modes' student gradients are apart (the rounding the default mode applies).  Teacher attention is handed
over as CLS rows [B,H,1,N+1] (the same in both modes).  The working set of every configuration exceeds the 126 MB L2.

    python tools/gpu_fp32_tokens.py --out profiles/r3_fp32_tokens.txt
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

CONFIGS = [dict(name="cfg1", B=32, N=196, Ds=192, Dt=384, Lt=12, H=6), dict(name="cfg2", B=256, N=196, Ds=192, Dt=768, Lt=12, H=12)]
P, STUDENT_DEPTH = 4, 12
SLOTS = ("split_pack", "project", "gram", "colsum", "mix_teacher", "polar_prep", "wgrad_dots", "student_grad")


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
    from vit_bias_aware_structural_distillation_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda:0")
    B, N, Ds, Dt, Lt, H = cfg["B"], cfg["N"], cfg["Ds"], cfg["Dt"], cfg["Lt"], cfg["H"]
    g = torch.Generator(device=dev).manual_seed(0)

    def spiked(r):                                   # low-rank signal + noise, fp32 (not bf16-representable)
        basis = torch.linalg.qr(torch.randn(Dt, r, device=dev, generator=g))[0]
        return (torch.randn(B, N, r, device=dev, generator=g) * 4.0) @ basis.T + torch.randn(B, N, Dt, device=dev, generator=g)
    teacher = {j: spiked(16 + 4 * j) for j in range(Lt)}
    attn = {j: torch.softmax(2 * torch.randn(B, H, 1, N + 1, device=dev, generator=g), -1) for j in range(Lt)}
    torch.manual_seed(0)
    m = pkg.BASDLoss(nn.CrossEntropyLoss(), Ds, Dt, STUDENT_DEPTH, N, config=argparse.Namespace(num_extraction_points=P),
                     teacher_has_cls_token=True).to(dev)
    basis = torch.linalg.qr(torch.randn(Ds, Ds, device=dev, generator=g))[0]
    spec = 3.0 * 0.97 ** torch.arange(Ds, device=dev)
    student = {l: ((torch.randn(B, N, Ds, device=dev, generator=g) * spec) @ basis.T).requires_grad_() for l in m.token_layers}
    logits = torch.randn(B, 1000, device=dev, generator=g).requires_grad_()
    targets = torch.randint(0, 1000, (B,), device=dev, generator=g)

    def step(mode):
        m.token_precision = mode
        loss = m(logits, targets, student, teacher, attn)
        loss.backward()
        return loss

    grads = {}
    for mode in ("bf16", "fp32"):
        for _ in range(warmup):
            for t in student.values():
                t.grad = None
            step(mode)
        grads[mode] = {l: t.grad.clone() for l, t in student.items()}
    gdiff = max(((grads["fp32"][l] - grads["bf16"][l]).norm() / grads["fp32"][l].norm()).item() for l in student)
    res = {"bf16": [], "fp32": []}
    for _ in range(2):                               # alternate the two modes: the spread of a shared host shows up
        for mode in res:
            res[mode].append(time_ms(lambda: step(mode), steps))
    slots = {}
    for mode in res:
        lib.basd_timing_reset()
        lib.basd_timing_enable(1)
        time_ms(lambda: step(mode), steps)
        lib.basd_timing_enable(0)
        slots[mode] = {k: v[0] / steps for k, v in _lib.timing_read().items()}
    lib.basd_timing_reset()
    tok_bytes = 4 * B * N * (Lt * Dt + P * Ds)
    log(f"config {cfg['name']}: B={B} N={N} D_s={Ds} D_t={Dt} L_t={Lt} P={P}, fp32 student and teacher tokens ({tok_bytes / 1e9:.2f} GB per step)")
    for mode, label in (("bf16", 'default (rounded to bf16) '), ("fp32", 'token_precision="fp32"   ')):
        log(f"  step {label}: " + ", ".join(f"{t:.3f}" for t in res[mode]) + " ms")
    ratio = min(res["fp32"]) / min(res["bf16"])
    log(f"  fp32 mode / default: {ratio:.3f} (best of each)")
    log("  kernel groups, ms per step (CUDA-event brackets):   default    fp32 mode")
    for k in SLOTS:
        log(f"    {k:14s}                                     {slots['bf16'][k]:8.3f}   {slots['fp32'][k]:8.3f}")
    tot = {mode: sum(slots[mode].values()) for mode in slots}
    log(f"    {'all brackets':14s}                                     {tot['bf16']:8.3f}   {tot['fp32']:8.3f}")
    log(f"  student gradients, fp32 mode vs default: {gdiff:.2e} Frobenius-relative (worst point)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
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
