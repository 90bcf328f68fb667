#!/usr/bin/env python
"""bench.py — BASD loss fwd+bwd samples/s (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path  (one JSON line on rank 0)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own PyTorch loss on the host CPU cores

A "step" is one forward + backward of the BASD loss (selector + interpolation + Procrustes + UW-SO, gradients to the P
student tensors and log_temperatures) on synthetic activations of BASELINE.json configs[1]
(DeiT-Ti <- DeiT-B, 224 px, 196 tokens, batch 256 per GPU, bf16 tokens).  Backbones are excluded (SURVEY.md §8d).
`value` is measured with the inputs resident in HBM; `e2e` goes through the same public module call but copies every
input from pinned host memory each step and reads the loss back.  Multi-GPU: weak scaling, batch sharded, pooled
statistics all-reduced over NCCL (two small collectives per step).
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

METRIC = "BASD loss fwd+bwd samples/s (DeiT-Ti<-DeiT-B, 224px)"
UNIT = "samples/s"


# ------------------------------------------------------------------------------------------------ workload
def workload(batch, name: str = "cfg2"):
    """BASELINE.json configs[1] (the configuration the metric is quoted on) unless another one is named."""
    from oracle import synth
    w = synth.CONFIGS[name]
    return dataclasses.replace(w, B=batch) if batch else w


def algorithmic_bytes(w, act_bytes=2, attn_bytes=2):
    """SURVEY.md §8(d): W_alg = 2 X_T + 4 X_S + A_needed (per step)."""
    xt = w.Lt * w.B * w.Nt * w.Dt * act_bytes
    xs = w.P * w.B * w.Ns * w.Ds * act_bytes
    an = w.Lt * w.B * w.H * w.Nt * attn_bytes if w.has_cls else w.Lt * w.B * w.H * w.Nt * w.Nt * attn_bytes
    return 2 * xt + 4 * xs + an


def tensor_flops(w):
    """SURVEY.md §8(d): F_tc (algorithmic tensor-core flops per step)."""
    return 2 * w.B * (w.Lt * w.Nt * w.Ds * (w.Dt + w.Ds) + 2 * w.P * w.Ns * w.Ds ** 2 + 3 * w.P * w.Ns * w.Ds * w.Dt)


def device_inputs(w, dev, seed, structure_seed=1234):
    """Spiked synthetic activations (SURVEY.md Appendix D) generated on the device.  `seed` draws the samples (one stream
    per rank); the signal subspaces of the layers - the distribution the samples come from - are drawn from `structure_seed`,
    the same on every rank: a batch-sharded job sees ONE dataset.  (With per-rank subspaces the pooled teacher covariance of N
    ranks carries N times the spikes, the Marchenko-Pastur ranks grow with N up to the D_s - 1 clamp and the 'weak scaling'
    run measures a different problem at every N: that, not the all-reduces, was 0.36 of the 0.43 ms lost at N = 2.)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    gs = torch.Generator(device=dev).manual_seed(structure_seed)

    def spiked(B, N, D, r):
        basis = torch.linalg.qr(torch.randn(D, r, generator=gs, device=dev))[0]
        amp = 4.0 * torch.linspace(1.0, 0.2, r, device=dev)
        return ((torch.randn(B, N, r, generator=g, device=dev) * amp) @ basis.T + torch.randn(B, N, D, generator=g, device=dev)).bfloat16()

    def geometric(B, N, D, rho=0.985, amp=3.0):
        basis = torch.linalg.qr(torch.randn(D, D, generator=gs, device=dev))[0]
        return ((torch.randn(B, N, D, generator=g, device=dev) * (amp * rho ** torch.arange(D, device=dev))) @ basis.T).bfloat16()

    logits = torch.randn(w.B, w.num_classes, generator=g, device=dev)
    targets = torch.randint(0, w.num_classes, (w.B,), generator=g, device=dev)
    student = {l: geometric(w.B, w.Ns, w.Ds) for l in w.token_layers()}
    teacher = {j: spiked(w.B, w.Nt, w.Dt, (16 + 4 * j) if w.Lt > 1 else 64) for j in range(w.Lt)}
    if w.has_cls:
        attn = {j: torch.softmax(2 * torch.randn(w.B, w.H, w.Nt + 1, w.Nt + 1, generator=g, device=dev), -1).bfloat16() for j in range(w.Lt)}
    else:                                  # CNN teachers: uniform attention (teacher.py:188-191)
        attn = {j: (torch.ones(w.B, 1, w.Nt, w.Nt, device=dev) / w.Nt).bfloat16() for j in range(w.Lt)}
    return logits, targets, student, teacher, attn


DUMP_BYTES = 60 << 20          # payload of all .npy files together; headers keep the total under 64 MB


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Writes {name: tensor} as out_dir/<name>.npy: float64 stays float64, every other dtype becomes float32 (exact for bf16).
    Smaller arrays are written whole first; an array larger than its share of what is left of `budget` is written as the
    1-D sample of its flattened elements at sorted flat indices drawn with numpy's default_rng(0), so runs with the same
    arguments write the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    todo = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = budget
    for i, (name, t) in enumerate(todo):
        t = t.detach().cpu()
        a = (t if t.dtype == torch.float64 else t.float()).numpy()
        k = min(a.size, left // (len(todo) - i) // a.itemsize)
        if k < a.size:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        left -= a.nbytes


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """One streaming `nvidia-smi -lms 50` process (a fresh nvidia-smi per sample takes longer than a short timed region)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.proc = index, [], None
        self.t_start = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append((time.perf_counter(), [x.strip() for x in line.strip().split(",")]))
        except Exception:
            pass

    def mark(self):
        """Start of the timed region: only samples taken after this are reported."""
        self.t_start = time.perf_counter()

    def finish(self):
        t_end = time.perf_counter()
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=3)
        rows = [s for t, s in self.samples if self.t_start is None or (self.t_start <= t <= t_end + 0.05)]
        if not rows:
            rows = [s for _, s in self.samples[-1:]]
        sm = sorted(int(float(s[1])) for s in rows if len(s) > 2 and s[1].replace(".", "").isdigit())
        mx = [int(float(s[2])) for s in rows if len(s) > 2 and s[2].replace(".", "").isdigit()]
        pw = [float(s[3]) for s in rows if len(s) > 3 and s[3].replace(".", "").isdigit()]
        reasons = set()
        for s in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(rows), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------ reference / CPU arm
def cpu_reference_step_fn(w, sample_batch):
    """Returns (step callable, kind, description).  kind 'reference' = the unmodified reference module copied by the
    survey into the git-ignored baseline/_ref (travels with gpurun); 'port' = oracle/basd_oracle.py."""
    from oracle import basd_oracle, synth
    ws = dataclasses.replace(w, B=sample_batch)
    inp = synth.make_inputs(ws)
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    kind = "port"
    if os.path.isdir(os.path.join(ref_root, "src", "losses")):
        try:
            sys.path.insert(0, ref_root)
            from src.losses.combined import BASDLoss as RefLoss  # the reference itself
            kind = "reference"
        except Exception:
            kind = "port"
    torch.manual_seed(0)
    if kind == "reference":
        m = RefLoss(nn.CrossEntropyLoss(label_smoothing=0.001), ws.Ds, ws.Dt, ws.student_depth, ws.Ns,
                    config=synth.module_config(ws), teacher_has_cls_token=ws.has_cls)
        S = {l: v.float().requires_grad_() for l, v in inp["student"].items()}
        T = {j: v.float() for j, v in inp["teacher"].items()}
        logits = inp["logits"].clone().requires_grad_()

        def step():
            for t in S.values():
                t.grad = None
            m.zero_grad(set_to_none=True)
            loss = m(logits, inp["targets"], S, T, inp["attn"])
            loss.backward()
            return float(loss)
    else:
        proj_s = torch.empty(ws.Ds, ws.Ds); proj_t = torch.empty(ws.Ds, ws.Dt)
        nn.init.orthogonal_(proj_s); nn.init.orthogonal_(proj_t)
        import math
        logt = torch.full((ws.P,), math.log(math.e - 1))

        def step():
            out = basd_oracle.run_case(inp, proj_s, proj_t, logt, ws.token_layers(), has_cls=ws.has_cls, n_student_tokens=ws.Ns,
                                       label_smoothing=0.001)
            return float(out["loss"])
    desc = f"{ws.name.replace(str(w.B), str(sample_batch))}: batch {sample_batch} of the same shapes, fp32, no autocast"
    return step, kind, desc


def time_cpu(step, steps, warmup):
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return sum(ts) / len(ts)


def host_ram_gb():
    try:
        import psutil
        return psutil.virtual_memory().available / 1e9
    except Exception:
        return 0.0


def run_reference_arm(args):
    """bench.py --impl reference: the UNMODIFIED reference (baseline/_ref; oracle port if absent) on the host cores, on OUR
    arm's configuration - the full per-GPU batch when the host has the RAM for the reference's [L_t,B,H,N+1,N+1] attention
    stack (same_config: true), a batch-32 sample of the same shapes otherwise - and for as many of the K steps as fit ~2.5
    minutes (at least one; the count is reported as `steps`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    w = workload(args.batch, args.workload)
    # fp32 attention stack + its mixed copies + autograd temporaries: ~ 6 x L_t B H (N+1)^2 x 4 bytes
    need_gb = 6 * w.Lt * w.B * w.H * (w.Nt + 1) ** 2 * 4 / 1e9 + 8
    full = args.cpu_sample_batch <= 0 or (args.cpu_sample_batch == 32 and host_ram_gb() > need_gb and w.B <= 256)
    sample = w.B if full else min(args.cpu_sample_batch, w.B)
    step, kind, desc = cpu_reference_step_fn(w, sample)
    budget_s = 150.0
    t_begin = time.perf_counter()
    step()                                                    # warm-up (allocator, thread pool)
    ts = []
    for _ in range(max(1, args.steps)):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin + ts[-1] > budget_s:
            break
    sec = sum(ts) / len(ts)
    val = sample / sec
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(ts),
            "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": w.name, "sample": desc, "same_config": sample == w.B, "steps_requested": args.steps, "l2": "cpu"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": desc},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
_ORIGINAL_AFFINITY = None


def bind_to_gpu_numa_node(index):
    """One process per GPU: run on the CPUs next to that GPU (NVML's ideal affinity), so the pinned host buffers of the end-to-end
    leg are first touched on the GPU's own NUMA node and eight ranks do not share one socket's memory controllers.  Returns the
    number of CPUs the process is bound to (None when NVML or the call is unavailable - the bench runs unbound then)."""
    global _ORIGINAL_AFFINITY
    try:
        import pynvml
        _ORIGINAL_AFFINITY = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        n = len(os.sched_getaffinity(0))
        torch.set_num_threads(max(1, min(torch.get_num_threads(), n)))
        return n
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (weak scaling); 0 = the named configuration's own (256; cfg5: 128)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json configs[0..4]; the metric is quoted on cfg2")
    ap.add_argument("--cpu-sample-batch", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--views", action="store_true",
                    help="hand the tokens over as the CLS-stripped views out[:, 1:, :] of [B, N+1, D] tensors, like trainer.py:29 / teacher.py:157 do "
                         "(consumed in place; default: dense tensors)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what rank 0's last timed step returned (loss, gradients of the logits, of "
                         "log_temperatures and of each student tensor) as DIR/<name>.npy, float32; arrays past a 60 MiB total "
                         "are written as a fixed seeded sample of their elements (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpu_affinity = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as graft
    if not os.path.exists(graft.LIB):
        graft.build()
    import vit_bias_aware_structural_distillation_b200 as pkg
    from vit_bias_aware_structural_distillation_b200 import _lib
    lib = pkg.load()

    w = workload(args.batch, args.workload)
    from oracle import synth
    logits, targets, student, teacher, attn = device_inputs(w, dev, seed=1234 + rank)
    torch.manual_seed(0)
    m = pkg.BASDLoss(nn.CrossEntropyLoss(label_smoothing=0.001), w.Ds, w.Dt, w.student_depth, w.Ns, config=synth.module_config(w),
                     teacher_has_cls_token=w.has_cls).to(dev)
    if args.views:
        def cls_view(t):
            full = torch.zeros(t.shape[0], t.shape[1] + 1, t.shape[2], device=t.device, dtype=t.dtype)
            full[:, 1:] = t
            return full[:, 1:, :]
        student = {k: cls_view(v) for k, v in student.items()}
        teacher = {k: cls_view(v) for k, v in teacher.items()}
    logits.requires_grad_()
    for t in student.values():
        t.requires_grad_()

    def step(lg, tg, st, te, at):
        for t in st.values():
            t.grad = None
        m.zero_grad(set_to_none=True)
        lg.grad = None
        loss = m(lg, tg, st, te, at)
        loss.backward()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(logits, targets, student, teacher, attn)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)                       # let the streaming nvidia-smi come up before the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark()
    lib.basd_timing_reset()               # (resets the launch counter too; the per-kernel event brackets stay off here)
    e0.record()
    for _ in range(args.steps):
        loss = step(logits, targets, student, teacher, attn)
    e1.record()
    barrier()
    clocks = sampler.finish()
    ms_total = e0.elapsed_time(e1)
    launches = int(lib.basd_launch_count())
    if args.dump_outputs and rank == 0:
        outs = {"loss": loss, "grad_logits": logits.grad, "grad_log_temperatures": m.layer_selector.log_temperatures.grad}
        outs.update({f"grad_student_{l}": t.grad for l, t in student.items()})
        dump_outputs(args.dump_outputs, outs)
    # per-kernel breakdown: the same steps again with a CUDA-event bracket around every launch group (kept out of the
    # timed region above: ~150 event records per step cost 0.1-0.2 ms and keep consecutive kernels from overlapping)
    lib.basd_timing_reset()
    lib.basd_timing_enable(1)
    breakdown_steps = min(args.steps, 10)
    for _ in range(breakdown_steps):
        step(logits, targets, student, teacher, attn)
    barrier()
    lib.basd_timing_enable(0)
    kern = _lib.timing_read()
    t_ms = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_step = t_ms.item() / args.steps
    value = world * w.B / (ms_step * 1e-3)
    loss_val = float(loss.detach())

    # ---- end to end: every step's inputs start in pinned HOST memory and go through the public host-buffer API
    # (HostStager: copy stream + double-buffered device slots, so the transfer of step i+1 overlaps the loss of step i;
    # of the attention maps only the CLS rows the loss reads are gathered and copied); the loss is read back every step.
    e2e = None
    if not args.no_e2e:
        host = {"logits": logits.detach().cpu().pin_memory(), "targets": targets.cpu().pin_memory(),
                "student": {k: v.detach().cpu().pin_memory() for k, v in student.items()},
                "teacher": {k: v.cpu().pin_memory() for k, v in teacher.items()},
                "attn": {k: v.cpu().pin_memory() for k, v in attn.items()}}
        del attn, teacher
        torch.cuda.empty_cache()
        stager = pkg.HostStager(m, dev)

        def submit():
            return stager.submit(host["logits"], host["targets"], host["student"], host["teacher"], host["attn"])

        def finish(h):
            m.zero_grad(set_to_none=True)
            out = stager.run(h)
            out.backward()
            return out.item()                      # device -> host read of the step's result

        nxt = submit()
        for _ in range(2):                         # warm the pipeline (allocates both slots)
            cur, nxt = nxt, submit()
            finish(cur)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cur, nxt = nxt, submit()               # copies of the next step are in flight while this one computes
            finish(cur)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * w.B * args.steps / dt.item(), "unit": UNIT, "h2d_bytes_per_step": int(stager.h2d_bytes_last), "d2h_bytes_per_step": 4,
               "api": "HostStager.submit/run (host buffers -> copy stream -> BASDLoss.forward/backward), 2-deep pipeline",
               "host_attention_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host["attn"].values()))}
        del host

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tc_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    per_step = {k: v[0] / breakdown_steps for k, v in kern.items() if v[1] > 0}
    dom = max(per_step, key=per_step.get) if per_step else None
    w_alg = algorithmic_bytes(w)
    f_tc = tensor_flops(w)
    # dominant kernel: algorithmic work per launch / its average launch duration (CUDA events on the launching stream)
    n_prob = w.P * w.B
    ksteps = int(lib.basd_polar_steps())
    per_ns_step = int(lib.basd_polar_launches_per_step(w.Ds, w.Ns))      # 3: A = T W^T and the polynomial in A fused (A stays on chip)
    polar_launches = per_ns_step * ksteps + 2
    polar_flops = n_prob * (ksteps * (2 * w.Ds * w.Ns * w.Ns + 2 * w.Ds * w.Ds * w.Ns + 2 * w.Ds ** 3 + 2 * w.Ds * w.Ds * w.Ns)
                            + 2 * w.Ns * w.Ns * w.Ds + 2 * w.Ns * w.Ds * w.Ns)
    # polar_gemm as launched: every product streams its split-bf16 (hi + lo = 4 B per element) operands in and its result
    # out once per launch; these are the algorithmic bytes of the MULTI-LAUNCH formulation (unpadded), DESIGN.md section 5
    D, N = w.Ds, w.Ns
    ab_bytes = (2 * D * N + D * D) if per_ns_step == 3 else (2 * D * N + D * D) + 2 * D * D      # fused: T, W in, Bm out
    polar_bytes = n_prob * 4 * (ksteps * ((2 * D * N + N * N) + ab_bytes + (D * D + 2 * D * N))
                                + (N * N + D * N + N * D) + (2 * N * D + N * N))
    eig_bytes = 4 * ((w.Lt + w.P) * (D * D + D) + (w.Lt + w.P) * (2 * D * D + D))
    table = {   # slot -> (bound, algorithmic units per step, launches per step, description)
        "polar_gemm": ("hbm", polar_bytes, polar_launches,
                       f"Newton-Schulz polar iteration, ({per_ns_step} x steps + 2) batched launches per step: split-bf16 operands read once and the "
                       "result written once per launch (4 B per element, unpadded).  Tensor view of the same kernel: "
                       f"{polar_flops / polar_launches / 1e9:.1f} GFLOP of plain 2mnk per launch (3 split MMAs per product not counted)"),
        "pooled_eig": ("hbm", eig_bytes, 1,
                       f"{w.Lt + w.P} eigenproblems (Cholesky + one-sided Jacobi, fp32 CUDA cores; MP ranks from the secular equation), one thread-block "
                       "cluster each: a dependent-latency chain, neither roofline applies; bytes = Gram statistics in, eigenpairs out"),
    }
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tr.get(dom, {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    feature_form = w.Ds <= min(w.Ns, w.Nt) - 1          # the byte model above is the student-feature form's
    # SURVEY.md section 8(d): the Procrustes stage's share of the algorithmic tensor flops F_tc is the cross-covariance
    # s_w^T t_w (forward) and the two products with the polar factor (backward): 3 x 2 N_s D_s D_t per (point, sample).
    # The Newton-Schulz products that replace the batched SVD are implementation extras and do not count.
    procrustes_flops = 3 * 2 * n_prob * w.Ns * w.Ds * w.Dt
    if dom == "polar_gemm":
        n_l = polar_launches if feature_form else None
        ms_dom = per_step[dom]
        ach_tf = procrustes_flops / (ms_dom * 1e-3) / 1e12
        roofline = {"bound": "tensor", "achieved": ach_tf, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach_tf / tc_peak, "traffic": traffic,
                    "kernel": dom,
                    "what": "Procrustes stage (relational.py:47-48 and its backward) = the launches of the Newton-Schulz polar iteration; achieved = "
                            "its SURVEY 8(d) share of F_tc (3 x 2 N_s D_s D_t flops per point and sample) / the stage's time per step, "
                            "against the measured sustained bf16 peak",
                    "algorithmic_flops_per_step": procrustes_flops, "ms_per_step": ms_dom}
        if feature_form:
            ms_launch = ms_dom / n_l
            fb = polar_bytes / n_l / (ms_launch * 1e-3) / 1e9
            roofline.update({"launches_per_step": n_l, "avg_launch_ms": ms_launch, "algorithmic_flops_per_launch": procrustes_flops / n_l})
            roofline["formulation_view"] = {
                "what": table[dom][3], "bound": "hbm", "bytes_per_launch": polar_bytes / n_l, "achieved_gbs": fb, "peak_gbs": hbm_peak,
                "frac": fb / hbm_peak, "plain_2mnk_tflops": polar_flops / n_l / (ms_launch * 1e-3) / 1e12,
                "note": "how well the launches stream the operands of THIS formulation (14.8 GB per step at cfg2); not the section 8(d) quantity"}
    elif dom in table and table[dom][1] > 0 and feature_form:
        bound, units, n_l, what = table[dom]
        ms_launch = per_step[dom] / n_l
        ach = units / n_l / (ms_launch * 1e-3) / 1e9
        roofline = {"bound": bound, "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic,
                    "kernel": dom, "what": what, "launches_per_step": n_l, "avg_launch_ms": ms_launch,
                    "algorithmic_bytes_per_launch": units / n_l}
    else:
        achieved = w_alg / (ms_step * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                    "kernel": "whole step"}
    roofline.update({
        "peak_source": peak_src,
        "step": {"hbm": {"algorithmic_bytes_per_step": w_alg, "achieved_gbs": w_alg / (ms_step * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                         "frac": w_alg / (ms_step * 1e-3) / 1e9 / hbm_peak},
                 "tensor": {"algorithmic_flops_per_step": f_tc, "achieved_tflops": f_tc / (ms_step * 1e-3) / 1e12, "peak_tflops": tc_peak,
                            "frac": f_tc / (ms_step * 1e-3) / 1e12 / tc_peak},
                 "scope": "W_alg = 2 X_T + 4 X_S + A_needed and F_tc of SURVEY.md section 8d over the whole step time"},
        "other_kernels": {k: {"bound": table[k][0], "achieved_gbs": table[k][1] / table[k][2] / (per_step[k] / table[k][2] * 1e-3) / 1e9,
                              "frac": table[k][1] / table[k][2] / (per_step[k] / table[k][2] * 1e-3) / 1e9 / hbm_peak,
                              "ms_per_step": per_step[k]} for k in table if k != dom and k in per_step and feature_form},
        "dominant_kernel": dom, "dominant_kernel_ms_per_step": per_step.get(dom) if dom else None,
        "dominant_kernel_share": (per_step[dom] / ms_step) if dom else None,
        "kernel_ms_per_step": {k: round(v, 4) for k, v in sorted(per_step.items(), key=lambda kv: -kv[1])}})

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        if _ORIGINAL_AFFINITY is not None:           # the CPU baseline uses every host core, not just the GPU's NUMA node
            os.sched_setaffinity(0, _ORIGINAL_AFFINITY)
        torch.set_num_threads(os.cpu_count() or 1)
        cpu_b = min(args.cpu_sample_batch, w.B)
        stepfn, kind, desc = cpu_reference_step_fn(w, cpu_b)
        sec = time_cpu(stepfn, 3, 1)
        cpu_baseline = {"value": cpu_b / sec, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": desc}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": w.name, "per_gpu_batch": w.B, "global_batch": w.B * world, "Ns": w.Ns, "Nt": w.Nt, "Ds": w.Ds, "Dt": w.Dt,
                       "Lt": w.Lt, "H": w.H, "P": w.P, "token_tensors": "CLS-stripped [:,1:,:] views, consumed in place" if args.views else "dense",
                       "parallelism": f"dp{world} (batch-sharded, pooled statistics all-reduced)",
                       "arithmetic": "bf16 tokens, fp32 accumulation, split-bf16 (hi+lo) tensor-core products, fp32 Jacobi",
                       "l2": f"inputs ({(w.Lt * w.B * w.Nt * w.Dt + w.P * w.B * w.Ns * w.Ds) * 2 / 1e9:.1f} GB of tokens per step) exceed the 126 MB L2; no explicit flush"},
            "clocks": clocks, "e2e": e2e, "cpu_affinity": cpu_affinity, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline, "loss": loss_val}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
