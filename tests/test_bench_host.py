"""bench.py: the host-side pieces that do not need a GPU (the workload table against BASELINE.json's configurations, SURVEY.md
section 8a; the NUMA binding helper's behaviour on a box without NVML; the output dump and argument checks) and, on a GPU,
that --dump-outputs writes what the timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_workloads_are_the_baseline_configurations():
    # SURVEY.md section 8a: B, N_s / N_t, D_s / D_t, L_t / H per configuration (cfg5: the per-GPU shard of the global batch 1024)
    want = {"cfg1": (32, 196, 196, 192, 384, 12, 6), "cfg2": (256, 196, 196, 192, 768, 12, 12), "cfg3": (256, 196, 49, 384, 2048, 1, 1),
            "cfg4": (256, 196, 196, 384, 1024, 24, 16), "cfg5": (128, 576, 576, 384, 768, 12, 12)}
    for name, (B, Ns, Nt, Ds, Dt, Lt, H) in want.items():
        w = bench.workload(0, name)
        assert (w.B, w.Ns, w.Nt, w.Ds, w.Dt, w.Lt, w.H) == (B, Ns, Nt, Ds, Dt, Lt, H), name
    assert bench.workload(64, "cfg2").B == 64                      # --batch overrides the per-GPU batch (weak scaling)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == len(want)


def test_numa_binding_is_optional():
    """Without a driver / NVML the helper returns None and leaves the affinity alone (the bench then runs unbound)."""
    before = os.sched_getaffinity(0)
    n = bench.bind_to_gpu_numa_node(0)
    assert n is None or (isinstance(n, int) and n >= 1)
    if n is None:
        assert os.sched_getaffinity(0) == before
    else:
        os.sched_setaffinity(0, before)


def test_dump_outputs_budget_and_fixed_sample(tmp_path):
    g = torch.Generator().manual_seed(0)
    # the big arrays hold their own flat indices, so what is written is the list of sampled indices
    arrays = {"loss": torch.tensor(1.5), "small": torch.randn(3, 5, generator=g, dtype=torch.float64),
              "half": torch.randn(4, 4, generator=g).bfloat16(), "big_a": torch.arange(2000.0).reshape(40, 50),
              "big_b": torch.arange(2000.0)}
    budget = 4 + 15 * 8 + 16 * 4 + 2 * 4 * 600    # the three small ones whole, then 600 float32 elements of each big array
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=budget)
    out = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in arrays}
    assert sum(a.nbytes for a in out.values()) <= budget
    assert out["loss"].dtype == np.float32 and out["loss"] == 1.5
    assert out["small"].dtype == np.float64 and np.array_equal(out["small"], arrays["small"].numpy())
    assert out["half"].dtype == np.float32 and np.array_equal(out["half"], arrays["half"].float().numpy())
    for n in ("big_a", "big_b"):
        idx = out[n]
        assert idx.dtype == np.float32 and idx.shape == (600,)
        assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < 2000     # distinct flat indices, in order
        assert np.array_equal(idx, np.load(tmp_path / "b" / f"{n}.npy"))         # same arguments, same elements
    # the sample is fixed: 4 of 10 elements are always these
    bench.dump_outputs(str(tmp_path / "c"), {"x": torch.arange(10.0)}, budget=16)
    assert np.load(tmp_path / "c" / "x.npy").tolist() == [2.0, 4.0, 5.0, 7.0]


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_step_results(tmp_path, lib, cuda_dev):
    """bench.py --dump-outputs writes the loss and gradients of its last timed step: the same values one call of the module
    returns on bench.py's inputs.  Every step on the same inputs gives the same values, so this checks what is written, not
    which step wrote it; that --steps timed steps ran shows only in the reported count."""
    import torch.nn as nn

    import vit_bias_aware_structural_distillation_b200 as pkg
    from oracle import synth
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--batch", "8", "--steps", "2",
                        "--warmup", "3", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    w = bench.workload(8, "cfg1")
    logits, targets, student, teacher, attn = bench.device_inputs(w, cuda_dev, seed=1234)
    torch.manual_seed(0)
    m = pkg.BASDLoss(nn.CrossEntropyLoss(label_smoothing=0.001), w.Ds, w.Dt, w.student_depth, w.Ns, config=synth.module_config(w),
                     teacher_has_cls_token=w.has_cls).to(cuda_dev)
    logits.requires_grad_()
    for t in student.values():
        t.requires_grad_()
    loss = m(logits, targets, student, teacher, attn)
    loss.backward()
    want = {"loss": loss, "grad_logits": logits.grad, "grad_log_temperatures": m.layer_selector.log_temperatures.grad}
    want.update({f"grad_student_{l}": t.grad for l, t in student.items()})
    assert sorted(os.listdir(tmp_path)) == sorted(f"{n}.npy" for n in want)
    assert np.load(tmp_path / "loss.npy") == np.float32(line["loss"])
    for n, t in want.items():
        got, ref = np.load(tmp_path / f"{n}.npy"), t.detach().float().cpu().numpy()
        assert got.dtype == np.float32 and got.shape == ref.shape, n
        assert np.linalg.norm(got - ref) <= 1e-5 * np.linalg.norm(ref), n
