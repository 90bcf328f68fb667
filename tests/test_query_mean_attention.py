"""Query-mean attention rows for teachers without a CLS token: the kernel (basd_query_mean_attention) against an fp64
softmax(q k^T * scale).mean(2), the loss fed with those rows (basd_shape.has_cls = BASD_ATTN_QUERY_MEAN) against the oracle on the
full maps and against the same module on the full maps, the standalone pair loss and the host-staged path.  CPU tests check
the ABI and the argument checks; the rest is marked gpu."""
import ctypes
import os

import pytest
import torch
import torch.nn as nn

from oracle import basd_oracle as O
from oracle import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL_LOSS, TOL_TGRAD, TOL_SGRAD = 1e-3, 1e-3, 1e-2


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30)).item()


# ------------------------------------------------------------------------------------------------ CPU: ABI and argument checks
def test_symbol_declared_and_exported(lib):
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "basd_b200.h")).read()
    assert "int basd_query_mean_attention(" in text and "#define BASD_ATTN_QUERY_MEAN 2" in text
    assert hasattr(lib, "basd_query_mean_attention")
    import vit_bias_aware_structural_distillation_b200 as pkg
    assert callable(pkg.query_mean_attention) and "query_mean_attention" in pkg.__all__


def test_workspace_bytes_accepts_query_mean_rows(lib):
    from vit_bias_aware_structural_distillation_b200._lib import ATTN_QUERY_MEAN, Shape
    n0, n2 = ctypes.c_size_t(), ctypes.c_size_t()
    kw = dict(B=256, Ns=196, Nt=196, Ds=192, Dt=768, Lt=12, P=4, H=12, act_dtype=1, attn_dtype=0, world_size=1)
    assert lib.basd_workspace_bytes(ctypes.byref(Shape(has_cls=0, **kw)), ctypes.byref(n0)) == 0
    assert lib.basd_workspace_bytes(ctypes.byref(Shape(has_cls=ATTN_QUERY_MEAN, **kw)), ctypes.byref(n2)) == 0, lib.basd_last_error().decode()
    assert n0.value == n2.value
    for bad in (3, -1):
        assert lib.basd_workspace_bytes(ctypes.byref(Shape(has_cls=bad, **kw)), ctypes.byref(n2)) != 0
        assert "has_cls" in lib.basd_last_error().decode()


def _call(lib, B=2, H=3, S=196, dh=64, dtype=1, qs=None, ks=None, q=256, k=512):
    qs = qs or (H * S * dh, S * dh, dh, 1)
    ks = ks or qs
    return lib.basd_query_mean_attention(q, k, dtype, B, H, S, dh, (ctypes.c_int64 * 4)(*qs), (ctypes.c_int64 * 4)(*ks), 0.125, 1024, None)


@pytest.mark.parametrize("kw,needle", [(dict(dh=60), "multiple of 8"), (dict(dh=264), "multiple of 8"), (dict(dh=0), "multiple of 8"),
                                       (dict(S=0), "S=0"), (dict(S=4096), "S=4096"), (dict(B=0), "invalid B"),
                                       (dict(qs=(3 * 196 * 64, 196 * 64, 64, 2)), "head-dim stride"),
                                       (dict(qs=(3 * 196 * 68, 196 * 68, 68, 1), dh=64, S=196), "multiples of 8"),
                                       (dict(q=264), "16-byte aligned"), (dict(dtype=5), "dtype")])
def test_entry_point_rejects_bad_arguments(lib, kw, needle):
    """Validated on the host before anything reaches a device (the pointers here are never dereferenced)."""
    assert _call(lib, **kw) != 0
    assert needle in lib.basd_last_error().decode()


def test_python_entry_rejects_mismatched_shapes_and_cpu_tensors(lib):
    import vit_bias_aware_structural_distillation_b200 as pkg
    q = torch.randn(2, 3, 49, 64)
    with pytest.raises(pkg.BasdError, match="must both be"):
        pkg.query_mean_attention(q, torch.randn(2, 3, 50, 64))
    with pytest.raises(pkg.BasdError, match="must both be"):
        pkg.query_mean_attention(q[0], q[0])
    with pytest.raises(pkg.BasdError, match="CUDA tensors required"):
        pkg.query_mean_attention(q, torch.randn(2, 3, 49, 64))


# ------------------------------------------------------------------------------------------------ GPU: the kernel
def _qk(B, H, S, dh, dt, strided, mul, seed, bf16_values=False):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, S, 3, H, dh, generator=g)
    qkv[:, :, 0] *= mul
    if dt == torch.bfloat16 or bf16_values:
        qkv = qkv.bfloat16()
    qkv = qkv.to(dt)
    if strided:                                      # timm: reshape(B, S, 3, H, dh).permute(2, 0, 3, 1, 4)
        q, k, _ = qkv.permute(2, 0, 3, 1, 4).unbind(0)
    else:
        q, k = (qkv[:, :, i].permute(0, 2, 1, 3).contiguous() for i in range(2))
    return q, k


def _reference(q, k):
    return torch.softmax((q.double() @ k.double().transpose(-2, -1)) * q.shape[-1] ** -0.5, dim=-1).mean(2, keepdim=True)


def _check(pkg, q, k, tol):
    out = pkg.query_mean_attention(q, k)
    ref = _reference(q, k)
    assert out.shape == (q.shape[0], q.shape[1], 1, q.shape[2]) and out.dtype == torch.float32
    assert torch.isfinite(out).all()
    err = rel(out, ref)
    assert err <= tol, f"Frobenius-relative error {err:.3e}"
    assert (out.double().sum(-1) - 1).abs().max().item() <= 1e-5
    assert torch.equal(out, pkg.query_mean_attention(q, k))          # fixed-order sums: bitwise repeatable
    return out


SIZES = [1, 7, 49, 128, 129, 196, 256, 577, 1024]
DHS, HEADS = [32, 64, 72, 128], [1, 3, 12]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("S", SIZES)
def test_kernel_against_fp64_softmax(lib, cuda_dev, S, dt):
    """Every token count crosses every head width and head count over the sizes; each size runs strided fused-qkv views and
    contiguous tensors, plain and with q scaled x30 (near one-hot rows)."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    i0 = SIZES.index(S)
    for i, (strided, mul) in enumerate([(True, 1.0), (False, 1.0), (True, 30.0), (False, 30.0)]):
        dh, H = DHS[(i0 + i) % 4], HEADS[(i0 + i) % 3]
        q, k = _qk(2, H, S, dh, dt, strided, mul, seed=100 * i0 + i)
        # fp32 runs as split-bf16 pairs: operands resolved to ~2^-17 relative, so logits of magnitude ~100 (q x30) carry ~1e-5
        # absolute error and the mean rows ~2e-5 relative (an fp32 emulation of the three-term product shows 1.8e-5 there)
        tol = 3e-5 if (dt == torch.float32 and mul == 30.0) else 1e-5
        _check(pkg, q.to(cuda_dev), k.to(cuda_dev), tol)
        if dt == torch.float32 and mul == 30.0:
            # the same near one-hot rows from fp32 tensors that hold bf16 values: the split is exact, so is the product
            qb, kb = _qk(2, H, S, dh, dt, strided, mul, seed=100 * i0 + i, bf16_values=True)
            _check(pkg, qb.to(cuda_dev), kb.to(cuda_dev), 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("dh", [8, 88, 136, 200, 256])
def test_kernel_head_widths(lib, cuda_dev, dh):
    """Head widths off the main grid: one k-block padded from 8, 88 (a real model's), and the widths where the fp32 pairs no
    longer fit shared memory at once (dh > 128: two k-blocks at a time)."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    for dt in (torch.bfloat16, torch.float32):
        for strided in (True, False):
            q, k = _qk(3, 2, 300, dh, dt, strided, 1.0, seed=dh)
            _check(pkg, q.to(cuda_dev), k.to(cuda_dev), 1e-5)


@pytest.mark.gpu
def test_kernel_odd_strides_and_scale(lib, cuda_dev):
    """Unaligned views are copied once by the Python entry; an explicit scale is honoured."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    g = torch.Generator().manual_seed(5)
    base = torch.randn(2, 3, 100, 68, generator=g).bfloat16()
    q, k = base[..., :64], base[..., 4:]                              # row stride 68: not a multiple of 8
    out = pkg.query_mean_attention(q.to(cuda_dev), k.to(cuda_dev), scale=0.05)
    ref = torch.softmax((q.double() @ k.double().transpose(-2, -1)) * 0.05, -1).mean(2, keepdim=True)
    assert rel(out.cpu(), ref) <= 1e-5


# ------------------------------------------------------------------------------------------------ GPU: the loss on query-mean rows
def _nocls_case(w, seed, dh=64):
    """Inputs of a multi-head teacher without CLS: full maps softmax(q k^T * scale) from seeded q, k (bf16) and the q, k."""
    inp = synth.make_inputs(w, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    qk = {j: (torch.randn(w.B, w.H, w.Nt, dh, generator=g).bfloat16(), torch.randn(w.B, w.H, w.Nt, dh, generator=g).bfloat16())
          for j in range(w.Lt)}
    inp["attn"] = {j: torch.softmax((q.float() @ k.float().transpose(-2, -1)) * dh ** -0.5, -1) for j, (q, k) in qk.items()}
    return inp, qk


def _module(w, dev):
    import vit_bias_aware_structural_distillation_b200 as pkg
    torch.manual_seed(0)
    return pkg.BASDLoss(nn.CrossEntropyLoss(label_smoothing=0.001), w.Ds, w.Dt, w.student_depth, w.Ns,
                        config=synth.module_config(w), teacher_has_cls_token=False).to(dev)


def _run(m, inp, attn, dev):
    S = {l: v.to(dev).detach().requires_grad_() for l, v in inp["student"].items()}
    T = {j: v.to(dev) for j, v in inp["teacher"].items()}
    logits = inp["logits"].to(dev).requires_grad_()
    m.zero_grad(set_to_none=True)
    loss = m(logits, inp["targets"].to(dev), S, T, attn)
    loss.backward()
    torch.cuda.synchronize()
    return dict(loss=loss.detach().cpu(), ranks=m.layer_selector.subspace_ranks, grad_student={l: S[l].grad.float().cpu() for l in S},
                grad_log_temperatures=m.layer_selector.log_temperatures.grad.cpu())


NOCLS_CASES = {
    "vit_b_h12": synth.Workload("nocls_h12", 8, 196, 196, 192, 768, 12, 12, False),
    "token_space_ds384": synth.Workload("nocls_ds384", 8, 196, 196, 384, 768, 3, 12, False),
    "finer_teacher_256_to_196": synth.Workload("nocls_finer", 8, 196, 256, 192, 768, 3, 12, False),
    "single_point_single_layer": synth.Workload("nocls_p1", 8, 196, 196, 192, 768, 1, 12, False, P=1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NOCLS_CASES))
def test_loss_on_query_mean_rows(lib, cuda_dev, name):
    """BASDLoss on query_mean_attention rows against the oracle on the full maps (north-star tolerances) and against the same
    module on the full maps (1e-5: only the order of the importance sums differs)."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    w = NOCLS_CASES[name]
    inp, qk = _nocls_case(w, seed=21)
    m = _module(w, cuda_dev)
    rows = {j: pkg.query_mean_attention(q.to(cuda_dev), k.to(cuda_dev)) for j, (q, k) in qk.items()}
    out = _run(m, inp, rows, cuda_dev)
    full = _run(m, inp, {j: a.to(cuda_dev) for j, a in inp["attn"].items()}, cuda_dev)
    sel = m.layer_selector
    ref = O.run_case(inp, sel.proj_s.cpu(), sel.proj_t.cpu(), sel.log_temperatures.detach().cpu(), m.token_layers, has_cls=False,
                     n_student_tokens=w.Ns, label_smoothing=0.001)
    assert out["ranks"] == ref["ranks"], f"MP ranks {out['ranks']} != {ref['ranks']}"
    assert abs(out["loss"].item() - ref["loss"].item()) <= TOL_LOSS * abs(ref["loss"].item())
    gt, rt = out["grad_log_temperatures"], ref["grad_log_temperatures"].float()
    floor = 1e-6 if w.Lt == 1 else 1e-7              # one teacher layer: the mixing weight is 1 and its gradient ~0
    assert ((gt - rt).abs() <= TOL_TGRAD * rt.abs() + floor).all(), f"temperature grads {gt.tolist()} vs {rt.tolist()}"
    for l in ref["grad_student"]:
        assert rel(out["grad_student"][l], ref["grad_student"][l]) < TOL_SGRAD, f"student grad layer {l}"
    # Rows and maps carry the same importance up to fp32 rounding (different summation orders, ~1e-7 relative).  The loss
    # agrees to 1e-5.  The temperature gradients are differences of nearly equal per-layer terms and amplify that rounding:
    # measured up to 2.2e-5 of the largest entry on the three-layer shapes, 1e-7 absolute with one layer.
    assert abs(out["loss"].item() - full["loss"].item()) <= 1e-5 * abs(full["loss"].item())
    gf = full["grad_log_temperatures"]
    assert ((out["grad_log_temperatures"] - gf).abs() <= 1e-4 * gf.abs().max() + floor).all(), \
        f"temperature grads {out['grad_log_temperatures'].tolist()} vs {gf.tolist()}"
    assert out["ranks"] == full["ranks"]


@pytest.mark.gpu
def test_standalone_pair_loss_on_query_mean_rows(lib, cuda_dev):
    """geometric_relational_loss on query-mean rows: through its resampling branch against the committed pair_nocls golden of
    the unmodified reference, and on the student's own grid (has_cls = BASD_ATTN_QUERY_MEAN) against the same call on full maps."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    from vit_bias_aware_structural_distillation_b200 import loss as L
    g = torch.load(os.path.join(GOLD, "standalone.pt"), weights_only=False)
    w, inp, t_al, attn_same, attn_nocls = synth.standalone_inputs()
    layer0 = w.token_layers()[0]
    rows = attn_nocls.mean(2, keepdim=True)
    for act in (torch.bfloat16, torch.float32):
        s = inp["student"][layer0].to(cuda_dev).to(act).requires_grad_()
        loss = pkg.geometric_relational_loss(s, t_al.to(cuda_dev).to(act), rows.to(cuda_dev), has_cls_token=False)
        loss.backward()
        assert abs(loss.item() - g["pair_nocls"]["loss"].item()) <= TOL_LOSS * abs(g["pair_nocls"]["loss"].item())
        assert rel(s.grad.float().cpu(), g["pair_nocls"]["grad_student"]) < TOL_SGRAD
    gen = torch.Generator().manual_seed(9)
    full = torch.softmax(2 * torch.randn(w.B, 4, w.Ns, w.Ns, generator=gen), -1).to(cuda_dev)      # already on the student's grid
    rows = full.mean(2, keepdim=True)
    s0 = inp["student"][layer0].to(cuda_dev)
    tt = t_al.to(cuda_dev)
    shape, _, _ = L._prepare([s0], [tt], [rows], torch.empty(0), torch.empty(0), torch.zeros(1), False, 1, 0, L.MODE_PAIR)
    assert shape.has_cls == L.ATTN_QUERY_MEAN
    res = []
    for a in (full, rows):
        s = s0.clone().requires_grad_()
        loss = pkg.geometric_relational_loss(s, tt, a, has_cls_token=False)
        loss.backward()
        res.append((loss.detach().cpu(), s.grad.float().cpu()))
    assert abs(res[1][0].item() - res[0][0].item()) <= 1e-5 * abs(res[0][0].item())
    # (the student gradient of this 3-sample, 48-token pair comes out of ten split-bf16 Newton-Schulz steps that amplify the
    #  fp32 rounding in which the two importance sums differ: measured 1.1e-3; the golden comparison above holds it to 1e-2)
    assert rel(res[1][1], res[0][1]) <= 5e-3


@pytest.mark.gpu
def test_host_stager_with_query_mean_rows(lib, cuda_dev):
    """Pinned host rows [B,H,1,N] through HostStager give the device path's loss and gradients, and only the rows' bytes move
    for the attention."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    w = synth.Workload("nocls_stager", 4, 196, 196, 192, 768, 12, 12, False)
    m = _module(w, cuda_dev)
    stager = pkg.HostStager(m)
    for seed in (3, 4):
        inp, qk = _nocls_case(w, seed=seed)
        rows = {j: pkg.query_mean_attention(q.to(cuda_dev), k.to(cuda_dev)) for j, (q, k) in qk.items()}
        ref = _run(m, inp, rows, cuda_dev)
        pin = lambda t: t.pin_memory()
        h = stager.submit(pin(inp["logits"]), pin(inp["targets"]), {l: pin(v) for l, v in inp["student"].items()},
                          {j: pin(v) for j, v in inp["teacher"].items()}, {j: pin(r.cpu()) for j, r in rows.items()})
        m.zero_grad(set_to_none=True)
        loss = stager.run(h)
        loss.backward()
        torch.cuda.synchronize()
        assert abs(loss.item() - ref["loss"].item()) <= 1e-5 * abs(ref["loss"].item())
        assert rel(m.layer_selector.log_temperatures.grad.cpu(), ref["grad_log_temperatures"]) < TOL_TGRAD
        for l in ref["grad_student"]:
            assert torch.equal(h["leaf_student"][l].grad.float().cpu(), ref["grad_student"][l])
        nbytes = lambda ts: sum(t.numel() * t.element_size() for t in ts)
        expected = (nbytes([inp["logits"], inp["targets"]]) + nbytes(inp["student"].values()) + nbytes(inp["teacher"].values())
                    + w.Lt * w.B * w.H * 1 * w.Nt * 4)
        assert stager.h2d_bytes_last == expected
