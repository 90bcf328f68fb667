"""fp32 student and teacher tokens carried as split-bf16 pairs through the BASD loss (token_precision="fp32",
basd_shape.act_dtype = BASD_DTYPE_F32_SPLIT).

By default fp32 tokens are rounded to bf16 on entry.  On fp32 values that bf16 cannot represent, that rounding alone moves the
student gradients of the fp64 oracle by 3.7e-2 at cfg1 shapes with a 3 * 0.97^i student spectrum - beyond the project's 1e-2
tolerance whatever the kernels do.  In the opt-in mode every product reads the tokens as hi*hi + hi*lo + lo*hi and every
streaming kernel as hi + lo; the GPU tests below check that this mode meets the tolerances on such inputs against the fp64 oracle
on the same fp32 values, that it adds no error beyond the path's own floor, and that the default mode misses them (the control).

The inputs are those of the fp64 CPU emulation that measured the gap: synth's generators without their bf16 rounding.
"""
import ctypes
import dataclasses

import pytest
import torch
import torch.nn as nn

from oracle import basd_oracle as O
from oracle import synth

TOL_LOSS, TOL_TGRAD, TOL_SGRAD = 1e-3, 1e-3, 1e-2


# --------------------------------------------------------------------------------------------- inputs
def spiked(B, N, D, r, g):
    basis = torch.linalg.qr(torch.randn(D, r, generator=g))[0]
    return (torch.randn(B, N, r, generator=g) * 4.0 * torch.linspace(1.0, 0.2, r)) @ basis.T + torch.randn(B, N, D, generator=g)


def geometric(B, N, D, g, rho):
    basis = torch.linalg.qr(torch.randn(D, D, generator=g))[0]
    return (torch.randn(B, N, D, generator=g) * 3.0 * rho ** torch.arange(D)) @ basis.T


def fp32_inputs(w, rho=0.97, seed=1234):
    """fp32 tokens that are NOT bf16-representable (student spectrum 3 rho^i, spiked teachers), softmaxed attention."""
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(w.B, w.num_classes, generator=g)
    targets = torch.randint(0, w.num_classes, (w.B,), generator=g)
    student = {l: geometric(w.B, w.Ns, w.Ds, g, rho) for l in w.token_layers()}
    teacher = {j: spiked(w.B, w.Nt, w.Dt, 16 + 4 * j, g) for j in range(w.Lt)}
    n = w.Nt + 1 if w.has_cls else w.Nt
    attn = {j: torch.softmax(2 * torch.randn(w.B, w.H, n, n, generator=g), -1) for j in range(w.Lt)}
    return dict(logits=logits, targets=targets, student=student, teacher=teacher, attn=attn)


def rounded(inp):
    """The same inputs with every token rounded to bf16 (what the default mode reads), kept as fp32."""
    return dict(inp, student={k: v.bfloat16().float() for k, v in inp["student"].items()},
                teacher={k: v.bfloat16().float() for k, v in inp["teacher"].items()})


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30)).item()


CFG1_B8 = dataclasses.replace(synth.CONFIGS["cfg1"], B=8)
TOKEN_SPACE = synth.Workload("tiny_cnn", 6, 64, 16, 48, 128, 1, 1, False)       # D_s > min(N_s, N_t) - 1: token-space polar form
# D_s > 192: unfused column sums, two-tile Grams.  (At D_s = 256 the 0.97^i spectrum ends at 4e-4 and the polar iteration's own
# floor - the default mode on the bf16-rounded copy against the oracle on that copy - is 1.2e-2 on the student gradients; the split
# mode gives 1.3e-2 there.  D_s = 224 keeps the path inside its tolerance: floor 2.9e-3, split 2.3e-3, default 5.6e-2.)
WIDE = synth.Workload("wide", 4, 300, 300, 224, 512, 3, 2, True, P=2)


# --------------------------------------------------------------------------------------------- CPU
def _shape(**kw):
    from vit_bias_aware_structural_distillation_b200._lib import Shape
    base = dict(B=8, Ns=196, Nt=196, Ds=192, Dt=384, Lt=12, P=4, H=6, has_cls=1, act_dtype=0, attn_dtype=0, world_size=1)
    base.update(kw)
    return Shape(**base)


def test_workspace_bytes_accepts_split_tokens_and_rejects_unknown_dtypes(lib):
    from vit_bias_aware_structural_distillation_b200 import _lib
    sizes = {}
    for code in (_lib.DTYPE_F32, _lib.DTYPE_BF16, _lib.DTYPE_F32_SPLIT):
        n = ctypes.c_size_t()
        assert lib.basd_workspace_bytes(ctypes.byref(_shape(act_dtype=code)), ctypes.byref(n)) == 0, lib.basd_last_error().decode()
        sizes[code] = n.value
    # the split mode adds exactly one more packed copy of every token tensor (the lo halves)
    assert sizes[_lib.DTYPE_F32_SPLIT] >= sizes[_lib.DTYPE_F32] > sizes[_lib.DTYPE_BF16]
    assert sizes[_lib.DTYPE_F32_SPLIT] - sizes[_lib.DTYPE_F32] >= 2 * 8 * 196 * (12 * 384 + 4 * 192)
    for kw, needle in ((dict(act_dtype=3), "act_dtype"), (dict(act_dtype=-1), "act_dtype"), (dict(attn_dtype=2), "attn_dtype")):
        n = ctypes.c_size_t()
        assert lib.basd_workspace_bytes(ctypes.byref(_shape(**kw)), ctypes.byref(n)) != 0
        assert needle in lib.basd_last_error().decode()


def test_bad_token_precision_raises_before_device_work(lib):
    import vit_bias_aware_structural_distillation_b200 as pkg
    from vit_bias_aware_structural_distillation_b200 import loss as L
    w = synth.Workload("t", 2, 36, 36, 32, 32, 2, 1, True, P=2)
    inp = fp32_inputs(w)
    m = pkg.BASDLoss(nn.CrossEntropyLoss(), w.Ds, w.Dt, w.student_depth, w.Ns, config=synth.module_config(w), teacher_has_cls_token=True)
    assert m.token_precision == "bf16" and m.layer_selector.token_precision == "bf16"
    for bad in ("fp16", "FP32", None, 32):
        m.token_precision = bad
        with pytest.raises(pkg.BasdError, match="token_precision"):
            m(inp["logits"], inp["targets"], inp["student"], inp["teacher"], inp["attn"])
        with pytest.raises(pkg.BasdError, match="token_precision"):
            pkg.geometric_relational_loss(inp["student"][w.token_layers()[0]], inp["teacher"][0], inp["attn"][0], has_cls_token=True,
                                          token_precision=bad)
        with pytest.raises(pkg.BasdError, match="token_precision"):
            L._prepare(list(inp["student"].values()), list(inp["teacher"].values()), list(inp["attn"].values()), m.layer_selector.proj_s,
                       m.layer_selector.proj_t, m.layer_selector.log_temperatures, True, 1, 0, L.MODE_LOSS, bad)
        m.layer_selector.token_precision = bad
        with pytest.raises(pkg.BasdError, match="token_precision"):
            m.layer_selector.mixing_weights(list(inp["student"].values()), list(inp["teacher"].values()))


# --------------------------------------------------------------------------------------------- GPU
def build_module(w, dev, token_precision, polar_steps=0):
    """A fresh module (the same parameters every time).  Every comparison below runs each arm on a fresh module at a fixed
    Newton-Schulz step count: a module raises its step count after a forward whose polar residual stayed above
    BASDLoss.POLAR_RESIDUAL_OK, so a reused module can run its next arm with a different schedule."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    torch.manual_seed(0)
    m = pkg.BASDLoss(nn.CrossEntropyLoss(label_smoothing=0.001), w.Ds, w.Dt, w.student_depth, w.Ns,
                     config=synth.module_config(w), teacher_has_cls_token=w.has_cls).to(dev)
    m.token_precision = token_precision
    m.polar_steps = polar_steps
    return m


def settled_polar_steps(w, inp, dev):
    """The Newton-Schulz step count a module settles on for these inputs in the split mode: forwards are repeated until one
    leaves the count unchanged (each forward reads the previous one's residual and raises the count by one if it is too large)."""
    import warnings
    m = build_module(w, dev, "fp32")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        run_module(m, inp, dev)
        for _ in range(8):
            before = m.polar_steps
            run_module(m, inp, dev)
            if m.polar_steps == before:
                break
    return m.polar_steps


def run_module(m, inp, dev, student_view=None, teacher_view=None):
    """One forward + backward; *_view(t) may hand a tensor over as a strided view of other storage."""
    S = {l: v.to(dev) for l, v in inp["student"].items()}
    if student_view:
        S = {l: student_view(v) for l, v in S.items()}
    S = {l: v.detach().requires_grad_() for l, v in S.items()}
    T = {j: v.to(dev) for j, v in inp["teacher"].items()}
    if teacher_view:
        T = {j: teacher_view(v) for j, v in T.items()}
    A = {j: v.to(dev) for j, v in inp["attn"].items()}
    logits = inp["logits"].to(dev).requires_grad_()
    m.zero_grad(set_to_none=True)
    loss = m(logits, inp["targets"].to(dev), S, T, A)
    loss.backward()
    torch.cuda.synchronize()
    return dict(loss=loss.detach().cpu(), ranks=m.layer_selector.subspace_ranks, grad_student={l: S[l].grad.cpu() for l in S},
                grad_log_temperatures=m.layer_selector.log_temperatures.grad.cpu())


def oracle64(m, inp, w):
    sel = m.layer_selector
    return O.run_case(inp, sel.proj_s.cpu(), sel.proj_t.cpu(), sel.log_temperatures.detach().cpu(), m.token_layers, has_cls=w.has_cls,
                      n_student_tokens=w.Ns, label_smoothing=0.001, dtype=torch.float64)


def errors(out, ref):
    gt, rt = out["grad_log_temperatures"].double(), ref["grad_log_temperatures"].double()
    return dict(loss=abs(out["loss"].item() - ref["loss"].item()) / abs(ref["loss"].item()),
                tgrad=((gt - rt).abs().max() / rt.abs().max().clamp(min=1e-30)).item() if rt.abs().max() > 1e-12 else gt.abs().max().item(),
                sgrad=max(rel(out["grad_student"][l], ref["grad_student"][l]) for l in ref["grad_student"]))


def bitwise_equal(a, b):
    return (a["ranks"] == b["ranks"] and torch.equal(a["loss"], b["loss"]) and torch.equal(a["grad_log_temperatures"], b["grad_log_temperatures"])
            and all(torch.equal(a["grad_student"][l], b["grad_student"][l]) for l in a["grad_student"]))


@pytest.mark.gpu
@pytest.mark.parametrize("w", [CFG1_B8, TOKEN_SPACE, WIDE], ids=lambda w: w.name)
def test_split_tokens_against_fp64_oracle(lib, cuda_dev, w):
    """fp32 tokens that bf16 cannot represent: the split mode meets the tolerances against the fp64 oracle on the same values and
    adds no error beyond the path's own floor (the default mode on the bf16-rounded copy against the oracle on that copy); the
    default mode on the fp32 values misses the student-gradient tolerance (it reads them rounded)."""
    inp = fp32_inputs(w)
    # every arm at the step count the module settles on (cfg1's cross-covariance needs 11 steps: residual 0.87 after 10)
    steps = settled_polar_steps(w, inp, cuda_dev)
    m = build_module(w, cuda_dev, "fp32", steps)
    ref = oracle64(m, inp, w)
    split = run_module(m, inp, cuda_dev)
    e = errors(split, ref)
    print(f"\n{w.name} ({steps or 'default'} polar steps): fp32 mode vs fp64 oracle: {e}")
    assert split["ranks"] == ref["ranks"]
    assert e["loss"] <= TOL_LOSS and e["tgrad"] <= TOL_TGRAD and e["sgrad"] <= TOL_SGRAD, e
    inp_r = rounded(inp)
    m = build_module(w, cuda_dev, "bf16", steps)
    floor = errors(run_module(m, inp_r, cuda_dev), oracle64(m, inp_r, w))
    print(f"{w.name}: default mode on the bf16-rounded copy vs its fp64 oracle (the floor): {floor}")
    assert e["sgrad"] <= 1.5 * floor["sgrad"] + 1e-4, (e, floor)
    m = build_module(w, cuda_dev, "bf16", steps)
    control = errors(run_module(m, inp, cuda_dev), ref)
    print(f"{w.name}: default mode on the fp32 values vs fp64 oracle (control): {control}")
    if w is not TOKEN_SPACE:                # (its 48-wide spectrum ends at 0.23: the fp64 emulation puts its rounding gap at 1.9e-3)
        assert control["sgrad"] > TOL_SGRAD, control


@pytest.mark.gpu
def test_standalone_entry_points_with_split_tokens(lib, cuda_dev):
    """geometric_relational_loss and GrassmannianLayerSelector.mixing_weights on fp32 tokens in the split mode against the fp64
    oracle's pair loss and mixing weights (and their gradients) on the same values."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    w = CFG1_B8
    inp = fp32_inputs(w)
    l0 = w.token_layers()[0]
    s64 = inp["student"][l0].double().requires_grad_()
    ref_loss = O.geometric_relational_loss(s64, inp["teacher"][0].double(), inp["attn"][0].double(), has_cls=True, dtype=torch.float64)
    ref_loss.backward()
    s = inp["student"][l0].to(cuda_dev).requires_grad_()
    loss = pkg.geometric_relational_loss(s, inp["teacher"][0].to(cuda_dev), inp["attn"][0].to(cuda_dev), has_cls_token=True, token_precision="fp32")
    loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= TOL_LOSS * abs(ref_loss.item())
    e_pair = rel(s.grad.cpu(), s64.grad)
    s_d = inp["student"][l0].to(cuda_dev).requires_grad_()
    pkg.geometric_relational_loss(s_d, inp["teacher"][0].to(cuda_dev), inp["attn"][0].to(cuda_dev), has_cls_token=True).backward()
    e_pair_default = rel(s_d.grad.cpu(), s64.grad)
    print(f"\npair: student grad vs fp64 oracle: fp32 mode {e_pair:.2e}, default {e_pair_default:.2e}")
    assert e_pair <= TOL_SGRAD and e_pair < e_pair_default

    torch.manual_seed(0)
    sel = pkg.GrassmannianLayerSelector(num_extraction_points=w.P, student_dim=w.Ds, teacher_dim=w.Dt).to(cuda_dev)
    sel.token_precision = "fp32"
    layers = w.token_layers()
    S = {l: inp["student"][l].to(cuda_dev).requires_grad_() for l in layers}
    T = {j: inp["teacher"][j].to(cuda_dev) for j in range(w.Lt)}
    A = {j: inp["attn"][j].to(cuda_dev) for j in range(w.Lt)}
    probes = {l: torch.randn(w.B, w.Ns, w.Dt, generator=torch.Generator().manual_seed(6 + i)) for i, l in enumerate(layers)}
    mt, _ = sel(S, T, A, layers)                 # mixing_weights (BASD_MODE_SELECTOR) + the reference's weighted sums
    sum((mt[l] * probes[l].to(cuda_dev)).sum() for l in layers).backward()
    S64 = {l: inp["student"][l].double().requires_grad_() for l in layers}
    logt = sel.log_temperatures.detach().cpu().double().requires_grad_()
    mt64, _, ranks = O.selector_forward(S64, {j: inp["teacher"][j].double() for j in range(w.Lt)}, {j: inp["attn"][j][:, :, :1] for j in range(w.Lt)},
                                        sel.proj_s.cpu(), sel.proj_t.cpu(), logt, layers, dtype=torch.float64)
    sum((mt64[l] * probes[l].double()).sum() for l in layers).backward()
    assert sel.subspace_ranks == ranks
    e_sel = max(rel(S[l].grad.cpu(), S64[l].grad) for l in layers)
    gt, rt = sel.log_temperatures.grad.cpu().double(), logt.grad
    print(f"selector: mixed tokens {max(rel(mt[l].detach().cpu(), mt64[l].detach()) for l in layers):.2e}, student grad {e_sel:.2e}, "
          f"temperature grad {((gt - rt).abs().max() / rt.abs().max()).item():.2e}")
    for l in layers:
        assert rel(mt[l].detach().cpu(), mt64[l].detach()) < 1e-4
    assert e_sel <= TOL_SGRAD
    assert (gt - rt).abs().max() <= TOL_TGRAD * rt.abs().max()


@pytest.mark.gpu
@pytest.mark.parametrize("w", [CFG1_B8, TOKEN_SPACE, WIDE], ids=lambda w: w.name)
def test_bf16_representable_fp32_tokens_give_the_default_bits(lib, cuda_dev, w):
    """fp32 tokens that hold bf16 values have lo = 0 everywhere: the split mode's extra terms add exact zeros, so loss, ranks and
    every gradient are bitwise those of the default mode."""
    inp = rounded(fp32_inputs(w))
    a = run_module(build_module(w, cuda_dev, "bf16"), inp, cuda_dev)
    b = run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev)
    assert bitwise_equal(a, b)


@pytest.mark.gpu
def test_split_tokens_views_repeatability_and_workspace(lib, cuda_dev):
    """In the split mode: CLS-stripped fp32 views of students and teachers give the bits of contiguous inputs, two executions are
    bitwise equal, and zero-, NaN- or random-filled workspace gives identical bits."""
    from vit_bias_aware_structural_distillation_b200 import loss as L
    w = CFG1_B8
    inp = fp32_inputs(w)
    ref = run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev)

    def cls_view(v):
        full = torch.zeros(v.shape[0], v.shape[1] + 1, v.shape[2], device=v.device, dtype=v.dtype)
        full[:, 1:] = v
        return full[:, 1:, :]
    assert bitwise_equal(ref, run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev, student_view=cls_view, teacher_view=cls_view))
    assert bitwise_equal(ref, run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev))
    fills = {"zero": lambda ws: ws.zero_(), "nan": lambda ws: ws.fill_(0xFF),
             "rand": lambda ws: ws.copy_(torch.randint(0, 256, ws.shape, dtype=torch.uint8, device=ws.device))}
    try:
        for name, f in fills.items():
            L._debug_workspace_fill = f
            assert bitwise_equal(ref, run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev)), name
    finally:
        L._debug_workspace_fill = None


@pytest.mark.gpu
def test_split_tokens_cnn_transposed_teacher_view(lib, cuda_dev):
    """A CNN teacher hands its feature map [B, C, H, W] over as the transposed view [B, HW, C] (teacher.py:155): read in place by the
    pack kernel's strides, it gives the bits of the contiguous tensor in the split mode."""
    w = TOKEN_SPACE
    inp = fp32_inputs(w)
    ref = run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev)

    def cnn_view(v):                            # [B, HW, C] -> storage [B, C, HW] -> transposed view
        return v.transpose(1, 2).contiguous().transpose(1, 2)
    out = run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev, teacher_view=cnn_view)
    assert bitwise_equal(ref, out)


@pytest.mark.gpu
def test_host_stager_with_pinned_fp32_tokens(lib, cuda_dev):
    """HostStager follows its module's token_precision: pinned fp32 host tokens give the bits of a direct call in the split mode."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    inp = fp32_inputs(w)
    ref = run_module(build_module(w, cuda_dev, "fp32"), inp, cuda_dev)
    m = build_module(w, cuda_dev, "fp32")
    stager = pkg.HostStager(m)
    pin = lambda t: t.pin_memory()
    h = stager.submit(pin(inp["logits"]), pin(inp["targets"]), {l: pin(v) for l, v in inp["student"].items()},
                      {j: pin(v) for j, v in inp["teacher"].items()}, {j: pin(v) for j, v in inp["attn"].items()})
    m.zero_grad(set_to_none=True)
    loss = stager.run(h)
    loss.backward()
    torch.cuda.synchronize()
    out = dict(loss=loss.detach().cpu(), ranks=m.layer_selector.subspace_ranks, grad_log_temperatures=m.layer_selector.log_temperatures.grad.cpu(),
               grad_student={l: h["leaf_student"][l].grad.cpu() for l in inp["student"]})
    assert bitwise_equal(ref, out)
