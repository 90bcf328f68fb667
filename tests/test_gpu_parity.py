"""GPU parity tests (run with `-m gpu` on a B200): the CUDA path, called through the C ABI of include/basd_b200.h
(ctypes binding in vit_bias_aware_structural_distillation_b200/_lib.py), against
  * the CPU oracle (oracle/basd_oracle.py) on the same seeded inputs,
  * the committed golden outputs of the UNMODIFIED reference (tests/golden/*.pt, made by oracle/make_golden.py),
  * size-independent properties at BASELINE.json's full sizes.

Tolerances are BASELINE.json north_star's: 1e-3 relative on the loss and on the log_temperatures gradients,
1e-2 relative (Frobenius) on the student-feature gradients; Marchenko-Pastur ranks are integers and must be EXACT.
SVD sign/rotation ambiguity: only invariants are compared (cosines of principal angles, d2, mixing weights, nuclear
norm, loss, gradients) — never raw singular vectors.
"""
import ctypes
import dataclasses
import math
import os

import pytest
import torch
import torch.nn as nn

from oracle import basd_oracle as O
from oracle import kernel_model as K
from oracle import synth

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL_LOSS, TOL_TGRAD, TOL_SGRAD = 1e-3, 1e-3, 1e-2


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30)).item()


def load_golden(name):
    g = torch.load(os.path.join(GOLD, f"{name}.pt"), weights_only=False)
    return g, synth.Workload(**g["workload"])


def build_module(w, dev):
    import vit_bias_aware_structural_distillation_b200 as pkg
    torch.manual_seed(0)
    return pkg.BASDLoss(nn.CrossEntropyLoss(label_smoothing=0.001), w.Ds, w.Dt, w.student_depth, w.Ns,
                        config=synth.module_config(w), teacher_has_cls_token=w.has_cls).to(dev)


def run_module(m, inp, dev, act_dtype=torch.bfloat16, attn_dtype=torch.float32, views=False):
    """One forward + backward through the drop-in module.  views=True hands over CLS-stripped, non-contiguous views
    like trainer.py:29 / teacher.py:157 do."""
    def tok(v):
        v = v.to(dev).to(act_dtype)
        if views:
            full = torch.zeros(v.shape[0], v.shape[1] + 1, v.shape[2], device=dev, dtype=act_dtype)
            full[:, 1:] = v
            v = full[:, 1:, :]
        return v
    S = {l: tok(v).detach().requires_grad_() for l, v in inp["student"].items()}
    T = {j: tok(v) for j, v in inp["teacher"].items()}
    A = {j: v.to(dev).to(attn_dtype) for j, v in inp["attn"].items()}
    logits = inp["logits"].to(dev).requires_grad_()
    m.zero_grad(set_to_none=True)
    loss = m(logits, inp["targets"].to(dev), S, T, A)
    loss.backward()
    torch.cuda.synchronize()
    return dict(loss=loss.detach().cpu(), geo=m.last_geo_loss.cpu(), ranks=m.layer_selector.subspace_ranks,
                w=m.layer_selector.last_mixing_weights.cpu(), grad_student={l: S[l].grad.float().cpu() for l in S},
                grad_log_temperatures=m.layer_selector.log_temperatures.grad.cpu(), grad_logits=logits.grad.cpu())


def oracle_case(m, inp, w, dtype=torch.float32):
    sel = m.layer_selector
    return O.run_case(inp, sel.proj_s.cpu(), sel.proj_t.cpu(), sel.log_temperatures.detach().cpu(), m.token_layers,
                      has_cls=w.has_cls, n_student_tokens=w.Ns, label_smoothing=0.001, dtype=dtype)


def assert_parity(out, ref, w, tgrad_floor=1e-7, tgrad_tol=TOL_TGRAD, sgrad_tol=TOL_SGRAD):
    assert out["ranks"] == ref["ranks"], f"MP ranks {out['ranks']} != {ref['ranks']}"        # integer work: exact
    assert abs(out["loss"].item() - ref["loss"].item()) <= TOL_LOSS * abs(ref["loss"].item())
    assert (out["w"] - ref["w"].float()).abs().max() < 1e-4
    gt, rt = out["grad_log_temperatures"], ref["grad_log_temperatures"].float()
    assert ((gt - rt).abs() <= tgrad_tol * rt.abs() + tgrad_floor).all(), f"temperature grads {gt.tolist()} vs {rt.tolist()}"
    for l in ref["grad_student"]:
        assert rel(out["grad_student"][l], ref["grad_student"][l]) < sgrad_tol, f"student grad layer {l}"
    assert rel(out["grad_logits"], ref["grad_logits"]) < 1e-3


# ------------------------------------------------------------------------------------------------ building blocks
def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("variant,M,N,Kd", [(0, 128, 192, 64), (0, 300, 200, 384), (0, 1000, 384, 768),
                                            (1, 192, 192, 1000), (1, 384, 384, 640), (1, 48, 48, 256),
                                            (2, 196, 128, 200), (2, 196, 768, 200), (2, 64, 96, 64),
                                            (3, 196, 196, 768), (3, 64, 64, 96), (3, 200, 200, 128),
                                            (3, 9, 9, 64)])
def test_tcgen05_gemm_variants(lib, cuda_dev, variant, M, N, Kd):
    """Every operand-major combination the path uses (K-major x K-major, MN x MN split-K, K x MN, split-bf16 Gram)
    against an fp32 torch matmul of the same bf16 values: fp32-accumulate accuracy."""
    gen = torch.Generator().manual_seed(variant * 1000 + M + N + Kd)
    if variant == 0:
        A = torch.randn(M, Kd, generator=gen).bfloat16(); B = torch.randn(N, Kd, generator=gen).bfloat16()
        ref = A.float() @ B.float().T
    elif variant == 1:
        A = torch.randn(Kd, M, generator=gen).bfloat16(); B = torch.randn(Kd, N, generator=gen).bfloat16()
        ref = A.float().T @ B.float()
    elif variant == 2:
        A = torch.randn(M, Kd, generator=gen).bfloat16(); B = torch.randn(Kd, N, generator=gen).bfloat16()
        ref = A.float() @ B.float()
    else:
        X = torch.randn(M, Kd, generator=gen); A = X.bfloat16(); B = (X - A.float()).bfloat16(); N = M
        ref = A.float() @ A.float().T + A.float() @ B.float().T + B.float() @ A.float().T
    Ad, Bd = A.to(cuda_dev), B.to(cuda_dev)
    C = torch.zeros(M, N, device=cuda_dev)
    rc = lib.basd_selftest_gemm(variant, Ad.data_ptr(), Bd.data_ptr(), C.data_ptr(), M, N, Kd, _stream())
    assert rc == 0, lib.basd_last_error().decode()
    torch.cuda.synchronize()
    assert (C.cpu() - ref).abs().max().item() <= 1e-4 * ref.abs().max().item()


@pytest.mark.parametrize("n", [16, 33, 48, 51, 77, 100, 130, 191, 192, 224, 228, 256, 330, 384])
def test_jacobi_eigensolver(lib, cuda_dev, n):
    """One-sided Jacobi vs LAPACK (fp64): eigenvalues, residual, orthogonality.  n <= 224: cluster kernel with the matrix
    in shared memory; larger: the global-memory variant (ViT-S students, D_s = 384)."""
    torch.manual_seed(n)
    X = torch.randn(4 * n, n) * (0.97 ** torch.arange(n))
    G = X.T @ X
    Gd = G.to(cuda_dev)
    ev = torch.zeros(n, device=cuda_dev); evec = torch.zeros(n, n, device=cuda_dev)
    sw = torch.zeros(4, dtype=torch.int32, device=cuda_dev)
    ws = torch.zeros(4 * (3 * n * n + 8 * n) + 16384, dtype=torch.uint8, device=cuda_dev)
    rc = lib.basd_selftest_eig(Gd.data_ptr(), n, ev.data_ptr(), evec.data_ptr(), sw.data_ptr(), ws.data_ptr(), _stream())
    assert rc == 0, lib.basd_last_error().decode()
    torch.cuda.synchronize()
    ref = torch.linalg.eigvalsh(G.double()).flip(0)
    V = evec.cpu().double()
    assert ((ev.cpu().double() - ref).abs().max() / ref.max()).item() < 3e-5
    assert ((G.double() @ V.T - V.T * ev.cpu().double()).norm() / G.double().norm()).item() < 3e-5
    assert (V @ V.T - torch.eye(n, dtype=torch.float64)).abs().max().item() < 2e-5
    assert 0 < sw[0].item() < 40


@pytest.mark.parametrize("M,D,r", [(4096, 48, 5), (20000, 192, 24), (6000, 96, 11), (120, 192, 6), (40, 64, 3),   # last two: M < D branch (:14-15)
                                   (8000, 384, 30), (6000, 768, 40), (300, 384, 8), (5000, 1024, 50)])   # unprojected D_t-wide features (teacher.py:177)
def test_marchenko_pastur_rank_free_function(lib, cuda_dev, M, D, r):
    """layer_selector.py:8-20 (second consumer teacher.py:177): exact integer agreement with the oracle."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    g = torch.Generator().manual_seed(M + D)
    f = synth.spiked(1, M, D, r, g)[0]
    assert pkg.marchenko_pastur_rank(f.to(cuda_dev)) == O.mp_rank(f.float())
    assert pkg.marchenko_pastur_rank(f.float().to(cuda_dev)) == O.mp_rank(f.float())


# ------------------------------------------------------------------------------------------------ stage checks
def test_phase_buffers_match_kernel_model(lib, cuda_dev):
    """Phase 1/2 intermediates through the raw C ABI (no module, no autograd): importance rows, pooled Gram + column
    sums, ranks, Grassmann distances, cosines, mixing weights, per-sample nuclear norm and traces."""
    from vit_bias_aware_structural_distillation_b200 import _lib, loss as L
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    inp = synth.make_inputs(w)
    m = build_module(w, cuda_dev)
    sel = m.layer_selector
    students = [inp["student"][l].to(cuda_dev) for l in m.token_layers]
    teachers = [inp["teacher"][j].to(cuda_dev) for j in sorted(inp["teacher"])]
    attns = [inp["attn"][j].to(cuda_dev) for j in sorted(inp["attn"])]
    shape, cin, keep = L._prepare(students, teachers, attns, sel.proj_s, sel.proj_t, sel.log_temperatures, w.has_cls, 1)
    nb = ctypes.c_size_t()
    _lib.check(lib.basd_workspace_bytes(ctypes.byref(shape), ctypes.byref(nb)), "workspace_bytes")
    ws = torch.zeros(nb.value, dtype=torch.uint8, device=cuda_dev)
    geo = torch.zeros((), device=cuda_dev)
    _lib.check(lib.basd_forward_stats(ctypes.byref(shape), ctypes.byref(cin), ws.data_ptr(), _stream()), "forward_stats")
    _lib.check(lib.basd_forward_solve(ctypes.byref(shape), ctypes.byref(cin), ws.data_ptr(), geo.data_ptr(), _stream()), "forward_solve")
    torch.cuda.synchronize()
    V = lambda n, dt=torch.float32: L.workspace_view(shape, ws, n, dt).cpu()
    ref = oracle_case(m, inp, w)

    rows_ref = torch.stack([O.importance_rows(inp["attn"][j].float(), w.has_cls) for j in sorted(inp["attn"])])
    assert (V("rows").view_as(rows_ref) - rows_ref).abs().max() < 1e-7
    n = w.Ds
    stats = V("stats").view(w.Lt + w.P, n * n + n)
    X = inp["teacher"][0].float().reshape(-1, w.Dt)
    Z = X.double() @ sel.proj_t.cpu().double().T               # projected teacher tokens are kept as a split pair: fp32 class
    G0 = Z.T @ Z
    assert (stats[0, :n * n].view(n, n).double() - G0).abs().max() <= 2e-5 * G0.abs().max()
    assert (stats[0, n * n:].double() - Z.sum(0)).abs().max() <= 2e-5 * Z.abs().sum(0).max()
    Gs, cs, _ = K.student_stats(inp["student"][m.token_layers[0]].float(), torch.float32)
    assert (stats[w.Lt, :n * n].view(n, n) - Gs).abs().max() <= 2e-5 * Gs.abs().max()
    assert V("ranks", torch.int32).tolist() == [ref["ranks"][j] for j in sorted(ref["ranks"])]
    assert rel(V("d2").view(w.P, w.Lt), ref["d2"]) < 2e-4
    assert (V("w").view(w.P, w.Lt) - ref["w"]).abs().max() < 1e-4
    cosv = V("cos").view(w.P, w.Lt, n)
    for i in range(w.P):
        for j in range(w.Lt):
            k = ref["ranks"][j]
            assert (cosv[i, j, :k] - ref["cos"][i][j]).abs().max() < 1e-3          # invariants of the subspace pair
    dbg = V("dbg").view(w.P, w.B, 5)
    assert rel(dbg[..., 0], ref["nuc"]) < 2e-4 and rel(dbg[..., 1], ref["tr_s"]) < 1e-5 and rel(dbg[..., 2], ref["tr_t"]) < 1e-4
    assert abs(geo.item() - ref["geo"].item()) <= 2e-4 * abs(ref["geo"].item())
    del keep


# ------------------------------------------------------------------------------------------------ whole path
@pytest.mark.parametrize("name", ["tiny_cls", "tiny_up", "tiny_down", "tiny_cnn_down", "tiny_interp", "tiny_cnn"])
def test_tiny_cases_against_oracle_and_reference_golden(lib, cuda_dev, name):
    """Edge cases of SURVEY.md §4 with the reference's full gradients in the fixtures: the plain CLS case, token-count
    resampling up (56 -> 64) and down (100 -> 64, the DINOv2 256 -> 196 situation), a single-layer CNN teacher without
    CLS (w == 1, zero temperature gradient, attention averaged over queries).  tiny_interp / tiny_cnn up-sample so few
    teacher tokens (36 / 16 -> 64) that the cross-covariance is rank deficient (rank N_t - 1 < D_s, SURVEY.md hazard 13):
    the polar iteration then runs in the teacher's token space (DESIGN.md section 3)."""
    g, w = load_golden(name)
    inp = synth.make_inputs(w, seed=g["seed"])
    m = build_module(w, cuda_dev)
    out = run_module(m, inp, cuda_dev)
    ref = oracle_case(m, inp, w)
    # Temperature gradients of these 256-row problems: the softmax derivative is a difference of nearly equal per-layer
    # terms, which amplifies the 2^-17 relative precision of the split-bf16 polar products; entries are held to 1e-3 of
    # the LARGEST entry plus 1e-3 of themselves (the BASELINE shapes, cfg1 / cfg2 below, to 1e-3 of each entry).
    tfloor = 1e-3 * ref["grad_log_temperatures"].abs().max().item() + 1e-7
    assert_parity(out, ref, w, tgrad_floor=tfloor)
    assert out["ranks"] == g["ranks"]
    assert abs(out["loss"].item() - g["loss"].item()) <= TOL_LOSS * abs(g["loss"].item())
    for l in g["token_layers"]:
        assert rel(out["grad_student"][l], g["grad_student"][l]) < TOL_SGRAD
    if name.startswith("tiny_cnn"):
        # softmax over a single layer: w == 1 and no temperature gradient (an fma leaves ~1e-7 of rounding, the reference 0)
        assert out["grad_log_temperatures"].abs().max() < 1e-6 and (out["w"] == 1).all()
    else:
        assert ((out["grad_log_temperatures"] - g["grad_log_temperatures"]).abs()
                <= TOL_TGRAD * g["grad_log_temperatures"].abs() + tfloor).all()


@pytest.mark.parametrize("act_dtype,views", [(torch.bfloat16, False), (torch.float32, False), (torch.float32, True),
                                             (torch.bfloat16, True)])
def test_cfg1_against_reference_golden(lib, cuda_dev, act_dtype, views):
    """BASELINE.json configs[0] at its full size (B=32) against the reference's own output: bf16 tokens, the fp32
    tokens the reference flow delivers, and CLS-stripped non-contiguous views (trainer.py:29, teacher.py:157)."""
    g, w = load_golden("cfg1")
    inp = synth.make_inputs(w, seed=g["seed"])
    m = build_module(w, cuda_dev)
    out = run_module(m, inp, cuda_dev, act_dtype=act_dtype, views=views)
    assert out["ranks"] == g["ranks"]
    assert abs(out["loss"].item() - g["loss"].item()) <= TOL_LOSS * abs(g["loss"].item())
    assert ((out["grad_log_temperatures"] - g["grad_log_temperatures"]).abs() <= TOL_TGRAD * g["grad_log_temperatures"].abs()).all()
    for l in g["token_layers"]:
        assert abs(out["grad_student"][l].norm() - g["grad_student_norm"][l]) <= TOL_SGRAD * g["grad_student_norm"][l]
        assert rel(out["grad_student"][l].flatten()[::997], g["grad_student_sub"][l]) < TOL_SGRAD
        pr = torch.stack([(out["grad_student"][l] * p).sum() for p in _probes(out["grad_student"][l].shape)])
        assert rel(pr, g["grad_student_probe"][l]) < TOL_SGRAD


def test_cls_stripped_bf16_views_are_consumed_in_place(lib, cuda_dev):
    """trainer.py:29 / teacher.py:157 hand over out[:, 1:, :] views of [B, N+1, D] tensors.  bf16 views reach the kernels
    without a copy (TMA descriptors / batch strides follow the view) and give the dense path's result."""
    from vit_bias_aware_structural_distillation_b200 import loss as L
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    inp = synth.make_inputs(w)
    m = build_module(w, cuda_dev)
    dense = run_module(m, inp, cuda_dev, views=False)
    viewed = run_module(m, inp, cuda_dev, views=True)
    assert viewed["ranks"] == dense["ranks"]
    assert abs(viewed["loss"].item() - dense["loss"].item()) <= 1e-6 * abs(dense["loss"].item())
    assert rel(viewed["grad_log_temperatures"], dense["grad_log_temperatures"]) < 1e-4
    for l in dense["grad_student"]:
        assert rel(viewed["grad_student"][l], dense["grad_student"][l]) < 2e-3        # (bf16 gradient storage: 2^-9 per element)
    assert_parity(viewed, oracle_case(m, inp, w), w)
    # no copy: the pointers the C ABI receives are the views' own
    def view(v):
        full = torch.zeros(v.shape[0], v.shape[1] + 1, v.shape[2], device=cuda_dev, dtype=torch.bfloat16)
        full[:, 1:] = v.to(cuda_dev)
        return full[:, 1:, :]
    sel = m.layer_selector
    students = [view(inp["student"][l]) for l in m.token_layers]
    teachers = [view(inp["teacher"][j]) for j in sorted(inp["teacher"])]
    attns = [inp["attn"][j].to(cuda_dev) for j in sorted(inp["attn"])]
    shape, cin, keep = L._prepare(students, teachers, attns, sel.proj_s, sel.proj_t, sel.log_temperatures, w.has_cls, 1)
    assert [cin.student[i] for i in range(w.P)] == [t.data_ptr() for t in students]
    assert [cin.teacher[j] for j in range(w.Lt)] == [t.data_ptr() for t in teachers]
    assert cin.student_strides[0] == (w.Ns + 1) * w.Ds and cin.teacher_strides[0] == (w.Nt + 1) * w.Dt
    del keep


def _probes(shape, n=4, seed=99):
    gen = torch.Generator().manual_seed(seed)
    return [torch.randn(shape, generator=gen) for _ in range(n)]


def test_cfg1_small_batch_against_oracle(lib, cuda_dev):
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    inp = synth.make_inputs(w)
    m = build_module(w, cuda_dev)
    # (every reduction is fixed-order now: the 3x tolerance this case needed while the split-K Grams used atomics is gone)
    assert_parity(run_module(m, inp, cuda_dev), oracle_case(m, inp, w), w)
    assert m.last_polar_residual.item() <= m.POLAR_RESIDUAL_OK


def test_bf16_attention_maps(lib, cuda_dev):
    w = dataclasses.replace(synth.CONFIGS["cfg2"], B=6)
    inp = synth.make_inputs(w)            # attention values are bf16-representable already
    m = build_module(w, cuda_dev)
    a = run_module(m, inp, cuda_dev, attn_dtype=torch.float32)
    b = run_module(m, inp, cuda_dev, attn_dtype=torch.bfloat16)
    assert abs(a["loss"].item() - b["loss"].item()) <= 1e-6 * abs(a["loss"].item())
    # the values are bf16-representable, so both dtypes feed identical numbers: identical results, bit for bit
    for l in a["grad_student"]:
        assert torch.equal(a["grad_student"][l], b["grad_student"][l])
    assert torch.equal(a["grad_log_temperatures"], b["grad_log_temperatures"])
    assert_parity(b, oracle_case(m, inp, w), w)


def test_cfg2_full_size_against_reference_golden(lib, cuda_dev):
    """BASELINE.json configs[1] — the configuration the metric is quoted on — at its full size (B=256, bf16 tokens):
    loss, exact ranks, temperature gradients and student-gradient norms / subsamples / probes of the reference
    (tests/golden/cfg2.pt; the reference took ~40 s and 24 GB of host RAM for this step)."""
    g, w = load_golden("cfg2")
    inp = synth.make_inputs(w, seed=g["seed"])
    m = build_module(w, cuda_dev)
    out = run_module(m, inp, cuda_dev, attn_dtype=torch.bfloat16)
    assert out["ranks"] == g["ranks"]
    assert abs(out["loss"].item() - g["loss"].item()) <= TOL_LOSS * abs(g["loss"].item())
    assert ((out["grad_log_temperatures"] - g["grad_log_temperatures"]).abs() <= TOL_TGRAD * g["grad_log_temperatures"].abs()).all()
    for l in g["token_layers"]:
        assert abs(out["grad_student"][l].norm() - g["grad_student_norm"][l]) <= TOL_SGRAD * g["grad_student_norm"][l]
        assert rel(out["grad_student"][l].flatten()[::997], g["grad_student_sub"][l]) < TOL_SGRAD


@pytest.mark.parametrize("name", ["cfg3_b8", "cfg4_b4", "cfg5_b2"])
def test_cfg345_reduced_batch_against_reference_golden(lib, cuda_dev, name):
    """BASELINE.json configs[2..4] - ResNet-50 7x7 grid -> ViT-S (rank-deficient cross-covariance, 49 -> 196 resampling,
    uniform attention), ViT-S <- ViT-L (D_s = 384 > N - 1, 24-way mixing), DeiT-S <- DeiT-B at 576 tokens - with every
    dimension of the named configuration except the batch, against the UNMODIFIED reference (tests/golden, made by
    `python -m oracle.make_golden small`) and the oracle, at the north-star tolerances."""
    g, w = load_golden(name)
    inp = synth.make_inputs(w, seed=g["seed"])
    m = build_module(w, cuda_dev)
    out = run_module(m, inp, cuda_dev)
    assert out["ranks"] == g["ranks"]
    assert abs(out["loss"].item() - g["loss"].item()) <= TOL_LOSS * abs(g["loss"].item())
    gt, rt = out["grad_log_temperatures"], g["grad_log_temperatures"]
    # (single-layer teacher: w == 1 and the reference's temperature gradient is exactly 0; an fma leaves ~1e-7 of rounding here)
    assert ((gt - rt).abs() <= TOL_TGRAD * rt.abs() + (1e-6 if w.Lt == 1 else 1e-7)).all(), f"temperature grads {gt.tolist()} vs {rt.tolist()}"
    for l in g["token_layers"]:
        assert abs(out["grad_student"][l].norm() - g["grad_student_norm"][l]) <= TOL_SGRAD * g["grad_student_norm"][l]
        assert rel(out["grad_student"][l].flatten()[::997], g["grad_student_sub"][l]) < TOL_SGRAD
        pr = torch.stack([(out["grad_student"][l] * p).sum() for p in _probes(out["grad_student"][l].shape)])
        assert (pr - g["grad_student_probe"][l]).abs().max() <= TOL_SGRAD * g["grad_student_norm"][l] * math.sqrt(out["grad_student"][l].numel()) * 0.05
    assert_parity(out, oracle_case(m, inp, w), w, tgrad_floor=1e-6 if w.Lt == 1 else 1e-7)


@pytest.mark.parametrize("shape", [dict(B=4, Ns=196, Nt=196, Ds=192, Dt=384, Lt=12, H=6, has_cls=True),        # cfg1 at B=4: feature form, fused polar kernel
                                   dict(B=3, Ns=220, Nt=110, Ds=216, Dt=256, Lt=2, H=2, has_cls=True),         # teacher-token form with resampling
                                   dict(B=4, Ns=300, Nt=300, Ds=256, Dt=512, Lt=3, H=2, has_cls=True)])        # global-memory eigen-solver, tiled products
def test_two_executions_are_bitwise_equal(lib, cuda_dev, shape):
    """Every cross-CTA reduction (split-K Grams, column sums, traces, weight-gradient dots, centring correction) is a
    fixed-order two-stage sum: two executions of the same step give the same bits (loss, every gradient)."""
    w = synth.Workload("repeat", shape["B"], shape["Ns"], shape["Nt"], shape["Ds"], shape["Dt"], shape["Lt"], shape["H"], shape["has_cls"])
    inp = synth.make_inputs(w, seed=5)
    m = build_module(w, cuda_dev)
    a = run_module(m, inp, cuda_dev)
    b = run_module(m, inp, cuda_dev)
    assert torch.equal(a["loss"], b["loss"]) and torch.equal(a["grad_log_temperatures"], b["grad_log_temperatures"])
    for l in a["grad_student"]:
        assert torch.equal(a["grad_student"][l], b["grad_student"][l])


def test_ill_conditioned_cross_covariance(lib, cuda_dev):
    """A steep student spectrum (0.94^i: kappa(C) ~ 2e5, smallest singular value 2e-6 ||C||_F - below the 3e-5 floor of the
    default 10-step schedule).  The reference's SVD gives every singular direction unit weight in the gradient
    (relational.py:48), so: (1) the residual reported by the default run exceeds the bound, (2) the module raises its step
    count on the next call with a warning, (3) with the longer schedule loss and student gradients match the fp64 oracle at
    the north-star tolerances."""
    import warnings
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    inp = synth.make_inputs(w)
    gen = torch.Generator().manual_seed(77)
    inp["student"] = {l: synth.geometric(w.B, w.Ns, w.Ds, gen, rho=0.94) for l in inp["student"]}
    m = build_module(w, cuda_dev)
    out10 = run_module(m, inp, cuda_dev)
    assert m.last_polar_residual.item() > m.POLAR_RESIDUAL_OK                 # (1) not converged, and reported
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        run_module(m, inp, cuda_dev)                                           # (2) the next call reads the residual back
    assert m.polar_steps == 11 and any("polar iteration" in str(r.message) for r in rec)       # one step at a time
    m.polar_steps = 14
    out = run_module(m, inp, cuda_dev)
    assert m.last_polar_residual.item() <= m.POLAR_RESIDUAL_OK
    ref = oracle_case(m, inp, w, dtype=torch.float64)
    assert out["ranks"] == ref["ranks"]
    assert abs(out["loss"].item() - ref["loss"].item()) <= TOL_LOSS * abs(ref["loss"].item())
    worst10 = max(rel(out10["grad_student"][l], ref["grad_student"][l]) for l in ref["grad_student"])
    for l in ref["grad_student"]:
        assert rel(out["grad_student"][l], ref["grad_student"][l]) < TOL_SGRAD, f"student grad layer {l} (10 steps gave {worst10:.2e})"


# ------------------------------------------------------------------------------------------------ properties
def _device_case(w, dev, seed=7):
    import bench
    return bench.device_inputs(w, dev, seed)


def _geo_and_grads(m, student, teacher, attn):
    S = {l: v.detach().clone().requires_grad_() for l, v in student.items()}
    m.zero_grad(set_to_none=True)
    geo = m.geo_loss(S, teacher, attn)
    geo.backward()
    torch.cuda.synchronize()
    return geo.detach(), {l: S[l].grad for l in S}, m.layer_selector.log_temperatures.grad.clone(), m.layer_selector.subspace_ranks


def test_full_size_properties(lib, cuda_dev):
    """At BASELINE.json configs[1] size (B=256), on inputs generated on the device:
      (1) scaling student and teacher tokens by 2 (exact in bf16) multiplies the Procrustes loss by 4 and leaves
          ranks and mixing weights unchanged (subspaces and angles are scale invariant);
      (2) permuting the batch leaves the loss unchanged (pooled statistics are sums) and permutes the gradients;
      (3) a teacher that is an orthogonal image of the student gives (near) zero Procrustes residual
          (relational.py:36-50 is min_R ||s_w R - t_w||^2, SURVEY.md A.10)."""
    w = synth.CONFIGS["cfg2"]
    m = build_module(w, cuda_dev)
    _, _, student, teacher, attn = _device_case(w, cuda_dev)
    geo, gs, gt, ranks = _geo_and_grads(m, student, teacher, attn)
    w0 = m.layer_selector.last_mixing_weights.clone()
    assert math.isfinite(geo.item()) and all(r >= 1 for r in ranks.values())

    geo2, gs2, gt2, ranks2 = _geo_and_grads(m, {l: v * 2 for l, v in student.items()}, {j: v * 2 for j, v in teacher.items()}, attn)
    assert ranks2 == ranks
    assert abs(geo2.item() - 4 * geo.item()) <= 2e-4 * abs(4 * geo.item())
    assert (m.layer_selector.last_mixing_weights - w0).abs().max() < 1e-4
    for l in gs:
        assert rel(gs2[l].float(), 2 * gs[l].float()) < TOL_SGRAD

    perm = torch.randperm(w.B, device=cuda_dev)
    geo3, gs3, gt3, ranks3 = _geo_and_grads(m, {l: v[perm] for l, v in student.items()}, {j: v[perm] for j, v in teacher.items()},
                                            {j: v[perm] for j, v in attn.items()})
    assert ranks3 == ranks
    assert abs(geo3.item() - geo.item()) <= 1e-4 * abs(geo.item())
    assert rel(gt3, gt) < TOL_TGRAD
    for l in gs:
        assert rel(gs3[l].float(), gs[l][perm].float()) < TOL_SGRAD

    gen = torch.Generator(device=cuda_dev).manual_seed(5)
    R = torch.linalg.qr(torch.randn(w.Dt, w.Dt, generator=gen, device=cuda_dev))[0][: w.Ds]      # Ds x Dt, R R^T = I
    s_last = student[w.token_layers()[-1]].float()
    noise = 1e-2 * torch.randn(w.B, w.Nt, w.Dt, generator=gen, device=cuda_dev)      # keeps the teacher token Gram full rank
    rot = {j: (s_last @ R + noise).bfloat16() for j in teacher}
    same = {l: student[w.token_layers()[-1]] for l in student}
    geo4, _, _, _ = _geo_and_grads(m, same, rot, attn)
    assert abs(geo4.item()) < 2e-3 * abs(geo.item())


def _two_rank_case(cuda_dev, tmp_path, env_extra):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "ranks"
    out.mkdir()
    port = 29500 + (os.getpid() % 2000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tests", "sharded_worker.py"), str(out)]
    env = dict(os.environ, **env_extra)
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=8)
    inp = synth.make_inputs(w)
    m = build_module(w, cuda_dev)
    single = run_module(m, inp, cuda_dev)
    parts = [torch.load(out / f"rank{r_}.pt", weights_only=False) for r_ in range(2)]
    assert parts[0]["ranks"] == single["ranks"] == parts[1]["ranks"]
    for p in parts:
        assert abs(p["loss"].item() - single["loss"].item()) <= 1e-4 * abs(single["loss"].item())
        assert (p["w"] - single["w"]).abs().max() < 1e-5
        # every rank holds the gradient of the GLOBAL-mean loss w.r.t. the (replicated) log_temperatures
        assert rel(p["grad_log_temperatures"], single["grad_log_temperatures"]) < TOL_TGRAD
    for l in single["grad_student"]:
        # per-rank loss is the mean over the local half batch -> local gradients are 2x the global-mean gradients
        cat = torch.cat([parts[0]["grad_student"][l], parts[1]["grad_student"][l]]) / 2
        assert rel(cat, single["grad_student"][l]) < TOL_SGRAD


def test_two_rank_sharding_matches_single_process(lib, cuda_dev, tmp_path):
    """SURVEY.md §8(e): two ranks each holding half the batch, pooled statistics and d loss / d w summed across
    ranks, against ONE process on the concatenated batch.  Both ranks share cuda:0 (gloo moves the CUDA buffers),
    so the test runs on a single-GPU box; the NCCL variant below needs two GPUs."""
    _two_rank_case(cuda_dev, tmp_path, {"BASD_SHARD_DEVICE": "cuda:0"})


def test_two_rank_nccl_on_two_gpus_matches_single_process(lib, cuda_dev, tmp_path):
    """The same comparison with one rank per GPU over NCCL (the configuration bench.py and a real run use): loss, ranks,
    mixing weights, temperature gradients and the concatenated student gradients of two ranks on two B200s against a
    single process on the whole batch.  Skipped on single-GPU boxes."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _two_rank_case(cuda_dev, tmp_path, {})


def test_host_stager_matches_device_path(lib, cuda_dev):
    """The host-buffer entry (HostStager: CLS-row gather, copy stream, double-buffered slots) gives the same loss and
    gradients as handing device tensors to the module, for two consecutive submissions that reuse the slots."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    m = build_module(w, cuda_dev)
    stager = pkg.HostStager(m)
    for seed in (1234, 99, 7):
        inp = synth.make_inputs(w, seed=seed, attn_dtype=torch.bfloat16)
        ref = run_module(m, inp, cuda_dev, attn_dtype=torch.bfloat16)
        pin = lambda t: t.pin_memory()
        h = stager.submit(pin(inp["logits"]), pin(inp["targets"]), {l: pin(v) for l, v in inp["student"].items()},
                          {j: pin(v) for j, v in inp["teacher"].items()}, {j: pin(v) for j, v in inp["attn"].items()})
        m.zero_grad(set_to_none=True)
        loss = stager.run(h)
        loss.backward()
        torch.cuda.synchronize()
        assert abs(loss.item() - ref["loss"].item()) <= 1e-5 * abs(ref["loss"].item())
        assert rel(m.layer_selector.log_temperatures.grad.cpu(), ref["grad_log_temperatures"]) < TOL_TGRAD
        for l in ref["grad_student"]:
            # same kernels on the same values: bitwise the same gradients
            assert torch.equal(h["leaf_student"][l].grad.float().cpu(), ref["grad_student"][l])
        assert stager.h2d_bytes_last < 1.05 * (sum(v.numel() * 2 for v in inp["teacher"].values()) + sum(v.numel() * 2 for v in inp["student"].values())
                                               + inp["logits"].numel() * 4 + 8 * w.B + w.Lt * w.B * w.H * (w.Nt + 1) * 2)


def test_cls_attention_rows_from_q_k(lib, cuda_dev):
    """SURVEY.md section 8(f) rank 1: the CLS attention row straight from q and k equals row 0 of the reference hook's
    softmax(q k^T * scale) (src/models/teacher.py:33-37), for fp32 and bf16, contiguous and fused-qkv strided views; and
    feeding those rows to the loss gives the same result as feeding the full maps."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    w = dataclasses.replace(synth.CONFIGS["cfg1"], B=4)
    B, H, S, dh = w.B, w.H, w.Nt + 1, 64
    g = torch.Generator().manual_seed(3)
    qkv = torch.randn(B, S, 3, H, dh, generator=g).bfloat16()          # timm layout: reshape(B, S, 3, H, dh).permute(2, 0, 3, 1, 4)
    q, k, _ = qkv.permute(2, 0, 3, 1, 4).unbind(0)                      # strided views [B, H, S, dh]
    full = torch.softmax((q.float() @ k.float().transpose(-2, -1)) * dh ** -0.5, dim=-1)
    for dt in (torch.float32, torch.bfloat16):
        for contiguous in (False, True):
            qd, kd = q.to(dt).to(cuda_dev), k.to(dt).to(cuda_dev)
            if contiguous:
                qd, kd = qd.contiguous(), kd.contiguous()
            rows = pkg.cls_attention_rows(qd, kd)
            assert rows.shape == (B, H, 1, S)
            assert (rows.cpu() - full[:, :, 0:1, :]).abs().max() < 2e-6
    inp = synth.make_inputs(w)
    m = build_module(w, cuda_dev)
    S_ = {l: v.to(cuda_dev) for l, v in inp["student"].items()}
    T_ = {j: v.to(cuda_dev) for j, v in inp["teacher"].items()}
    maps = {j: full.to(cuda_dev) for j in T_}
    rows_only = {j: pkg.cls_attention_rows(q.to(cuda_dev), k.to(cuda_dev)) for j in T_}
    a = m.geo_loss(S_, T_, maps)
    b = m.geo_loss(S_, T_, rows_only)
    assert abs(a.item() - b.item()) <= 1e-5 * abs(a.item())


@pytest.mark.parametrize("shape", [dict(B=5, Ns=36, Nt=36, Ds=32, Dt=32, Lt=4, H=1, P=1), dict(B=2, Ns=70, Nt=90, Ds=64, Dt=136, Lt=2, H=2, P=4),
                                   dict(B=9, Ns=210, Nt=210, Ds=200, Dt=256, Lt=2, H=2, P=2), dict(B=4, Ns=300, Nt=300, Ds=256, Dt=512, Lt=3, H=2, P=2),
                                   dict(B=3, Ns=220, Nt=110, Ds=216, Dt=256, Lt=2, H=2, P=2), dict(B=4, Ns=196, Nt=196, Ds=192, Dt=768, Lt=12, H=12, P=4)])
def test_workspace_contents_do_not_matter(lib, cuda_dev, shape):
    """No kernel reads workspace bytes that it, or an earlier kernel of the same step, has not written: the loss and every
    gradient are bitwise identical whether the freshly allocated workspace holds zeros, NaN bit patterns or random bytes
    (padding rows / columns of the tiled operands, split-K partials, scratch of the eigen-solver ...)."""
    from vit_bias_aware_structural_distillation_b200 import loss as L
    w = synth.Workload("garbage", shape["B"], shape["Ns"], shape["Nt"], shape["Ds"], shape["Dt"], shape["Lt"], shape["H"], True, P=shape["P"])
    inp = synth.make_inputs(w, seed=11)
    fills = {"zero": lambda ws: ws.zero_(), "nan": lambda ws: ws.fill_(0xFF),
             "rand": lambda ws: ws.copy_(torch.randint(0, 256, ws.shape, dtype=torch.uint8, device=ws.device))}
    res = {}
    try:
        for name, f in fills.items():
            L._debug_workspace_fill = f
            res[name] = run_module(build_module(w, cuda_dev), inp, cuda_dev)
    finally:
        L._debug_workspace_fill = None
    ref = res["zero"]
    for name in ("nan", "rand"):
        o = res[name]
        assert o["ranks"] == ref["ranks"]
        assert torch.equal(o["loss"], ref["loss"]) and torch.equal(o["grad_log_temperatures"], ref["grad_log_temperatures"]), name
        for l in ref["grad_student"]:
            assert torch.equal(o["grad_student"][l], ref["grad_student"][l]), f"{name}: student grad layer {l}"


@pytest.mark.parametrize("shape", [
    dict(B=3, Ns=50, Nt=50, Ds=40, Dt=72, Lt=2, H=3, P=3),          # nothing a multiple of 16; three extraction points
    dict(B=5, Ns=36, Nt=36, Ds=32, Dt=32, Lt=4, H=1, P=1),          # a single extraction point (combined.py:34-36), D_t == D_s
    dict(B=2, Ns=130, Nt=130, Ds=96, Dt=200, Lt=3, H=2, P=2),       # N > 128: two 128-row output tiles in the N x N products
    dict(B=2, Ns=70, Nt=90, Ds=64, Dt=136, Lt=2, H=2, P=4),         # down-sampling 90 -> 70 with D_s exactly one column block
    dict(B=9, Ns=210, Nt=210, Ds=200, Dt=256, Lt=2, H=2, P=2),      # D_s > 192: 7-chunk cluster Jacobi, unfused polar products, 4 column blocks
    dict(B=3, Ns=160, Nt=160, Ds=144, Dt=192, Lt=2, H=2, P=2),      # fused polar kernel with a partial second row tile (144 = 128 + 16)
    dict(B=4, Ns=320, Nt=320, Ds=192, Dt=384, Lt=3, H=2, P=2),      # N > 256: column-tiled polar products, tiled token Gram
    dict(B=4, Ns=300, Nt=300, Ds=256, Dt=512, Lt=3, H=2, P=2),      # D_s > 224: global-memory eigen-solver, three row tiles
    dict(B=4, Ns=100, Nt=100, Ds=136, Dt=160, Lt=2, H=2, P=2),      # D_s > N - 1 (teacher-token form), nothing a multiple of 64
    dict(B=3, Ns=220, Nt=110, Ds=216, Dt=256, Lt=2, H=2, P=2),      # teacher-token form with resampling 110 -> 220, D_s % 16 == 8
    dict(B=3, Ns=240, Nt=220, Ds=232, Dt=256, Lt=2, H=2, P=2),      # teacher-token form, N_t > 208: two column tiles in the polynomial product
    dict(B=3, Ns=100, Nt=140, Ds=136, Dt=160, Lt=2, H=2, P=2),      # D_s > N_s - 1 with a FINER teacher grid: token-space form on the student's grid
    dict(B=1, Ns=50, Nt=50, Ds=64, Dt=96, Lt=2, H=2, P=2),          # pooled rows M = 50 < D_s (layer_selector.py:14-15: the M eigenvalues of F F^T / M)
    dict(B=2, Ns=40, Nt=40, Ds=96, Dt=128, Lt=3, H=2, P=2),         # M = 80 < D_s = 96, three teacher layers
])
def test_irregular_shapes_against_oracle(lib, cuda_dev, shape):
    """Shapes off the BASELINE grid: padding, tails and tile boundaries of every kernel against the fp32 oracle."""
    w = synth.Workload("irregular", shape["B"], shape["Ns"], shape["Nt"], shape["Ds"], shape["Dt"], shape["Lt"], shape["H"], True, P=shape["P"])
    inp = synth.make_inputs(w, seed=11)
    m = build_module(w, cuda_dev)
    out = run_module(m, inp, cuda_dev)
    ref = oracle_case(m, inp, w)
    assert out["ranks"] == ref["ranks"]
    assert abs(out["loss"].item() - ref["loss"].item()) <= TOL_LOSS * abs(ref["loss"].item())
    assert (out["w"] - ref["w"].float()).abs().max() < 2e-4
    gt, rt = out["grad_log_temperatures"], ref["grad_log_temperatures"].float()
    # Temperature gradients: entries that are themselves a cancellation to a few % of the largest one are judged against the
    # largest.  The softmax derivative is a difference of nearly equal per-layer terms; at these sizes (a few hundred pooled
    # rows, one to four layers) that amplifies the 2^-17 precision of the split-bf16 polar products to at most 3e-3 (measured
    # against the fp64 oracle: the reference's own fp32 is 1e-5 there, so this is OUR error, stated - not reference noise).
    # The BASELINE shapes are held to TOL_TGRAD = 1e-3 of each entry in the cfg1 - cfg5 tests.
    # That rounding noise averages out as 1 / sqrt(elements of the mixed teacher): shapes below the 2.5e4 elements of the
    # smallest other case get the bound scaled accordingly (P B N D_t = 5.8e3 in the single-point shape: measured -2.9e-3 and
    # +3.2e-3 on two builds whose mixing weights differ in the 7th digit).
    elems = shape["P"] * shape["B"] * shape["Ns"] * shape["Dt"]
    tg_tol = 3e-3 * max(1.0, math.sqrt(2.5e4 / elems))
    assert ((gt - rt).abs() <= tg_tol * rt.abs().max()).all(), f"temperature grads {gt.tolist()} vs {rt.tolist()}"
    for l in ref["grad_student"]:
        assert rel(out["grad_student"][l], ref["grad_student"][l]) < TOL_SGRAD, f"student grad layer {l}"
    if m.last_polar_residual.item() > m.POLAR_RESIDUAL_OK:
        # near-square cross-covariances (D_s within a few rows of N - 1) have a few singular values below the 3e-5 floor of
        # the default schedule: reported by the residual, and gone with the two extra steps the module would add by itself
        assert shape["Ds"] >= min(shape["Ns"], shape["Nt"]) - 10
        m.polar_steps = 12
        out = run_module(m, inp, cuda_dev)
        assert m.last_polar_residual.item() <= m.POLAR_RESIDUAL_OK
        for l in ref["grad_student"]:
            assert rel(out["grad_student"][l], ref["grad_student"][l]) < TOL_SGRAD


def _probe(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(shape, generator=g)


def test_standalone_entry_points_against_reference_golden(lib, cuda_dev):
    """The reference's three standalone entry points of the path, each through its own drop-in:
    geometric_relational_loss (relational.py:5-50; BASD_MODE_PAIR), _align_token_count (combined.py:9-14; its own two kernels) and
    GrassmannianLayerSelector.forward (layer_selector.py:116-152; BASD_MODE_SELECTOR) against tests/golden/standalone.pt."""
    import vit_bias_aware_structural_distillation_b200 as pkg
    g = torch.load(os.path.join(GOLD, "standalone.pt"), weights_only=False)
    w, inp, t_al, attn_same, attn_nocls = synth.standalone_inputs()
    layer0 = w.token_layers()[0]
    for key, attn, has_cls in (("pair_cls", attn_same, True), ("pair_cls_resampled", inp["attn"][0].float(), True), ("pair_nocls", attn_nocls, False)):
        for act in (torch.bfloat16, torch.float32):
            s = inp["student"][layer0].to(cuda_dev).to(act).requires_grad_()
            loss = pkg.geometric_relational_loss(s, t_al.to(cuda_dev).to(act), attn.to(cuda_dev), has_cls_token=has_cls)
            loss.backward()
            assert abs(loss.item() - g[key]["loss"].item()) <= TOL_LOSS * abs(g[key]["loss"].item()), key
            assert rel(s.grad.float().cpu(), g[key]["grad_student"]) < TOL_SGRAD, key
    for key, n_out in (("align_up", 48), ("align_down", 20), ("align_same", 36)):
        x = inp["teacher"][0].float().to(cuda_dev).requires_grad_()
        y = pkg.align_token_count(x, n_out)
        assert (y is x) == g[key]["same_object"]
        (y * _probe(y.shape, 5).to(cuda_dev)).sum().backward()
        assert torch.allclose(y.detach().cpu(), g[key]["out"], atol=1e-5), key
        assert torch.allclose(x.grad.cpu(), g[key]["grad_in"], atol=1e-5), key
        xv = torch.zeros(x.shape[0], x.shape[1] + 1, x.shape[2], device=cuda_dev, dtype=torch.bfloat16)     # a CLS-stripped bf16 view
        xv[:, 1:] = inp["teacher"][0].to(cuda_dev)
        yv = pkg.align_token_count(xv[:, 1:, :], n_out)
        assert rel(yv.float().cpu(), g[key]["out"]) < 4e-3, key                                               # bf16 output rounding
    torch.manual_seed(0)
    sel = pkg.GrassmannianLayerSelector(num_extraction_points=w.P, student_dim=w.Ds, teacher_dim=w.Dt).to(cuda_dev)
    S = {l: v.float().to(cuda_dev).requires_grad_() for l, v in inp["student"].items()}
    T = {j: v.float().to(cuda_dev) for j, v in inp["teacher"].items()}
    A = {j: v.float().to(cuda_dev) for j, v in inp["attn"].items()}
    mt, ma = sel(S, T, A, w.token_layers())
    total = sum((mt[l] * _probe(mt[l].shape, 6 + i).to(cuda_dev)).sum() for i, l in enumerate(w.token_layers()))
    total = total + sum((ma[l] * _probe(ma[l].shape, 16 + i).to(cuda_dev)).sum() for i, l in enumerate(w.token_layers()))
    total.backward()
    gs = g["selector"]
    assert sel.subspace_ranks == gs["ranks"]
    for l in w.token_layers():
        assert rel(mt[l].detach().cpu(), gs["mixed_tokens"][l]) < 1e-4
        assert rel(ma[l][:, :, 0, :].detach().cpu(), gs["mixed_attn_cls_row"][l]) < 1e-4
        assert rel(S[l].grad.cpu(), gs["grad_student"][l]) < TOL_SGRAD
    gt, rt = sel.log_temperatures.grad.cpu(), gs["grad_log_temperatures"]
    assert ((gt - rt).abs() <= TOL_TGRAD * rt.abs() + 1e-7).all(), f"temperature grads {gt.tolist()} vs {rt.tolist()}"


def test_uwso_combine_matches_the_reference_expression(lib, cuda_dev):
    """combined.py:78-85 as one kernel (basd_uwso_combine): bit-identical total, the reference's gradients, NaN propagation."""
    from vit_bias_aware_structural_distillation_b200.loss import _UwsoCombine
    torch.manual_seed(3)
    cases = [(2.3, 14.08), (6.9, 0.37), (1e-9, 5.0), (0.0, 1.0), (float("nan"), 1.0), (3.0, float("inf"))]
    for ce_v, geo_v in cases:
        ce = torch.tensor(ce_v, device=cuda_dev, requires_grad=True)
        geo = torch.tensor(geo_v, device=cuda_dev, requires_grad=True)
        out = _UwsoCombine.apply(ce, geo, ce.detach(), geo.detach())
        out.backward()
        ce_r = torch.tensor(ce_v, device=cuda_dev, requires_grad=True)
        geo_r = torch.tensor(geo_v, device=cuda_dev, requires_grad=True)
        vals = [ce_r, geo_r]
        eps = torch.finfo(torch.float32).eps
        inv = torch.stack([1.0 / v.detach().clamp(min=eps) for v in vals])
        wts = inv / inv.sum()
        ref = sum(wts[i] * vals[i] for i in range(2))
        ref.backward()
        assert torch.equal(out.isnan(), ref.isnan()), (ce_v, geo_v)
        if not ref.isnan():
            assert out.item() == ref.item(), (ce_v, geo_v, out.item(), ref.item())
            assert torch.equal(ce.grad, ce_r.grad) and torch.equal(geo.grad, geo_r.grad), (ce_v, geo_v)
