"""Drop-in replacement for the reference's `src/losses` package (BASD distillation loss), running the whole
selector + interpolation + Procrustes path and its analytic backward as sm_100a CUDA kernels behind the C ABI of
include/basd_b200.h.

Mirrors, with the same names / argument meaning / state_dict keys:
  * BASDLoss                      /root/reference/src/losses/combined.py:17-85
  * GrassmannianLayerSelector     /root/reference/src/losses/layer_selector.py:40-152
  * marchenko_pastur_rank         /root/reference/src/losses/layer_selector.py:8-20
  * geometric_relational_loss     /root/reference/src/losses/relational.py:5-50   (standalone: one pair, selector bypassed)
  * _align_token_count            /root/reference/src/losses/combined.py:9-14
Inside BASDLoss.forward the three are ONE fused op (shared statistics, resampling folded into the teacher mix); the
standalone entry points run the same kernels through basd_shape.mode (include/basd_b200.h).

CE (`base_criterion`) and the two-scalar UW-SO weighting (combined.py:56,78-85) stay stock PyTorch so that any
criterion and soft or hard targets keep working; everything between them is one custom op, `basd_b200::geo_forward`,
with a registered backward op `basd_b200::geo_backward` (no autograd through LAPACK).
"""
from __future__ import annotations

import ctypes
import math
from typing import List, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from ._lib import ATTN_QUERY_MEAN, DTYPE_BF16, DTYPE_F32, DTYPE_F32_SPLIT, MODE_LOSS, MODE_PAIR, MODE_SELECTOR, Inputs, Shape

# How the loss reads fp32 tokens: "bf16" rounds them to bf16 on entry (the default), "fp32" carries them as split-bf16 pairs
# hi + lo through every kernel that reads them (fp32-class accuracy; DESIGN.md section 8).  bf16 tokens read the same either way.
TOKEN_PRECISIONS = ("bf16", "fp32")


def _check_token_precision(token_precision) -> str:
    if not isinstance(token_precision, str) or token_precision not in TOKEN_PRECISIONS:
        raise _lib.BasdError(f"token_precision must be one of {TOKEN_PRECISIONS}, got {token_precision!r}")
    return token_precision


def _split_tokens(students, teachers, token_precision: str) -> bool:
    """True when the tokens go in as split-bf16 pairs: token_precision "fp32" and any token tensor that is not bf16."""
    return _check_token_precision(token_precision) == "fp32" and any(t.dtype != torch.bfloat16 for t in list(students) + list(teachers))


# --------------------------------------------------------------------------------------------- low-level plumbing
def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return DTYPE_F32
    if t.dtype == torch.bfloat16:
        return DTYPE_BF16
    raise _lib.BasdError(f"unsupported dtype {t.dtype} (float32 or bfloat16 expected)")


def _stream_ptr(dev=None) -> int:
    """Current stream of the tensors' device (not of whatever device happens to be current)."""
    return torch.cuda.current_stream(dev).cuda_stream


def _prepare(students: Sequence[torch.Tensor], teachers: Sequence[torch.Tensor], attns: Sequence[torch.Tensor],
             proj_s: torch.Tensor, proj_t: torch.Tensor, log_temperatures: torch.Tensor, has_cls: bool, world_size: int,
             polar_steps: int = 0, mode: int = MODE_LOSS, token_precision: str = "bf16"):
    """Builds the C structs.  Returns (shape, inputs, keepalive) — keepalive holds every tensor whose pointer is used.
    mode (include/basd_b200.h): MODE_PAIR reads no projections / temperatures, MODE_SELECTOR no attention maps.
    token_precision "fp32": if any token tensor is not bf16, all of them go in as fp32 split-bf16 pairs (BASD_DTYPE_F32_SPLIT)."""
    split = _split_tokens(students, teachers, token_precision)
    if not students or not teachers or (mode != MODE_SELECTOR and len(teachers) != len(attns)):
        raise _lib.BasdError("need >= 1 student tensor, >= 1 teacher tensor and one attention map per teacher layer")
    if mode == MODE_SELECTOR:
        attns = []
    dev = students[0].device
    if dev.type != "cuda":
        raise _lib.BasdError("the BASD loss path runs on a CUDA device only (no CPU fallback); got tensors on " + str(dev))
    act_dt = students[0].dtype
    if act_dt not in (torch.float32, torch.bfloat16) or split:      # (bf16 -> fp32 is exact)
        students = [s.float() for s in students]
        act_dt = torch.float32
    teachers = [t if t.dtype == act_dt else t.to(act_dt) for t in teachers]
    students = [s if s.dtype == act_dt else s.to(act_dt) for s in students]
    if act_dt == torch.bfloat16:
        # bf16 operands are consumed IN PLACE by TMA: dense [B,N,D] tensors, or the CLS-stripped views out[:, 1:, :] of dense
        # [B,N+1,D] tensors that the reference's extraction hooks hand over (trainer.py:29, teacher.py:157) - no copy for
        # either.  Anything else (e.g. the CNN [B,HW,C] transposed view, teacher.py:155) is made contiguous once.
        def in_place(t):
            n, d = t.shape[1], t.shape[2]
            return t.is_contiguous() or (t.stride() == ((n + 1) * d, d, 1) and t.data_ptr() % 16 == 0)
        if not all(in_place(s) for s in students) or len({s.stride() for s in students}) > 1:
            students = [s.contiguous() for s in students]
        if not all(in_place(t) for t in teachers) or len({t.stride() for t in teachers}) > 1:
            teachers = [t.contiguous() for t in teachers]
    else:                                   # fp32: the pack kernel reads through arbitrary strides; equalise them
        if len({s.stride() for s in students}) > 1:
            students = [s.contiguous() for s in students]
        if len({t.stride() for t in teachers}) > 1:
            teachers = [t.contiguous() for t in teachers]
    att_dt = attns[0].dtype if attns and attns[0].dtype in (torch.float32, torch.bfloat16) else torch.float32
    attns = [a if a.dtype == att_dt else a.to(att_dt) for a in attns]
    if len({a.stride() for a in attns}) > 1:
        attns = [a.contiguous() for a in attns]
    B, Ns, Ds = students[0].shape
    Bt, Nt, Dt = teachers[0].shape
    if Bt != B:
        raise _lib.BasdError("student and teacher batch sizes differ")
    # the kernels index every tensor of a list with the shape and strides of the first: check them all (the reference
    # raises from torch.stack / matmul on ragged inputs, layer_selector.py:128-129)
    for name, ts in (("student", students), ("teacher", teachers), ("attention", attns)):
        for k, t in enumerate(ts):
            if t.device != dev:
                raise _lib.BasdError(f"{name} tensor {k} is on {t.device}, expected {dev}")
            if t.shape != ts[0].shape or t.stride() != ts[0].stride():
                raise _lib.BasdError(f"{name} tensor {k} has shape {tuple(t.shape)} / strides {t.stride()}, tensor 0 has {tuple(ts[0].shape)} / {ts[0].stride()}")
    if len(students) > _lib.MAX_POINTS or len(teachers) > _lib.MAX_LAYERS:
        raise _lib.BasdError(f"at most {_lib.MAX_POINTS} extraction points and {_lib.MAX_LAYERS} teacher layers")
    if mode != MODE_PAIR:
        if tuple(proj_s.shape) != (Ds, Ds) or tuple(proj_t.shape) != (Ds, Dt):
            raise _lib.BasdError(f"proj_s {tuple(proj_s.shape)} / proj_t {tuple(proj_t.shape)} do not match student width {Ds} and teacher width {Dt} "
                                 "(was the module built with the right student_dim / teacher_dim?)")
        if log_temperatures.numel() != len(students):
            raise _lib.BasdError(f"{log_temperatures.numel()} log_temperatures for {len(students)} student extraction points")
    H = attns[0].shape[1] if attns else 1
    attn_code = int(has_cls)
    if attns:
        exp_attn = (B, H, Nt + 1, Nt + 1) if has_cls else (B, H, Nt, Nt)
        # rows only: the CLS query row (HostStager, cls_attention_rows; all relational.py:24 reads) or, without a CLS token, the
        # query mean per head (query_mean_attention; all relational.py:27 reads)
        rows_only = (B, H, 1, Nt + 1) if has_cls else (B, H, 1, Nt)
        got = tuple(attns[0].shape)
        if got not in (exp_attn, rows_only):
            raise _lib.BasdError(f"attention shape {got} != expected {exp_attn} (or rows {rows_only})")
        if not has_cls and got != exp_attn:
            attn_code = ATTN_QUERY_MEAN
    proj_s = proj_s.detach().to(device=dev, dtype=torch.float32).contiguous()
    proj_t = proj_t.detach().to(device=dev, dtype=torch.float32).contiguous()
    logt = log_temperatures.detach().to(device=dev, dtype=torch.float32).contiguous()
    shape = Shape(B=B, Ns=Ns, Nt=Nt, Ds=Ds, Dt=Dt, Lt=len(teachers), P=len(students), H=H, has_cls=attn_code,
                  act_dtype=DTYPE_F32_SPLIT if split else _dtype_code(students[0]), attn_dtype=_dtype_code(attns[0]) if attns else DTYPE_F32, world_size=world_size,
                  polar_steps=int(polar_steps), mode=int(mode))
    inp = Inputs()
    for i, s in enumerate(students):
        inp.student[i] = s.data_ptr()
    for j, t in enumerate(teachers):
        inp.teacher[j] = t.data_ptr()
    for j, a in enumerate(attns):
        inp.attn[j] = a.data_ptr()
    for k in range(3):
        inp.student_strides[k] = students[0].stride(k)
        inp.teacher_strides[k] = teachers[0].stride(k)
    for k in range(4):
        inp.attn_strides[k] = attns[0].stride(k) if attns else 0
    if mode != MODE_PAIR:
        inp.proj_s, inp.proj_t = proj_s.data_ptr(), proj_t.data_ptr()
    inp.log_temperatures = logt.data_ptr()
    keep = (students, teachers, attns, proj_s, proj_t, logt)
    return shape, inp, keep


def workspace_view(shape: Shape, ws: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    """Typed view of a named workspace region (tests, collectives)."""
    lib = _lib.load()
    ptr, cnt = ctypes.c_void_p(), ctypes.c_size_t()
    _lib.check(lib.basd_view(ctypes.byref(shape), ws.data_ptr(), name.encode(), ctypes.byref(ptr), ctypes.byref(cnt)), "basd_view")
    off = ptr.value - ws.data_ptr()
    nbytes = cnt.value * torch.empty((), dtype=dtype).element_size()
    return ws[off:off + nbytes].view(dtype)


def _world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist, dist.get_world_size()
    return None, 1


# Test hook (tests/test_gpu_parity.py::test_workspace_contents_do_not_matter): called with the freshly allocated, uninitialised
# workspace so that a test can poison it - no kernel may read workspace bytes it (or an earlier kernel of the step) has not written.
_debug_workspace_fill = None


def _allreduce_sum(dist, t: torch.Tensor):
    dist.all_reduce(t, op=dist.ReduceOp.SUM)


# --------------------------------------------------------------------------------------------- custom ops
@torch.library.custom_op("basd_b200::geo_forward", mutates_args=())
def geo_forward(students: List[torch.Tensor], teachers: List[torch.Tensor], attns: List[torch.Tensor], proj_s: torch.Tensor,
                proj_t: torch.Tensor, log_temperatures: torch.Tensor, has_cls: bool, polar_steps: int, mode: int,
                token_precision: str) -> List[torch.Tensor]:
    """(polar_steps / mode / token_precision have no defaults on purpose: torch drops default-valued arguments from the autograd inputs.)
    mode: MODE_LOSS (the geometric term of BASDLoss), MODE_PAIR (geometric_relational_loss of one pair), MODE_SELECTOR
    (mixing weights only; differentiable through output 3).  token_precision: "bf16" or "fp32" (TOKEN_PRECISIONS).
    Returns [geo_loss (0-dim fp32), workspace (uint8), ranks (int32 [Lt]), mixing weights (fp32 [P, Lt]),
    polar residual (fp32 [1]: largest ||X X^T - I||_F going into the last Newton-Schulz step; <= 0.1 = converged)]."""
    lib = _lib.load()
    dist, world = _world()
    shape, inp, keep = _prepare(students, teachers, attns, proj_s, proj_t, log_temperatures, has_cls, world, polar_steps, mode,
                                token_precision)
    nbytes = ctypes.c_size_t()
    _lib.check(lib.basd_workspace_bytes(ctypes.byref(shape), ctypes.byref(nbytes)), "basd_workspace_bytes")
    dev = students[0].device
    with torch.cuda.device(dev):             # the library launches on the CURRENT device: make it the tensors' device
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        if _debug_workspace_fill is not None:
            _debug_workspace_fill(ws)
        geo = torch.empty((), dtype=torch.float32, device=dev)
        st = _stream_ptr(dev)
        _lib.check(lib.basd_forward_stats(ctypes.byref(shape), ctypes.byref(inp), ws.data_ptr(), st), "basd_forward_stats")
        if dist is not None and mode != MODE_PAIR:
            _allreduce_sum(dist, workspace_view(shape, ws, "stats"))
        _lib.check(lib.basd_forward_solve(ctypes.byref(shape), ctypes.byref(inp), ws.data_ptr(), geo.data_ptr(), st), "basd_forward_solve")
        ranks = workspace_view(shape, ws, "ranks", torch.int32).clone()
        w = workspace_view(shape, ws, "w").clone().view(shape.P, shape.Lt)
        resid = workspace_view(shape, ws, "polar_resid").clone()
    del keep
    return [geo, ws, ranks, w, resid]


def _fake_workspace_bytes(students, teachers, attns, has_cls, mode=MODE_LOSS, token_precision="bf16") -> int:
    """Same size as the real op's workspace (basd_workspace_bytes is host-only arithmetic on the shape)."""
    B, Ns, Ds = students[0].shape
    _, Nt, Dt = teachers[0].shape
    code = lambda t: DTYPE_BF16 if t.dtype == torch.bfloat16 else DTYPE_F32
    shape = Shape(B=B, Ns=Ns, Nt=Nt, Ds=Ds, Dt=Dt, Lt=len(teachers), P=len(students), H=attns[0].shape[1] if attns else 1, has_cls=int(has_cls),
                  act_dtype=DTYPE_F32_SPLIT if _split_tokens(students, teachers, token_precision) else code(students[0]), attn_dtype=code(attns[0]) if attns else DTYPE_F32, world_size=_world()[1], mode=int(mode))
    nbytes = ctypes.c_size_t()
    _lib.check(_lib.load().basd_workspace_bytes(ctypes.byref(shape), ctypes.byref(nbytes)), "basd_workspace_bytes")
    return int(nbytes.value)


@geo_forward.register_fake
def _(students, teachers, attns, proj_s, proj_t, log_temperatures, has_cls, polar_steps, mode, token_precision):
    dev = students[0].device
    return [torch.empty((), dtype=torch.float32, device=dev),
            torch.empty(_fake_workspace_bytes(students, teachers, attns, has_cls, mode, token_precision), dtype=torch.uint8, device=dev),
            torch.empty(len(teachers), dtype=torch.int32, device=dev),
            torch.empty(len(students), len(teachers), dtype=torch.float32, device=dev),
            torch.empty(1, dtype=torch.float32, device=dev)]


@torch.library.custom_op("basd_b200::geo_backward", mutates_args=("workspace",))
def geo_backward(grad_geo: torch.Tensor, workspace: torch.Tensor, students: List[torch.Tensor], teachers: List[torch.Tensor],
                 attns: List[torch.Tensor], proj_s: torch.Tensor, proj_t: torch.Tensor, log_temperatures: torch.Tensor,
                 has_cls: bool, mode: int, grad_w: torch.Tensor, token_precision: str) -> List[torch.Tensor]:
    """Returns [grad_log_temperatures, grad_student_0, ..., grad_student_{P-1}].  grad_w: d(total)/d(mixing weights) [P, Lt]
    in MODE_SELECTOR (then grad_geo is the scalar that multiplies it), an empty tensor otherwise."""
    lib = _lib.load()
    dist, world = _world()
    shape, inp, keep = _prepare(students, teachers, attns, proj_s, proj_t, log_temperatures, has_cls, world, 0, mode, token_precision)
    dev = students[0].device
    with torch.cuda.device(dev):
        st = _stream_ptr(dev)
        g = grad_geo.detach().to(device=dev, dtype=torch.float32).contiguous()
        _lib.check(lib.basd_backward_dots(ctypes.byref(shape), ctypes.byref(inp), workspace.data_ptr(), st), "basd_backward_dots")
        if mode == MODE_SELECTOR:
            workspace_view(shape, workspace, "gw").copy_(grad_w.detach().to(device=dev, dtype=torch.float32).reshape(-1))
        if dist is not None and mode != MODE_PAIR:
            _allreduce_sum(dist, workspace_view(shape, workspace, "gw"))
        out_dtype = students[0].dtype if students[0].dtype in (torch.float32, torch.bfloat16) else torch.float32
        grads = [torch.empty(s.shape, dtype=out_dtype, device=dev) for s in students]
        glt = torch.empty(shape.P, dtype=torch.float32, device=dev)
        ptrs = (ctypes.c_void_p * len(grads))(*[t.data_ptr() for t in grads])
        _lib.check(lib.basd_backward_finish(ctypes.byref(shape), ctypes.byref(inp), workspace.data_ptr(), g.data_ptr(), ptrs,
                                            DTYPE_BF16 if out_dtype == torch.bfloat16 else DTYPE_F32, glt.data_ptr(), st),
                   "basd_backward_finish")
    if world > 1:
        glt = glt / world          # every rank holds the summed gradient; keep the DDP-average convention
    del keep
    return [glt] + grads


@geo_backward.register_fake
def _(grad_geo, workspace, students, teachers, attns, proj_s, proj_t, log_temperatures, has_cls, mode, grad_w, token_precision):
    return [torch.empty_like(log_temperatures, dtype=torch.float32)] + [torch.empty_like(s) for s in students]


def _setup_context(ctx, inputs, output):
    students, teachers, attns, proj_s, proj_t, log_temperatures, has_cls = inputs[:7]
    ctx.n_students, ctx.n_teachers, ctx.n_attns = len(students), len(teachers), len(attns)
    ctx.has_cls = has_cls
    ctx.mode = int(inputs[8])
    ctx.token_precision = inputs[9]
    ctx.student_dtypes = [s.dtype for s in students]
    # only geo_loss carries a gradient; without this autograd materialises zeros_like() for every other output in
    # backward, the multi-GB uint8 workspace included (0.85 ms of fill kernels per step at B=256)
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(output[1], proj_s, proj_t, log_temperatures, *students, *teachers, *attns)


def _backward(ctx, grads):
    grad_geo = grads[0]
    saved = ctx.saved_tensors
    ws, proj_s, proj_t, logt = saved[:4]
    P, Lt, La = ctx.n_students, ctx.n_teachers, ctx.n_attns
    students = list(saved[4:4 + P])
    teachers = list(saved[4 + P:4 + P + Lt])
    attns = list(saved[4 + P + Lt:4 + P + Lt + La])
    grad_w = torch.empty(0, device=ws.device)
    if ctx.mode == MODE_SELECTOR:              # the gradient arrives through the mixing weights (output 3)
        grad_w = grads[3] if grads[3] is not None else torch.zeros(P, Lt, device=ws.device)
        grad_geo = torch.ones((), device=ws.device)
    elif grad_geo is None:
        grad_geo = torch.zeros((), device=ws.device)
    out = geo_backward(grad_geo, ws, students, teachers, attns, proj_s, proj_t, logt, ctx.has_cls, ctx.mode, grad_w, ctx.token_precision)
    gs = [g.to(dt) if g.dtype != dt else g for g, dt in zip(out[1:], ctx.student_dtypes)]
    return gs, [None] * Lt, [None] * La, None, None, out[0].to(logt.dtype), None, None, None, None


geo_forward.register_autograd(_backward, setup_context=_setup_context)


# --------------------------------------------------------------------------------------------- host staging
class HostStager:
    """Feeds the loss from HOST buffers (what `trainer.py:133-136` does for images, done here for the activations of an
    offline / CPU-resident teacher): double-buffered device slots, copies issued on a dedicated copy stream so that the
    transfer of step i+1 overlaps the loss of step i.  Of every teacher attention map `[B,H,N+1,N+1]` only the CLS query
    row is gathered and copied (relational.py:24 reads nothing else): 14.5 MB instead of 2.9 GB per step at
    BASELINE.json configs[1].  Teachers without a CLS token (relational.py:27) get whatever they hand over copied as it is:
    the whole map [B,H,N,N], or - from `query_mean_attention` - the query-mean rows [B,H,1,N], 1/N of the map's bytes.

        stager = HostStager(loss_module)
        h = stager.submit(logits, targets, student, teacher_tokens, teacher_attns)   # host tensors (pinned = async)
        loss = stager.run(h); loss.backward()
    """

    def __init__(self, module: "BASDLoss", device=None, depth: int = 2):
        self.module = module
        self.device = torch.device(device) if device is not None else next(module.buffers()).device
        if self.device.type != "cuda":
            raise _lib.BasdError("HostStager needs the loss module on a CUDA device")
        self.depth = depth
        self.copy_stream = torch.cuda.Stream(self.device)
        self._slots = [dict() for _ in range(depth)]
        self._next = 0
        self.h2d_bytes_last = 0

    def _dev(self, slot, key, like, shape=None):
        shape = tuple(shape if shape is not None else like.shape)
        buf = slot.get(key)
        if buf is None or buf.shape != shape or buf.dtype != like.dtype:
            buf = torch.empty(shape, dtype=like.dtype, device=self.device)
            slot[key] = buf
        return buf

    def _pinned(self, slot, key, like, shape):
        buf = slot.get(key)
        if buf is None or buf.shape != tuple(shape) or buf.dtype != like.dtype:
            buf = torch.empty(tuple(shape), dtype=like.dtype, pin_memory=True)
            slot[key] = buf
        return buf

    def submit(self, student_output, targets, student_intermediates, all_teacher_tokens, all_teacher_attns):
        slot = self._slots[self._next]
        self._next = (self._next + 1) % self.depth
        has_cls = bool(self.module.teacher_has_cls_token)
        # The async H2D copies issued from this slot's pinned staging buffers `depth` submits ago may still be in flight if the
        # caller never synchronised in between: wait for them on the HOST before the staging buffers are rewritten
        # (copy_stream.wait_stream below only orders the device side).  Caller-owned pinned inputs must likewise stay
        # untouched until the event of the handle returned for them has completed.
        prev = slot.get("copy_event")
        if prev is not None:
            prev.synchronize()
        # Of a [B,H,N+1,N+1] map with a CLS token the loss reads query row 0 only.  Pinned maps: one pitched DMA per layer
        # straight out of the caller's tensor (basd_copy_cls_rows_h2d) - no host-side work at all.  Pageable or oddly
        # strided maps: gather the rows into a pinned staging buffer first.
        host_attn, dma_attn = {}, {}
        for j, a in all_teacher_attns.items():
            if has_cls and a.dim() == 4 and a.shape[2] > 1 and a.is_pinned() and a.stride(3) == 1 and a.dtype in (torch.float32, torch.bfloat16):
                dma_attn[j] = a
            elif has_cls and a.dim() == 4 and a.shape[2] > 1:
                rows = self._pinned(slot, ("pin_attn", j), a, (a.shape[0], a.shape[1], 1, a.shape[3]))
                rows.copy_(a[:, :, 0:1, :])
                host_attn[j] = rows
            else:
                host_attn[j] = a
        nbytes = 0
        self.copy_stream.wait_stream(torch.cuda.current_stream(self.device))     # the slot's previous consumer has been queued
        with torch.cuda.stream(self.copy_stream):
            def put(key, t):
                nonlocal nbytes
                d = self._dev(slot, key, t)
                d.copy_(t, non_blocking=True)
                nbytes += t.numel() * t.element_size()
                return d
            d_logits = put("logits", student_output)
            d_targets = put("targets", targets)
            d_student = {l: put(("s", l), t) for l, t in student_intermediates.items()}
            d_teacher = {j: put(("t", j), t) for j, t in all_teacher_tokens.items()}
            d_attn = {j: put(("a", j), t) for j, t in host_attn.items()}
            lib = _lib.load()
            for j, a in dma_attn.items():
                B_, H_, S_ = a.shape[0], a.shape[1], a.shape[3]
                d = self._dev(slot, ("a", j), a, (B_, H_, 1, S_))
                strides = (ctypes.c_int64 * 4)(*a.stride())
                _lib.check(lib.basd_copy_cls_rows_h2d(a.data_ptr(), a.element_size(), B_, H_, S_, strides, d.data_ptr(),
                                                      self.copy_stream.cuda_stream), "basd_copy_cls_rows_h2d")
                nbytes += B_ * H_ * S_ * a.element_size()
                d_attn[j] = d
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        slot["copy_event"] = ev
        self.h2d_bytes_last = nbytes
        return dict(event=ev, logits=d_logits, targets=d_targets, student=d_student, teacher=d_teacher, attn=d_attn)

    def run(self, handle):
        torch.cuda.current_stream(self.device).wait_event(handle["event"])
        logits = handle["logits"].detach().requires_grad_(handle["logits"].is_floating_point())
        student = {l: t.detach().requires_grad_() for l, t in handle["student"].items()}
        handle["leaf_logits"], handle["leaf_student"] = logits, student
        return self.module(logits, handle["targets"], student, handle["teacher"], handle["attn"])


# --------------------------------------------------------------------------------------------- teacher attention capture
def cls_attention_rows(q: torch.Tensor, k: torch.Tensor, scale: float | None = None) -> torch.Tensor:
    """CLS query row of softmax(q k^T * scale), shape [B, H, 1, S] fp32, straight from q and k [B, H, S, dh] (strided views
    of a fused qkv tensor are fine).  What the reference's attention hook (src/models/teacher.py:27-39) materialises as a
    full [B, H, S, S] map per block only for relational.py:24 to read row 0; pass the result as `all_teacher_attns[j]`."""
    lib = _lib.load()
    if q.device.type != "cuda" or k.device.type != "cuda":
        raise _lib.BasdError("cls_attention_rows: CUDA tensors required (no CPU fallback)")
    if q.dtype != k.dtype or q.dtype not in (torch.float32, torch.bfloat16):
        q, k = q.float(), k.float()
    if q.stride(3) != 1:
        q = q.contiguous()
    if k.stride(3) != 1:
        k = k.contiguous()
    B, H, S, dh = q.shape
    if scale is None:
        scale = dh ** -0.5
    if k.device != q.device or tuple(k.shape) != (B, H, S, dh):
        raise _lib.BasdError(f"cls_attention_rows: q {tuple(q.shape)} on {q.device} and k {tuple(k.shape)} on {k.device} do not match")
    with torch.cuda.device(q.device):
        out = torch.empty(B, H, 1, S, dtype=torch.float32, device=q.device)
        qs = (ctypes.c_int64 * 4)(*q.stride())
        ks = (ctypes.c_int64 * 4)(*k.stride())
        _lib.check(lib.basd_cls_attention_rows(q.data_ptr(), k.data_ptr(), _dtype_code(q), B, H, S, dh, qs, ks, float(scale), out.data_ptr(),
                                               _stream_ptr(q.device)), "basd_cls_attention_rows")
    return out


def query_mean_attention(q: torch.Tensor, k: torch.Tensor, scale: float | None = None) -> torch.Tensor:
    """Query mean of every head's softmax(q k^T * scale), shape [B, H, 1, S] fp32, straight from q and k [B, H, S, dh] (strided
    views of a fused qkv tensor are fine; dh a multiple of 8 up to 256, S up to 2048).  For teachers WITHOUT a CLS token
    relational.py:27 reads the attention only as attn.mean over heads and queries: pass the result as `all_teacher_attns[j]`
    (with teacher_has_cls_token=False) instead of the full [B, H, S, S] map the reference hook (src/models/teacher.py:27-39)
    materialises.  The kernel never stores an S x S map; fp32 inputs run as split-bf16 products (fp32-class accuracy)."""
    if q.dim() != 4 or tuple(k.shape) != tuple(q.shape):
        raise _lib.BasdError(f"query_mean_attention: q {tuple(q.shape)} and k {tuple(k.shape)} must both be [B, H, S, dh]")
    lib = _lib.load()
    if q.device.type != "cuda" or k.device.type != "cuda":
        raise _lib.BasdError("query_mean_attention: CUDA tensors required (no CPU fallback)")
    if k.device != q.device:
        raise _lib.BasdError(f"query_mean_attention: q on {q.device} and k on {k.device}")
    if q.dtype != k.dtype or q.dtype not in (torch.float32, torch.bfloat16):
        q, k = q.float(), k.float()
    B, H, S, dh = q.shape

    def aligned(t):             # read in place: d stride 1, 16-byte aligned base and (b, h, s) strides
        e = 8 if t.dtype == torch.bfloat16 else 4
        return t.stride(3) == 1 and t.data_ptr() % 16 == 0 and all(t.stride(i) % e == 0 or t.shape[i] == 1 for i in range(3))
    if not aligned(q):
        q = q.contiguous()
    if not aligned(k):
        k = k.contiguous()
    if scale is None:
        scale = dh ** -0.5
    with torch.cuda.device(q.device):
        out = torch.empty(B, H, 1, S, dtype=torch.float32, device=q.device)
        qs = (ctypes.c_int64 * 4)(*q.stride())
        ks = (ctypes.c_int64 * 4)(*k.stride())
        _lib.check(lib.basd_query_mean_attention(q.data_ptr(), k.data_ptr(), _dtype_code(q), B, H, S, dh, qs, ks, float(scale), out.data_ptr(),
                                                 _stream_ptr(q.device)), "basd_query_mean_attention")
    return out


# --------------------------------------------------------------------------------------------- reference API
def marchenko_pastur_rank(features: torch.Tensor) -> int:
    """layer_selector.py:8-20 on the GPU (tcgen05 Gram + one-sided Jacobi).  features: [M, D], D a multiple of 8 up to 4096
    (the second consumer, teacher.py:177, passes unprojected D_t-wide teacher features)."""
    lib = _lib.load()
    if features.device.type != "cuda":
        raise _lib.BasdError("marchenko_pastur_rank: CUDA tensor required (no CPU fallback)")
    if features.dtype not in (torch.float32, torch.bfloat16):
        features = features.float()
    if features.stride(1) != 1:
        features = features.contiguous()
    M, D = features.shape
    nb = ctypes.c_size_t()
    _lib.check(lib.basd_mp_rank_workspace_bytes(M, D, ctypes.byref(nb)), "basd_mp_rank_workspace_bytes")
    with torch.cuda.device(features.device):
        ws = torch.empty(nb.value, dtype=torch.uint8, device=features.device)
        out = torch.zeros(1, dtype=torch.int32, device=features.device)
        _lib.check(lib.basd_mp_rank(features.data_ptr(), M, D, _dtype_code(features), features.stride(0), out.data_ptr(), ws.data_ptr(),
                                    _stream_ptr(features.device)), "basd_mp_rank")
    return int(out.item())


# --------------------------------------------------------------------------------------------- standalone pieces of the path
@torch.library.custom_op("basd_b200::align_tokens", mutates_args=())
def _align_tokens_op(tokens: torch.Tensor, target_n: int) -> torch.Tensor:
    lib = _lib.load()
    if tokens.device.type != "cuda":
        raise _lib.BasdError("align_token_count: CUDA tensor required (no CPU fallback)")
    if tokens.dtype not in (torch.float32, torch.bfloat16):
        tokens = tokens.float()
    B, n_in, D = tokens.shape
    with torch.cuda.device(tokens.device):
        out = torch.empty(B, target_n, D, dtype=tokens.dtype, device=tokens.device)
        strides = (ctypes.c_int64 * 3)(*tokens.stride())
        _lib.check(lib.basd_align_tokens(tokens.data_ptr(), _dtype_code(tokens), strides, B, n_in, target_n, D, out.data_ptr(),
                                         _stream_ptr(tokens.device)), "basd_align_tokens")
    return out


@_align_tokens_op.register_fake
def _(tokens, target_n):
    return tokens.new_empty(tokens.shape[0], target_n, tokens.shape[2])


@torch.library.custom_op("basd_b200::align_tokens_bwd", mutates_args=())
def _align_tokens_bwd_op(grad_out: torch.Tensor, n_in: int) -> torch.Tensor:
    lib = _lib.load()
    g = grad_out.contiguous()
    if g.dtype not in (torch.float32, torch.bfloat16):
        g = g.float()
    B, n_out, D = g.shape
    with torch.cuda.device(g.device):
        gin = torch.empty(B, n_in, D, dtype=g.dtype, device=g.device)
        _lib.check(lib.basd_align_tokens_bwd(g.data_ptr(), _dtype_code(g), B, n_in, n_out, D, gin.data_ptr(), _stream_ptr(g.device)),
                   "basd_align_tokens_bwd")
    return gin


@_align_tokens_bwd_op.register_fake
def _(grad_out, n_in):
    return grad_out.new_empty(grad_out.shape[0], n_in, grad_out.shape[2])


def _align_setup(ctx, inputs, output):
    ctx.n_in = inputs[0].shape[1]
    ctx.in_dtype = inputs[0].dtype


def _align_backward(ctx, grad_out):
    return _align_tokens_bwd_op(grad_out, ctx.n_in).to(ctx.in_dtype), None


_align_tokens_op.register_autograd(_align_backward, setup_context=_align_setup)


def align_token_count(tokens: torch.Tensor, target_n: int) -> torch.Tensor:
    """combined.py:9-14: the same object when the token counts agree, else 1-D linear resampling along the flattened token
    axis (align_corners=False), differentiable.  [B, N, D] -> [B, target_n, D]."""
    if tokens.shape[1] == target_n:
        return tokens
    return _align_tokens_op(tokens, int(target_n))


_align_token_count = align_token_count      # the reference's (private) name


def geometric_relational_loss(student_tokens: torch.Tensor, teacher_tokens: torch.Tensor, teacher_attn: torch.Tensor, *,
                              has_cls_token: bool, polar_steps: int = 0, token_precision: str = "bf16") -> torch.Tensor:
    """relational.py:5-50 on its own: attention-weighted Procrustes loss of ONE student / teacher pair (teacher tokens already
    on the student's token grid, like combined.py:63-67 hands them over), mean over the batch.  Runs the same kernels as the
    fused loss with the layer selector bypassed (basd_shape.mode = BASD_MODE_PAIR).  The gradient flows to the student tokens;
    teacher tokens and attention are constants here, as everywhere on this path (teacher.py:123-124,180).
    token_precision "fp32": fp32 tokens are carried as split-bf16 pairs instead of being rounded to bf16 (TOKEN_PRECISIONS)."""
    _check_token_precision(token_precision)
    if student_tokens.device.type != "cuda":
        raise _lib.BasdError("geometric_relational_loss: CUDA tensors required (no CPU fallback)")
    B, n_s, _ = student_tokens.shape
    if teacher_tokens.shape[0] != B or teacher_tokens.shape[1] != n_s:
        raise _lib.BasdError(f"teacher tokens {tuple(teacher_tokens.shape)} must be aligned to the student's {n_s} tokens "
                             "(combined.py:63-67: _align_token_count first)")
    n_a = teacher_attn.shape[-1] - (1 if has_cls_token else 0)
    if n_a != n_s:
        # importance on the attention's own token grid, resampled to the student's (relational.py:22-32) and handed on as the
        # CLS row of a one-head map - the path normalises it (relational.py:34)
        imp = teacher_attn[:, :, 0, 1:].float().mean(dim=1) if has_cls_token else teacher_attn.float().mean(dim=(1, 2))
        imp = align_token_count(imp.unsqueeze(-1).contiguous(), n_s).squeeze(-1)
        if has_cls_token:
            teacher_attn = torch.cat([imp.new_zeros(B, 1), imp], dim=1).view(B, 1, 1, n_s + 1)
        else:
            teacher_attn = imp.view(B, 1, 1, n_s).expand(B, 1, n_s, n_s)
    dev = student_tokens.device
    none = torch.empty(0, device=dev)
    out = geo_forward([student_tokens], [teacher_tokens.detach()], [teacher_attn.detach()], none, none, torch.zeros(1, device=dev),
                      bool(has_cls_token), int(polar_steps), MODE_PAIR, token_precision)
    return out[0]


class GrassmannianLayerSelector(nn.Module):
    """Same constructor, buffers (`proj_s`, `proj_t`) and parameter (`log_temperatures`) as layer_selector.py:40-63.
    Inside BASDLoss the selector runs fused with the Procrustes term; `forward` is the reference's standalone entry point."""

    def __init__(self, num_extraction_points: int, student_dim: int, teacher_dim: int):
        super().__init__()
        self.student_dim = student_dim
        self._ranks_dev = None
        self._rank_keys: list[int] = []
        self.last_mixing_weights = None
        proj_s = torch.empty(student_dim, student_dim)
        proj_t = torch.empty(student_dim, teacher_dim)
        nn.init.orthogonal_(proj_s)
        nn.init.orthogonal_(proj_t)
        self.register_buffer("proj_s", proj_s)
        self.register_buffer("proj_t", proj_t)
        self.log_temperatures = nn.Parameter(torch.full((num_extraction_points,), math.log(math.exp(1.0) - 1)))
        # "bf16" (default): fp32 tokens are rounded to bf16 on entry; "fp32": carried as split-bf16 pairs (TOKEN_PRECISIONS)
        self.token_precision = "bf16"

    @property
    def temperatures(self) -> torch.Tensor:
        return F.softplus(self.log_temperatures)

    @property
    def subspace_ranks(self) -> dict:
        """layer_selector.py:49,74 — ranks of the last forward.  Kept on the device; reading this syncs once."""
        if self._ranks_dev is None:
            return {}
        return dict(zip(self._rank_keys, self._ranks_dev.tolist()))


    def mixing_weights(self, students: Sequence[torch.Tensor], teachers: Sequence[torch.Tensor], teacher_keys=None) -> torch.Tensor:
        """softmax(-d_Grassmann^2 / tau) of layer_selector.py:86-108 for every (student extraction point, teacher layer):
        [P, Lt] fp32, differentiable w.r.t. the student tokens and log_temperatures (closed-form backward, SURVEY.md B.3-B.5;
        basd_shape.mode = BASD_MODE_SELECTOR).  Updates `subspace_ranks` like layer_selector.py:74."""
        out = geo_forward(list(students), list(teachers), [], self.proj_s, self.proj_t, self.log_temperatures, True, 0, MODE_SELECTOR,
                          _check_token_precision(self.token_precision))
        self._ranks_dev = out[2]
        self._rank_keys = list(teacher_keys) if teacher_keys is not None else list(range(len(teachers)))
        self.last_mixing_weights = out[3].detach()
        return out[3]

    def forward(self, student_tokens_per_layer: dict, all_teacher_tokens: dict, all_teacher_attns: dict, extraction_indices: list):
        """layer_selector.py:116-152: (mixed_teachers, mixed_attentions), both keyed by student layer.  The spectral work (ranks,
        subspaces, principal angles, weights) runs in the CUDA kernels; the two weighted sums are the reference's own tensor
        expressions (:110-112) - BASDLoss never materialises the mixed attention maps, this standalone entry point has to."""
        t_idx = sorted(all_teacher_tokens.keys())
        teachers = [all_teacher_tokens[j] for j in t_idx]
        w = self.mixing_weights([student_tokens_per_layer[l] for l in extraction_indices], teachers, t_idx)
        stacked_tokens = torch.stack(teachers)
        stacked_attns = torch.stack([all_teacher_attns[j] for j in t_idx])
        mixed_teachers, mixed_attentions = {}, {}
        for i, s_layer in enumerate(extraction_indices):
            wi = w[i].to(stacked_tokens.dtype)
            mixed_teachers[s_layer] = (wi.view(-1, 1, 1, 1) * stacked_tokens).sum(dim=0)
            mixed_attentions[s_layer] = (wi.view(-1, 1, 1, 1, 1).to(stacked_attns.dtype) * stacked_attns).sum(dim=0)
        return mixed_teachers, mixed_attentions


class _UwsoCombine(torch.autograd.Function):
    """UW-SO weighting (combined.py:78-85; Kirchdorfer et al. 2024): total = sum_i w_i L_i with w_i = (1/L_i) / sum_j (1/L_j) taken
    on the detached values - one kernel (basd_uwso_combine) instead of a dozen scalar torch ops; the backward scales the incoming
    gradient by the saved weights."""

    @staticmethod
    def forward(ctx, ce, geo, det_ce, det_geo):
        lib = _lib.load()
        with torch.cuda.device(ce.device):
            out = torch.empty(3, dtype=torch.float32, device=ce.device)
            ce_c, geo_c, dce, dgeo = ce.contiguous(), geo.contiguous(), det_ce.contiguous(), det_geo.contiguous()
            _lib.check(lib.basd_uwso_combine(ce_c.data_ptr(), geo_c.data_ptr(), dce.data_ptr(), dgeo.data_ptr(),
                                             float(torch.finfo(torch.float32).eps), out.data_ptr(), _stream_ptr(ce.device)), "basd_uwso_combine")
        ctx.save_for_backward(out)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        gw = g * out[1:]                   # one launch: [g w_ce, g w_geo]
        return gw[0], gw[1], None, None


class BASDLoss(nn.Module):
    """Drop-in for combined.py:17-85 (same constructor and forward signature, `token_layers`, state_dict keys)."""

    def __init__(self, base_criterion: nn.Module, student_dim: int, teacher_dim: int, student_depth: int,
                 num_student_tokens: int, *, config, teacher_has_cls_token: bool):
        super().__init__()
        self.base_criterion = base_criterion
        self.teacher_has_cls_token = teacher_has_cls_token
        self.num_student_tokens = num_student_tokens
        if config.num_extraction_points == 1:
            self.token_layers = [student_depth - 1]
        else:
            self.token_layers = [round(i * (student_depth - 1) / (config.num_extraction_points - 1))
                                 for i in range(config.num_extraction_points)]
        self.layer_selector = GrassmannianLayerSelector(num_extraction_points=len(self.token_layers),
                                                        student_dim=student_dim, teacher_dim=teacher_dim)
        self.last_geo_loss = None
        self.last_ce_loss = None
        # Newton-Schulz steps of the Procrustes polar iteration: 0 = the library default (10 steps: singular values of the
        # cross-covariance down to 3e-5 ||C||_F converge).  Every forward leaves the largest residual ||X X^T - I||_F it saw
        # going into its last step in `last_polar_residual` (device tensor, no sync).  It is read back asynchronously and
        # looked at by the NEXT forward: above POLAR_RESIDUAL_OK (an ill-conditioned cross-covariance) the step count goes
        # up by one (to at most 16) with a warning - one step late, never a host sync in the step.
        self.polar_steps = 0
        # How fp32 student / teacher tokens are read: "bf16" (default) rounds them to bf16 on entry, "fp32" carries them as
        # split-bf16 pairs hi + lo through every kernel (fp32-class accuracy for more bytes and MMAs; DESIGN.md section 8).
        # bf16 tokens read the same either way.  HostStager follows the module it feeds.
        self.token_precision = "bf16"
        self.last_polar_residual = None
        self._resid_host = None
        self._resid_event = None

    def geo_loss(self, student_intermediates, all_teacher_tokens, all_teacher_attns) -> torch.Tensor:
        sel = self.layer_selector
        t_idx = sorted(all_teacher_tokens.keys())
        students = [student_intermediates[l] for l in self.token_layers]
        if students[0].shape[1] != self.num_student_tokens:
            raise _lib.BasdError(f"student tensors carry {students[0].shape[1]} tokens, module was built for {self.num_student_tokens}")
        teachers = [all_teacher_tokens[j] for j in t_idx]
        attns = [all_teacher_attns[j] for j in t_idx]
        # Student-feature form of the polar iteration (D_s <= min(N_s, N_t) - 1) with a teacher token Gram that is rank deficient
        # BY CONSTRUCTION - a coarser teacher grid up-sampled to the student's (N_t < N_s), or a teacher narrower than the token
        # count (D_t < N_s - 1): the components of the iterate in the null space of that Gram are invisible to the iteration, grow
        # with every step and come back through rounding, so MORE steps make the result worse (DESIGN.md section 8) and the
        # residual stays large whatever the step count.  Such shapes run with the default schedule, never escalate, and say so.
        ns, nt, ds, dt = students[0].shape[1], teachers[0].shape[1], students[0].shape[2], teachers[0].shape[2]
        self._kt_deficient = ds <= min(ns, nt) - 1 and (nt < ns or dt < ns - 1)
        self._poll_polar_residual()
        geo, _ws, ranks, w, resid = geo_forward(students, teachers, attns, sel.proj_s, sel.proj_t, sel.log_temperatures,
                                                bool(self.teacher_has_cls_token), int(self.polar_steps), MODE_LOSS,
                                                _check_token_precision(self.token_precision))
        sel._ranks_dev, sel._rank_keys = ranks, t_idx
        sel.last_mixing_weights = w
        resid = resid.detach()
        self.last_polar_residual = resid
        if self._resid_event is None and resid.device.type == "cuda":      # (the previous read-back has been consumed)
            if self._resid_host is None:
                self._resid_host = torch.empty(1, dtype=torch.float32, pin_memory=True)
            self._resid_host.copy_(resid, non_blocking=True)
            self._resid_event = torch.cuda.Event()
            self._resid_event.record(torch.cuda.current_stream(resid.device))
        return geo

    POLAR_RESIDUAL_OK = 0.1        # every |sigma^2 - 1| <= 0.1 going into the last step => every sigma within 1e-3 of 1 after it
    POLAR_STEPS_MAX = 16

    def _poll_polar_residual(self):
        ev = self._resid_event
        if ev is None or not ev.query():
            return
        self._resid_event = None
        val = float(self._resid_host[0])
        if not val <= self.POLAR_RESIDUAL_OK and getattr(self, "_kt_deficient", False):
            if not getattr(self, "_kt_warned", False):
                self._kt_warned = True
                import warnings
                warnings.warn(f"BASD Procrustes polar iteration: residual {val:.3g} with a teacher token Gram that is rank deficient by construction "
                              "(teacher grid coarser than the student's, or teacher width below the token count): the step count is NOT raised "
                              "(more steps amplify the null-space components); student-gradient accuracy on such shapes is 2e-3 .. 1e-1 "
                              "(DESIGN.md section 8)", RuntimeWarning)
            return
        if not val <= self.POLAR_RESIDUAL_OK:                               # (NaN counts as not converged)
            cur = self.polar_steps if self.polar_steps else 10
            if cur < self.POLAR_STEPS_MAX:
                # one step at a time: every step beyond convergence multiplies the rounding noise of the early steps in the weak
                # singular directions (measured on near-square cross-covariances: student-gradient error 6e-3 at 10 steps, 1.2e-2 at
                # 11 - where the residual converges - and 1.2e-1 at 14; tools/scratch/near_square.py)
                self.polar_steps = min(cur + 1, self.POLAR_STEPS_MAX)
                import warnings
                warnings.warn(f"BASD Procrustes polar iteration: residual {val:.3g} > {self.POLAR_RESIDUAL_OK} after {cur} Newton-Schulz steps "
                              f"(ill-conditioned teacher-student cross-covariance); using {self.polar_steps} steps from now on", RuntimeWarning)
            else:
                import warnings
                warnings.warn(f"BASD Procrustes polar iteration: residual {val:.3g} after {cur} steps - the cross-covariance has singular values "
                              "below fp32/split-bf16 resolution; their directions carry unconverged gradient weight", RuntimeWarning)

    def forward(self, student_output, targets, student_intermediates, all_teacher_tokens, all_teacher_attns):
        _check_token_precision(self.token_precision)
        ce_loss = self.base_criterion(student_output, targets)
        geo_loss = self.geo_loss(student_intermediates, all_teacher_tokens, all_teacher_attns)
        self.last_geo_loss, self.last_ce_loss = geo_loss.detach(), ce_loss.detach()
        vals = [ce_loss, geo_loss.to(ce_loss.dtype) if ce_loss.dtype != geo_loss.dtype else geo_loss]
        det = [v.detach() for v in vals]
        dist, world = _world()
        if dist is not None:               # UW-SO weights from the global means (single-process semantics)
            pair = torch.stack([d.float() for d in det])
            dist.all_reduce(pair, op=dist.ReduceOp.SUM)
            det = [(pair[i] / world).to(vals[i].dtype) for i in range(2)]
        if all(v.dtype == torch.float32 and v.device.type == "cuda" and v.dim() == 0 for v in vals):
            return _UwsoCombine.apply(vals[0], vals[1], det[0], det[1])      # combined.py:78-85 in one launch (+ one in the backward)
        eps = torch.finfo(vals[0].dtype).eps                                 # other dtypes / criteria with reduction='none': the reference's expression
        inv = torch.stack([1.0 / d.clamp(min=eps) for d in det])
        wts = inv / inv.sum()
        return sum(wts[i] * vals[i] for i in range(len(vals)))
