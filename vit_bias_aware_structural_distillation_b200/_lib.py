"""ctypes binding of libbasd_b200.so (include/basd_b200.h).  There is NO CPU fallback: every compute entry point
needs the shared library and a CUDA device and raises otherwise."""
from __future__ import annotations

import ctypes
import os

MAX_POINTS = 8
MAX_LAYERS = 64
DTYPE_F32, DTYPE_BF16 = 0, 1
DTYPE_F32_SPLIT = 2             # basd_shape.act_dtype: fp32 tokens carried as split-bf16 pairs (token_precision="fp32")
MODE_LOSS, MODE_PAIR, MODE_SELECTOR = 0, 1, 2
ATTN_QUERY_MEAN = 2             # basd_shape.has_cls: no CLS token, attention given as query-mean rows [B,H,1,Nt]

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BASD_B200_LIB") or os.path.join(_HERE, "libbasd_b200.so")      # (override: A/B runs of two builds)


class Shape(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in
                ("B", "Ns", "Nt", "Ds", "Dt", "Lt", "P", "H", "has_cls", "act_dtype", "attn_dtype", "world_size", "polar_steps", "mode")]


class Inputs(ctypes.Structure):
    _fields_ = [
        ("student", ctypes.c_void_p * MAX_POINTS),
        ("teacher", ctypes.c_void_p * MAX_LAYERS),
        ("attn", ctypes.c_void_p * MAX_LAYERS),
        ("student_strides", ctypes.c_int64 * 3),
        ("teacher_strides", ctypes.c_int64 * 3),
        ("attn_strides", ctypes.c_int64 * 4),
        ("proj_s", ctypes.c_void_p),
        ("proj_t", ctypes.c_void_p),
        ("log_temperatures", ctypes.c_void_p),
    ]


EXPORTS = [
    "basd_workspace_bytes", "basd_forward_stats", "basd_forward_solve", "basd_backward_dots", "basd_backward_finish",
    "basd_view", "basd_mp_rank_workspace_bytes", "basd_mp_rank", "basd_selftest_gemm", "basd_selftest_eig",
    "basd_last_error", "basd_version", "basd_timing_enable", "basd_timing_reset", "basd_launch_count", "basd_timing_slots",
    "basd_timing_name", "basd_timing_read", "basd_polar_steps", "basd_polar_launches_per_step", "basd_cls_attention_rows",
    "basd_copy_cls_rows_h2d", "basd_align_tokens", "basd_align_tokens_bwd", "basd_uwso_combine", "basd_query_mean_attention",
]

_lib = None


class BasdError(RuntimeError):
    pass


def load():
    """Loads the shared library (built by __graft_entry__.build()).  Raises if it is missing — never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BasdError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a).  There is no CPU/PyTorch fallback for the BASD loss path.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz = ctypes.c_void_p, ctypes.c_size_t
    lib.basd_last_error.restype = ctypes.c_char_p
    lib.basd_version.restype = ctypes.c_char_p
    lib.basd_workspace_bytes.argtypes = [ctypes.POINTER(Shape), ctypes.POINTER(sz)]
    lib.basd_forward_stats.argtypes = [ctypes.POINTER(Shape), ctypes.POINTER(Inputs), vp, vp]
    lib.basd_forward_solve.argtypes = [ctypes.POINTER(Shape), ctypes.POINTER(Inputs), vp, vp, vp]
    lib.basd_backward_dots.argtypes = [ctypes.POINTER(Shape), ctypes.POINTER(Inputs), vp, vp]
    lib.basd_backward_finish.argtypes = [ctypes.POINTER(Shape), ctypes.POINTER(Inputs), vp, vp, ctypes.POINTER(vp), ctypes.c_int, vp, vp]
    lib.basd_view.argtypes = [ctypes.POINTER(Shape), vp, ctypes.c_char_p, ctypes.POINTER(vp), ctypes.POINTER(sz)]
    lib.basd_mp_rank_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int, ctypes.POINTER(sz)]
    lib.basd_mp_rank.argtypes = [vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int64, vp, vp, vp]
    lib.basd_selftest_gemm.argtypes = [ctypes.c_int, vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]
    lib.basd_selftest_eig.argtypes = [vp, ctypes.c_int, vp, vp, vp, vp, vp]
    lib.basd_cls_attention_rows.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64), ctypes.c_float, vp, vp]
    lib.basd_query_mean_attention.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64), ctypes.c_float, vp, vp]
    lib.basd_copy_cls_rows_h2d.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int64), vp, vp]
    lib.basd_align_tokens.argtypes = [vp, ctypes.c_int, ctypes.POINTER(ctypes.c_int64), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    lib.basd_align_tokens_bwd.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    lib.basd_uwso_combine.argtypes = [vp, vp, vp, vp, ctypes.c_float, vp, vp]
    lib.basd_launch_count.restype = ctypes.c_longlong
    lib.basd_timing_name.restype = ctypes.c_char_p
    lib.basd_timing_name.argtypes = [ctypes.c_int]
    lib.basd_timing_enable.argtypes = [ctypes.c_int]
    lib.basd_timing_read.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int)]
    for name in EXPORTS:
        getattr(lib, name)          # fail loudly on a stale library
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        raise BasdError(f"{what} failed: {load().basd_last_error().decode()}")


def timing_read():
    """{kernel group: (total ms, brackets)} recorded since the last basd_timing_reset()."""
    lib = load()
    out = {}
    for i in range(lib.basd_timing_slots()):
        ms, n = ctypes.c_float(), ctypes.c_int()
        check(lib.basd_timing_read(i, ctypes.byref(ms), ctypes.byref(n)), "basd_timing_read")
        out[lib.basd_timing_name(i).decode()] = (ms.value, n.value)
    return out
