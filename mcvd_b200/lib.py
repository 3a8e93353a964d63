"""ctypes binding of the C-ABI library (``include/mcvd_b200.h``).

The product path has no CPU or PyTorch fallback: if the library cannot be loaded (or built), or a
launch fails, a ``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

# ---- op kinds / flags (mirror of include/mcvd_b200.h) -------------------------------------------
OP_NCHW_TO_NHWC = 1
OP_NHWC_TO_NCHW = 2
OP_TIMESTEP_EMBED = 3
OP_LINEAR = 4
OP_GN_PARTIAL = 5
OP_GN_FINALIZE = 6
OP_APPLY = 7
OP_CONV_SIMT = 8
OP_ATTENTION = 9
OP_RESIZE_NEAREST = 10
OP_DIFFUSION_UPDATE = 11
OP_CONV_UMMA = 12
OP_CONV_SMALLN = 13
OP_COPY = 14
OP_ATTENTION_UMMA = 15
OP_CONV_UMMA2 = 16
OP_FRAME_METRICS = 17

F_ACT_IN = 1 << 0
F_ACT_OUT = 1 << 1
F_UP = 1 << 2
F_DOWN = 1 << 3
F_FILM = 1 << 4
F_CLIP = 1 << 5
F_PHILOX = 1 << 6
F_ROUND = 1 << 7
F_GAMMA = 1 << 8
F_NOISE = 1 << 9

ABI_VERSION = 5

EXPORTS = ["mcvd_abi_version", "mcvd_sizeof_op", "mcvd_last_error", "mcvd_device_arch", "mcvd_run_program",
           "mcvd_validate_program", "mcvd_count_launches", "mcvd_umma_pack_weights", "mcvd_umma_kblock",
           "mcvd_attention_scratch_bytes", "mcvd_umma2_plan", "mcvd_umma2_plan_info", "mcvd_umma2_stats_bytes", "mcvd_umma2_pack_weights"]


class McvdOp(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("flags", C.c_int32),
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("C0", C.c_int32), ("C1", C.c_int32), ("Cout", C.c_int32),
        ("i0", C.c_int32), ("i1", C.c_int32), ("i2", C.c_int32), ("i3", C.c_int32),
        ("f0", C.c_float), ("f1", C.c_float), ("f2", C.c_float), ("f3", C.c_float),
        ("f4", C.c_float), ("f5", C.c_float), ("f6", C.c_float), ("f7", C.c_float),
        ("src0", C.c_void_p), ("src1", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p),
        ("aux0", C.c_void_p), ("aux1", C.c_void_p), ("aux2", C.c_void_p),
        ("dst", C.c_void_p), ("dst2", C.c_void_p),
        ("src2", C.c_void_p), ("src3", C.c_void_p), ("C2", C.c_int32), ("C3", C.c_int32),
        ("i4", C.c_int32), ("i5", C.c_int32), ("i6", C.c_int32), ("i7", C.c_int32),
    ]


_lock = threading.Lock()
_lib = None


def library_path() -> str:
    return _build.LIB


def load():
    """Load (building first if the in-tree .so is missing or stale and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB
        if _build.needs_build():
            try:
                nvcc = _build._nvcc()
            except RuntimeError as e:       # no compiler on this box: the prebuilt library (if any) is all there is
                nvcc = None
                if not os.path.exists(path):
                    raise RuntimeError(f"mcvd_b200: CUDA library missing and cannot be built: {e}") from e
                import warnings
                warnings.warn("mcvd_b200: sources are newer than the prebuilt library and nvcc is not available; "
                              "using the prebuilt library")
            if nvcc is not None:
                # a compiler exists and the library is stale: a failed rebuild must not silently fall back to it
                _build.build()
        if not os.path.exists(path):
            raise RuntimeError(f"mcvd_b200: CUDA library not found at {path}")
        lib = C.CDLL(path)
        lib.mcvd_abi_version.restype = C.c_int
        lib.mcvd_sizeof_op.restype = C.c_int
        lib.mcvd_last_error.restype = C.c_char_p
        lib.mcvd_device_arch.restype = C.c_int
        lib.mcvd_run_program.restype = C.c_int
        lib.mcvd_run_program.argtypes = [C.POINTER(McvdOp), C.c_int, C.c_void_p]
        lib.mcvd_validate_program.restype = C.c_int
        lib.mcvd_validate_program.argtypes = [C.POINTER(McvdOp), C.c_int]
        lib.mcvd_count_launches.restype = C.c_int
        lib.mcvd_count_launches.argtypes = [C.POINTER(McvdOp), C.c_int]
        lib.mcvd_umma_pack_weights.restype = C.c_longlong
        lib.mcvd_umma_pack_weights.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                               C.c_int, C.c_void_p]
        lib.mcvd_umma_kblock.restype = C.c_int
        lib.mcvd_umma_kblock.argtypes = [C.c_int, C.c_int]
        lib.mcvd_attention_scratch_bytes.restype = C.c_longlong
        lib.mcvd_attention_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
        lib.mcvd_umma2_plan.restype = C.c_int
        lib.mcvd_umma2_plan.argtypes = [C.c_int] * 9
        lib.mcvd_umma2_plan_info.restype = C.c_int
        lib.mcvd_umma2_plan_info.argtypes = [C.c_int] * 9 + [C.POINTER(C.c_int)]
        lib.mcvd_umma2_stats_bytes.restype = C.c_longlong
        lib.mcvd_umma2_stats_bytes.argtypes = [C.c_int] * 5
        lib.mcvd_umma2_pack_weights.restype = C.c_longlong
        lib.mcvd_umma2_pack_weights.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                C.c_int, C.c_int, C.c_int, C.c_void_p]
        if lib.mcvd_abi_version() != ABI_VERSION:
            raise RuntimeError("mcvd_b200: ABI version mismatch between the Python binding and the library")
        if lib.mcvd_sizeof_op() != C.sizeof(McvdOp):
            raise RuntimeError(f"mcvd_b200: McvdOp layout mismatch ({lib.mcvd_sizeof_op()} vs {C.sizeof(McvdOp)})")
        _lib = lib
        return lib


def last_error() -> str:
    return load().mcvd_last_error().decode("utf-8", "replace")


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"mcvd_b200 {what} failed ({rc}): {last_error()}")


def make_ops(ops):
    arr = (McvdOp * len(ops))(*ops)
    return arr


def run_program(arr, n, stream_ptr: int):
    check(load().mcvd_run_program(arr, n, C.c_void_p(stream_ptr)), "run_program")


def validate_program(arr, n):
    check(load().mcvd_validate_program(arr, n), "validate_program")


def umma_kblock(c0: int, c1: int) -> int:
    return int(load().mcvd_umma_kblock(c0, c1))


def attention_scratch_bytes(B: int, T: int, C: int) -> int:
    """bytes of ``dst2`` scratch an OP_ATTENTION_UMMA op needs (fp16 hi/lo operand images of q, k, v)"""
    return int(load().mcvd_attention_scratch_bytes(B, T, C))


def umma2_plan(H: int, W: int, ks: int, c0: int, c1: int, c2: int, c3: int, n_tile: int, stats: bool) -> int:
    """channels per K-block (32 | 16 | 0 = not runnable) of an OP_CONV_UMMA2 op; host arithmetic only"""
    return int(load().mcvd_umma2_plan(H, W, ks, c0, c1, c2, c3, n_tile, 1 if stats else 0))


def umma2_stats_bytes(B: int, H: int, W: int, ks: int, cout: int) -> int:
    return int(load().mcvd_umma2_stats_bytes(B, H, W, ks, cout))


def umma2_plan_info(H, W, ks, c0, c1, c2, c3, n_tile, stats):
    """dict of the shared-memory plan (K-block, slab rows, ring depths, bytes) or None"""
    out = (C.c_int * 10)()
    if load().mcvd_umma2_plan_info(H, W, ks, c0, c1, c2, c3, n_tile, 1 if stats else 0, out) != 0:
        return None
    return dict(zip(("kb", "hp", "sa", "r", "nb", "nj", "tmem_cols", "smem", "j", "nsets"), list(out)))


def conv1x1_enabled() -> bool:
    """The input-stationary 1x1 kernel (csrc/conv1x1_umma.cu) is on unless MCVD_CONV1X1=0 (read by the library too)."""
    return os.environ.get("MCVD_CONV1X1", "1") != "0"


def umma2_pick_nt(cout: int, ks: int) -> int:
    """n tile of an OP_CONV_UMMA2 op: the largest multiple of 16 dividing Cout that is <= 128 for 3x3 convs (two or more
    position tiles then share every weight stage, TMEM holds two accumulator sets) and <= 256 for 1x1 convs (few
    weights; fewer n tiles mean fewer re-stagings of the input slab).  0 when Cout is not a multiple of 16."""
    cap = 128 if ks == 3 else 256
    best = 0
    for d in range(16, cap + 1, 16):
        if cout % d == 0:
            best = d
    return best
