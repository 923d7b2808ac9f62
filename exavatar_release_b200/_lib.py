"""ctypes binding of libb200raster.so (the C ABI in include/b200raster.h).

There is NO CPU fallback: if the shared library is missing or cannot be loaded, `load()` raises.  The library is built
in-tree by `exavatar_release_b200.build_ext.build()` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libb200raster.so")
LIB_PATH = os.environ.get("B2R_LIB", LIB_PATH)  # tuning experiments: an alternative build of the same library

ABI_VERSION = 3
B2R_OK = 0
B2R_FLAG_NO_TILE_CULL = 1
B2R_FLAG_DEBUG = 2
B2R_FLAG_CTX_CLEAN = 4

_fp = C.c_void_p  # device pointers travel as plain addresses


class B2RScene(C.Structure):
    _fields_ = [
        ("P", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("sh_degree", C.c_int32),
        ("sh_coeffs", C.c_int32), ("flags", C.c_uint32),
        ("scale_modifier", C.c_float), ("tanfovx", C.c_float), ("tanfovy", C.c_float),
        ("bg", _fp), ("viewmatrix", _fp), ("projmatrix", _fp), ("campos", _fp),
        ("means3D", _fp), ("shs", _fp), ("colors_precomp", _fp), ("opacities", _fp),
        ("scales", _fp), ("rotations", _fp), ("cov3D_precomp", _fp),
        # fused linear-blend skinning (SURVEY section 8f-2); all NULL / 0 = off
        ("skin_xyz", _fp), ("skin_weights", _fp), ("skin_joint_mats", _fp), ("skin_trans", _fp),
        ("skin_cam_Rinv", _fp), ("skin_cam_t", _fp), ("skin_means_out", _fp), ("skin_J", C.c_int32),
        ("sh_rows", C.c_int32),  # two colour sources: SH rows [0, sh_rows), colors_precomp for the rest
    ]


class B2RStatus(C.Structure):
    _fields_ = [
        ("num_dups", C.c_uint64), ("dup_capacity", C.c_uint64), ("overflow", C.c_uint32), ("num_visible", C.c_uint32),
        ("consumed_fwd", C.c_uint64), ("consumed_bwd", C.c_uint64), ("token", C.c_uint64), ("reserved", C.c_uint64 * 2),
    ]


class B2RWorkspace(C.Structure):
    _fields_ = [
        ("ctx", _fp), ("ctx_bytes", C.c_size_t), ("dup_ids", _fp), ("dup_capacity", C.c_uint64),
        ("scratch", _fp), ("scratch_bytes", C.c_size_t), ("status_mirror", _fp), ("status_token", C.c_uint64),
        ("checkpoints", _fp), ("checkpoint_bytes", C.c_size_t),  # ABI v3: segment table + blend-state checkpoints
    ]


class B2RView(C.Structure):
    _fields_ = [
        ("id_begin", C.c_uint32), ("id_end", C.c_uint32), ("bg", _fp), ("final_T", _fp), ("n_contrib", _fp),
        ("checkpoints", _fp), ("checkpoint_bytes", C.c_size_t), ("skip_below", C.c_uint32), ("reserved", C.c_uint32),
    ]


class B2RForwardOutputs(C.Structure):
    _fields_ = [("color", _fp), ("depth", _fp), ("alpha", _fp), ("radii", _fp)]


class B2RBackwardArgs(C.Structure):
    _fields_ = [
        ("dL_dcolor", _fp), ("dL_ddepth", _fp), ("dL_dalpha", _fp),
        ("dL_dmeans3D", _fp), ("dL_dmeans2D", _fp), ("dL_dshs", _fp), ("dL_dcolors", _fp), ("dL_dopacities", _fp),
        ("dL_dscales", _fp), ("dL_drotations", _fp), ("dL_dcov3D", _fp),
        ("flags", C.c_uint32), ("first_row", C.c_uint32),
        ("densify_grad_accum", _fp), ("densify_count", _fp), ("densify_radius_max", _fp),
        ("dL_dskin_xyz", _fp), ("dL_dskin_G", _fp),
        ("dL_dposed", _fp),  # ABI v3 INPUT: gradient arriving at the posed positions (fused skinning)
        ("densify_rows", C.c_uint32), ("reserved", C.c_uint32),
    ]


# B2RStatus.consumed_fwd / consumed_bwd: list entries staged per tile, x 8 (forward) / x 4 (backward) -- b200raster.h
CONSUMED_FWD_DIV = 8
CONSUMED_BWD_DIV = 4

B2R_BWD_ACCUMULATE = 1
B2R_BWD_SCRATCH_ZEROED = 2


def read_status(ctx_buf) -> dict:
    """The B2RStatus block at the head of a device ctx buffer (a uint8 tensor), copied back to the host (synchronises);
    for tests, bench accounting and overflow checks.  The composites count staged list entries per CTA; consumed_*_div
    turn those sums into entries per tile."""
    s = B2RStatus.from_buffer_copy(ctx_buf[: C.sizeof(B2RStatus)].cpu().numpy().tobytes())
    out = {name: int(getattr(s, name)) for name, _ in B2RStatus._fields_ if name != "reserved"}
    out.update(consumed_fwd_div=float(CONSUMED_FWD_DIV), consumed_bwd_div=float(CONSUMED_BWD_DIV))
    return out


# every symbol include/b200raster.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("b2r_abi_version", C.c_int, []),
    ("b2r_strerror", C.c_char_p, [C.c_int]),
    ("b2r_last_cuda_error", C.c_int, []),
    ("b2r_sizeof", C.c_size_t, [C.c_int]),
    ("b2r_ctx_bytes", C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    ("b2r_scratch_bytes", C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_uint64]),
    ("b2r_backward_scratch_bytes", C.c_size_t, [C.c_int32]),
    ("b2r_checkpoint_bytes", C.c_size_t, [C.c_int32, C.c_int32, C.c_uint64]),
    ("b2r_forward_bin", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), _fp]),
    ("b2r_forward_composite", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), C.POINTER(B2RView),
                                        C.POINTER(B2RForwardOutputs), _fp]),
    ("b2r_backward_composite", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), C.POINTER(B2RView),
                                         C.POINTER(B2RBackwardArgs), _fp, C.c_size_t, _fp]),
    ("b2r_backward_project", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), C.POINTER(B2RBackwardArgs), _fp,
                                       C.c_size_t, _fp]),
    ("b2r_forward_project", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), _fp, _fp]),
    ("b2r_forward_render", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), C.POINTER(B2RForwardOutputs), _fp]),
    ("b2r_forward", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), C.POINTER(B2RForwardOutputs), _fp]),
    ("b2r_backward", C.c_int, [C.POINTER(B2RScene), C.POINTER(B2RWorkspace), C.POINTER(B2RBackwardArgs), _fp,
                               C.c_size_t, _fp]),
    ("b2r_mark_visible", C.c_int, [C.c_int32, _fp, _fp, _fp, _fp]),
    ("b2r_profile_enable", None, [C.c_int]),
    ("b2r_profile_read", C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int]),
    ("b2r_launch_count", C.c_uint64, []),
    ("b2r_kernel_name", C.c_char_p, [C.c_int]),
    ("b2r_ctx_geom", _fp, [C.POINTER(B2RWorkspace), C.c_int32, C.c_int32, C.c_int32]),
    ("b2r_ctx_aux", _fp, [C.POINTER(B2RWorkspace), C.c_int32, C.c_int32, C.c_int32]),
    ("b2r_ctx_ranges", _fp, [C.POINTER(B2RWorkspace), C.c_int32, C.c_int32, C.c_int32]),
    ("b2r_ctx_final_T", _fp, [C.POINTER(B2RWorkspace), C.c_int32, C.c_int32, C.c_int32]),
    ("b2r_ctx_n_contrib", _fp, [C.POINTER(B2RWorkspace), C.c_int32, C.c_int32, C.c_int32]),
]

_lib = None


def load():
    """Loads the shared library (once).  Raises if it is absent -- the product path never falls back to CPU code."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"b200raster: {LIB_PATH} not found. Build it with `python -m exavatar_release_b200.build_ext` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.b2r_abi_version() != ABI_VERSION:
        raise RuntimeError("b200raster: ABI version mismatch between the Python binding and libb200raster.so")
    for idx, cls in enumerate((B2RScene, B2RStatus, B2RWorkspace, B2RForwardOutputs, B2RBackwardArgs, B2RView)):
        if lib.b2r_sizeof(idx) != C.sizeof(cls):
            raise RuntimeError(f"b200raster: struct layout drift for {cls.__name__}: "
                               f"{lib.b2r_sizeof(idx)} (C) vs {C.sizeof(cls)} (ctypes)")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != B2R_OK:
        lib = load()
        msg = lib.b2r_strerror(rc).decode()
        raise RuntimeError(f"b200raster: {what} failed: {msg} (code {rc}, cudaError {lib.b2r_last_cuda_error()})")
