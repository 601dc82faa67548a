"""ctypes binding of libdexr.so (the C ABI declared in include/dexr.h).

The library is built in-tree by `__graft_entry__.build()` / `python -m dex_retargeting_b200.build`
(nvcc, sm_100a).  There is NO fallback: if the shared object is missing or a call fails, this module
raises -- the product path never silently runs on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

MAX_LANES, MAX_LINKS, MAX_RES, MAX_GROUP, NUM_KEYPOINTS = 32, 16, 16, 4, 21
MAX_LINKS_PER_LANE = 4
LOSS_POSITION, LOSS_VECTOR, LOSS_DEXPILOT = 0, 1, 2
TABLE_MAGIC = 0x31525844

STATUS_MAXITER = 1 << 24
STATUS_NONFINITE = 1 << 25

_f, _i, _u = C.c_float, C.c_int32, C.c_uint32


class DexrTable(C.Structure):
    """Mirror of `dexr_table_t` (include/dexr.h) -- keep field order identical."""

    _fields_ = [
        ("magic", _u), ("nbytes", _u), ("dof", _i), ("n_var", _i), ("n_fixed", _i), ("n_links", _i),
        ("n_res", _i), ("loss", _i), ("n_rounds", _i), ("has_mimic", _i), ("num_fingers", _i),
        ("len_proj", _i), ("len_s1", _i), ("block_width", _i), ("arrow", _i), ("reserved", _i),
        ("R0", (_f * 9) * MAX_LANES), ("RA", (_f * 9) * MAX_LANES), ("RB", (_f * 9) * MAX_LANES),
        ("p0", (_f * 3) * MAX_LANES), ("d0", (_f * 3) * MAX_LANES), ("axis", (_f * 3) * MAX_LANES),
        ("jtype", _i * MAX_LANES), ("var_index", _i * MAX_LANES), ("fixed_index", _i * MAX_LANES),
        ("mimic_src", _i * MAX_LANES), ("mimic_mult", _f * MAX_LANES), ("mimic_off", _f * MAX_LANES),
        ("lower", _f * MAX_LANES), ("upper", _f * MAX_LANES), ("clip_lo", _f * MAX_LANES), ("clip_hi", _f * MAX_LANES),
        ("jump", _u * MAX_LANES), ("anc_mask", _u * MAX_LANES), ("desc_mask", _u * MAX_LANES),
        ("group_count", _i * MAX_LANES), ("group_lane", (_i * MAX_GROUP) * MAX_LANES),
        ("group_mult", (_f * MAX_GROUP) * MAX_LANES),
        ("link_parent", _i * MAX_LINKS), ("link_off", (_f * 3) * MAX_LINKS), ("link_anc_mask", _u * MAX_LINKS),
        ("res_task", _i * MAX_RES), ("res_origin", _i * MAX_RES), ("res_human_task", _i * MAX_RES),
        ("res_human_origin", _i * MAX_RES), ("s2_origin", _i * MAX_RES), ("s2_task", _i * MAX_RES),
    ]


class DexrParams(C.Structure):
    _fields_ = [
        ("huber_delta", _f), ("norm_delta", _f), ("scaling", _f), ("project_dist", _f), ("escape_dist", _f),
        ("eta1", _f), ("eta2", _f), ("lp_alpha", _f), ("tol", _f), ("lambda0", _f),
        ("max_iters", _i), ("clip_init", _i), ("preprocess", _i),
    ]


class DexrFrames(C.Structure):
    _fields_ = [
        ("keypoints", C.c_void_p), ("ref_value", C.c_void_p), ("fixed_qpos", C.c_void_p), ("last_qpos", C.c_void_p),
        ("projected", C.c_void_p), ("qpos_out", C.c_void_p), ("robot_qpos_out", C.c_void_p),
        ("status_out", C.c_void_p), ("cost_out", C.c_void_p), ("damping_io", C.c_void_p),
    ]


class DexrSequences(C.Structure):
    _fields_ = [
        ("keypoints", C.c_void_p), ("fixed_qpos", C.c_void_p), ("last_qpos", C.c_void_p), ("filter_state", C.c_void_p),
        ("filter_init", C.c_void_p), ("projected", C.c_void_p), ("robot_qpos_out", C.c_void_p), ("status_out", C.c_void_p),
        ("damping_state", C.c_void_p),
    ]


class DexrGroup(C.Structure):
    """Mirror of `dexr_group_t`: one (robot, batch) group of a mixed-robot launch."""

    _fields_ = [("robot", C.c_void_p), ("params", C.POINTER(DexrParams)), ("io", DexrFrames), ("num_frames", C.c_int64)]


MAX_GROUPS = 16


class DexrLaunchInfo(C.Structure):
    _fields_ = [("grid", _i), ("block", _i), ("smem_bytes", _i), ("frames_per_tile", _i), ("lanes_per_frame", _i),
                ("consumer_warps", _i), ("kernels_launched", _i)]


EXPORTS = [
    "dexr_version", "dexr_build_id", "dexr_last_error", "dexr_table_sizeof", "dexr_params_sizeof", "dexr_frames_sizeof",
    "dexr_sequences_sizeof", "dexr_default_params",
    "dexr_robot_create", "dexr_robot_create_from_device", "dexr_robot_device_table", "dexr_robot_destroy",
    "dexr_solve_frames", "dexr_solve_frames_multi", "dexr_solve_sequences", "dexr_solve_frames_host", "dexr_get_launch_info",
    "dexr_preprocess_keypoints",
]

_LIB = None
_GRAD = None

# The backward pass lives in a second library (include/dexr_grad.h); its exports are kept apart from EXPORTS, which mirrors dexr.h.
GRAD_EXPORTS = ["dexr_grad_version", "dexr_grad_build_id", "dexr_grad_last_error", "dexr_grad_frames_sizeof", "dexr_grad_frames",
                "dexr_grad_sequences_sizeof", "dexr_grad_sequences", "dexr_grad_lowpass"]

GRAD_STATUS_ACTIVE = 1 << 0
GRAD_STATUS_SHIFTED = 1 << 1
GRAD_STATUS_SINGULAR = 1 << 2
GRAD_STATUS_SKIPPED = 1 << 3
GRAD_STATUS_NONFINITE = 1 << 4


class DexrGradFrames(C.Structure):
    """Mirror of `dexr_grad_frames_t` (include/dexr_grad.h)."""

    _fields_ = [
        ("keypoints", C.c_void_p), ("ref_value", C.c_void_p), ("fixed_qpos", C.c_void_p), ("last_qpos", C.c_void_p),
        ("projected", C.c_void_p), ("qpos", C.c_void_p), ("status", C.c_void_p), ("grad_qpos", C.c_void_p),
        ("grad_keypoints", C.c_void_p), ("grad_ref_value", C.c_void_p), ("grad_last_qpos", C.c_void_p), ("grad_status", C.c_void_p),
    ]


class DexrGradSequences(C.Structure):
    """Mirror of `dexr_grad_sequences_t` (include/dexr_grad.h)."""

    _fields_ = [
        ("keypoints", C.c_void_p), ("fixed_qpos", C.c_void_p), ("last_qpos", C.c_void_p), ("projected", C.c_void_p),
        ("filter_init", C.c_void_p), ("qpos", C.c_void_p), ("status", C.c_void_p), ("grad_robot_qpos", C.c_void_p),
        ("grad_last_qpos_out", C.c_void_p), ("grad_filter_state_out", C.c_void_p), ("projected_ws", C.c_void_p),
        ("grad_keypoints", C.c_void_p), ("grad_last_qpos", C.c_void_p), ("grad_filter_state", C.c_void_p),
        ("grad_status", C.c_void_p),
    ]


def library_path() -> Path:
    env = os.environ.get("DEXR_LIBRARY")
    return Path(env) if env else Path(__file__).resolve().parent / "libdexr.so"


class DexrError(RuntimeError):
    pass


def load():
    """Load libdexr.so once; raise if it is missing or its struct layouts disagree with this file."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not path.exists():
        raise DexrError(
            f"{path} not found: build the CUDA library first (python -c 'import __graft_entry__ as g; g.build()' "
            f"or python -m dex_retargeting_b200.build).  There is no CPU fallback."
        )
    lib = C.CDLL(str(path))
    lib.dexr_version.restype = C.c_int
    lib.dexr_last_error.restype = C.c_char_p
    lib.dexr_build_id.restype = C.c_char_p
    lib.dexr_table_sizeof.restype = C.c_size_t
    lib.dexr_params_sizeof.restype = C.c_size_t
    lib.dexr_default_params.argtypes = [C.POINTER(DexrParams)]
    lib.dexr_default_params.restype = None
    lib.dexr_robot_create.argtypes = [C.POINTER(DexrTable), C.c_int, C.POINTER(C.c_void_p)]
    lib.dexr_robot_create_from_device.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
    lib.dexr_robot_device_table.argtypes = [C.c_void_p]
    lib.dexr_robot_device_table.restype = C.c_void_p
    lib.dexr_robot_destroy.argtypes = [C.c_void_p]
    lib.dexr_robot_destroy.restype = None
    lib.dexr_solve_frames.argtypes = [C.c_void_p, C.POINTER(DexrParams), C.POINTER(DexrFrames), C.c_int64, C.c_void_p]
    lib.dexr_solve_frames_multi.argtypes = [C.POINTER(DexrGroup), C.c_int32, C.c_void_p]
    lib.dexr_solve_sequences.argtypes = [C.c_void_p, C.POINTER(DexrParams), C.POINTER(DexrSequences), C.c_int64,
                                         C.c_int64, C.c_void_p]
    lib.dexr_solve_frames_host.argtypes = [C.c_void_p, C.POINTER(DexrParams), C.POINTER(DexrFrames), C.c_int64]
    lib.dexr_get_launch_info.argtypes = [C.c_void_p, C.POINTER(DexrLaunchInfo)]
    lib.dexr_preprocess_keypoints.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p]
    if lib.dexr_table_sizeof() != C.sizeof(DexrTable):
        raise DexrError(f"dexr_table_t layout mismatch: library {lib.dexr_table_sizeof()} vs binding {C.sizeof(DexrTable)}")
    if lib.dexr_params_sizeof() != C.sizeof(DexrParams):
        raise DexrError("dexr_params_t layout mismatch between library and binding")
    if hasattr(lib, "dexr_frames_sizeof"):
        lib.dexr_frames_sizeof.restype = C.c_size_t
        lib.dexr_sequences_sizeof.restype = C.c_size_t
        if lib.dexr_frames_sizeof() != C.sizeof(DexrFrames) or lib.dexr_sequences_sizeof() != C.sizeof(DexrSequences):
            raise DexrError("dexr_frames_t / dexr_sequences_t layout mismatch between library and binding (stale DEXR_LIBRARY?)")
    elif not os.environ.get("DEXR_LIBRARY"):
        raise DexrError(f"{path} does not export dexr_frames_sizeof: rebuild it (python -m dex_retargeting_b200.build --force)")
    # (an older A/B library named by DEXR_LIBRARY reads a prefix of the buffer structs -- fields are only ever appended -- so
    # the single-robot entry points still work with it; dexr_solve_frames_multi, whose groups embed the struct, does not)
    _LIB = lib
    return lib


def grad_library_path() -> Path:
    return Path(__file__).resolve().parent / "libdexr_grad.so"


def load_grad():
    """Load libdexr_grad.so once (lazily: only the backward pass needs it); raise if it is missing or its layout disagrees."""
    global _GRAD
    if _GRAD is not None:
        return _GRAD
    path = grad_library_path()
    if not path.exists():
        raise DexrError(f"{path} not found: build the CUDA libraries first (python -c 'import __graft_entry__ as g; g.build()' "
                        f"or python -m dex_retargeting_b200.build).  There is no CPU fallback.")
    lib = C.CDLL(str(path))
    lib.dexr_grad_version.restype = C.c_int
    lib.dexr_grad_build_id.restype = C.c_char_p
    lib.dexr_grad_last_error.restype = C.c_char_p
    lib.dexr_grad_frames_sizeof.restype = C.c_size_t
    lib.dexr_grad_frames.argtypes = [C.POINTER(DexrTable), C.c_void_p, C.POINTER(DexrParams), C.POINTER(DexrGradFrames), C.c_int64,
                                     C.c_int, C.c_void_p]
    lib.dexr_grad_sequences_sizeof.restype = C.c_size_t
    lib.dexr_grad_sequences.argtypes = [C.POINTER(DexrTable), C.c_void_p, C.POINTER(DexrParams), C.POINTER(DexrGradSequences),
                                        C.c_int64, C.c_int64, C.c_int, C.c_void_p]
    lib.dexr_grad_lowpass.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int64, C.c_int64, C.c_int,
                                      C.c_int, C.c_void_p]
    if lib.dexr_grad_frames_sizeof() != C.sizeof(DexrGradFrames):
        raise DexrError(f"dexr_grad_frames_t layout mismatch: library {lib.dexr_grad_frames_sizeof()} vs binding "
                        f"{C.sizeof(DexrGradFrames)}")
    if lib.dexr_grad_sequences_sizeof() != C.sizeof(DexrGradSequences):
        raise DexrError(f"dexr_grad_sequences_t layout mismatch: library {lib.dexr_grad_sequences_sizeof()} vs binding "
                        f"{C.sizeof(DexrGradSequences)}")
    _GRAD = lib
    return lib


def check_grad(code: int, what: str):
    if code != 0:
        msg = load_grad().dexr_grad_last_error().decode("utf-8", "replace")
        raise DexrError(f"{what} failed ({code}): {msg}")


def build_id() -> str:
    """The loaded library's source stamp (`dexr_build_id`)."""
    return load().dexr_build_id().decode()


def check(code: int, what: str):
    if code != 0:
        msg = load().dexr_last_error().decode("utf-8", "replace")
        raise DexrError(f"{what} failed ({code}): {msg}")


def default_params() -> DexrParams:
    p = DexrParams()
    load().dexr_default_params(C.byref(p))
    return p
