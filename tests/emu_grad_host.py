"""Host emulation of the backward-pass source (TEST INFRASTRUCTURE): builds tests/emu/emu_grad_driver.cpp -- which compiles
dex_retargeting_b200/csrc/dexr_grad_kernels.cuh through tests/emu/warp_shim.h -- with g++ and calls it through ctypes, like
tests/emu_host.py does for the forward solver.  Never used by the product (the product path is libdexr_grad.so only)."""
import ctypes as C
import subprocess
from functools import lru_cache
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
EMU = ROOT / "tests" / "emu"
OUT = EMU / "_build"
CSRC = ROOT / "dex_retargeting_b200" / "csrc"
SOURCES = [EMU / "emu_grad_driver.cpp", EMU / "warp_shim.h", CSRC / "dexr_grad_kernels.cuh", CSRC / "dexr_kernels.cuh",
           ROOT / "include" / "dexr.h", ROOT / "include" / "dexr_grad.h"]


@lru_cache(maxsize=None)
def load():
    OUT.mkdir(exist_ok=True)
    so = OUT / "libdexr_grad_emu.so"
    if not so.exists() or any(so.stat().st_mtime < p.stat().st_mtime for p in SOURCES):
        # -O0 for the same reason as tests/emu_host.py: the rendezvous protocol compares call sites
        cmd = ["g++", "-O0", "-std=c++17", "-fPIC", "-shared", f"-I{EMU / 'stub'}", "-o", str(so), str(EMU / "emu_grad_driver.cpp")]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("g++ failed building the backward host emulation:\n" + res.stderr[-4000:])
    lib = C.CDLL(str(so))
    lib.emu_grad_frames.restype = C.c_int
    return lib


def grad_frames(opt, last_qpos, qpos, grad_qpos, keypoints=None, ref_value=None, fixed_qpos=None, projected=None, status=None,
                clip_init=False):
    """Emulated dexr_grad_frames for an Optimizer of the host mirror.  Returns (grad_input [B,21,3] or [B,m,3],
    grad_last_qpos [B,n], grad_status [B])."""
    from dex_retargeting_b200 import _native as N

    lib = load()
    table, prm = opt.build_table(), opt.params(clip_init=clip_init)

    def f32(a):
        return None if a is None else np.ascontiguousarray(a, dtype=np.float32)

    kp, ref, last, fixed, q, gq = f32(keypoints), f32(ref_value), f32(last_qpos), f32(fixed_qpos), f32(qpos), f32(grad_qpos)
    assert (kp is None) != (ref is None)
    B, n = last.shape[0], table.n_var
    gin = np.full((B, 21, 3) if kp is not None else (B, table.n_res, 3), np.nan, np.float32)
    glast = np.full((B, n), np.nan, np.float32)
    gst = np.full(B, -1, np.int32)
    keep = [kp, ref, last, fixed, q, gq, gin, glast, gst]
    if projected is not None:
        projected = np.ascontiguousarray(projected, dtype=np.uint8)
        keep.append(projected)
    if status is not None:
        status = np.ascontiguousarray(status, dtype=np.int32)
        keep.append(status)

    def ptr(a):
        return None if a is None else a.ctypes.data

    io = N.DexrGradFrames()
    io.keypoints, io.ref_value, io.fixed_qpos, io.last_qpos = ptr(kp), ptr(ref), ptr(fixed), ptr(last)
    io.projected, io.qpos, io.status, io.grad_qpos = ptr(projected), ptr(q), ptr(status), ptr(gq)
    if kp is not None:
        io.grad_keypoints = ptr(gin)
    else:
        io.grad_ref_value = ptr(gin)
    io.grad_last_qpos, io.grad_status = ptr(glast), ptr(gst)
    err = C.create_string_buffer(600)
    rc = lib.emu_grad_frames(C.byref(table), C.byref(prm), C.byref(io), C.c_longlong(B), err, C.c_int(600))
    if rc != 0:
        raise RuntimeError(f"backward host emulation failed ({rc}): {err.value.decode()}")
    return gin, glast, gst
