"""Host emulation of the stream backward pass (TEST INFRASTRUCTURE): builds tests/emu/emu_grad_seq_driver.cpp -- which compiles
dex_retargeting_b200/csrc/dexr_grad_seq_kernels.cuh through tests/emu/warp_shim.h -- with g++, like tests/emu_grad_host.py does
for the frame backward pass.  The library also exports emu_grad_frames.  Never used by the product."""
import copy
import ctypes as C
import subprocess
from functools import lru_cache

import numpy as np

from emu_grad_host import CSRC, EMU, OUT, ROOT

SOURCES = [EMU / "emu_grad_seq_driver.cpp", EMU / "emu_grad_driver.cpp", EMU / "warp_shim.h", CSRC / "dexr_grad_seq_kernels.cuh",
           CSRC / "dexr_grad_kernels.cuh", CSRC / "dexr_kernels.cuh", ROOT / "include" / "dexr.h", ROOT / "include" / "dexr_grad.h"]


@lru_cache(maxsize=None)
def load():
    OUT.mkdir(exist_ok=True)
    so = OUT / "libdexr_grad_seq_emu.so"
    if not so.exists() or any(so.stat().st_mtime < p.stat().st_mtime for p in SOURCES):
        # -O0 for the same reason as tests/emu_host.py: the rendezvous protocol compares call sites
        cmd = ["g++", "-O0", "-std=c++17", "-fPIC", "-shared", f"-I{EMU / 'stub'}", "-o", str(so), str(EMU / "emu_grad_seq_driver.cpp")]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("g++ failed building the stream backward host emulation:\n" + res.stderr[-4000:])
    lib = C.CDLL(str(so))
    lib.emu_grad_sequences.restype = C.c_int
    return lib


def forward_trace(seq, keypoints, state=None):
    """Emulated forward of the autograd route: the stream solver with the filter off.  Returns (trace x* [S,T,n],
    q [S,T,dof] unfiltered, status [S,T], entry state, exit state)."""
    import emu_host

    unfiltered = copy.copy(seq)
    unfiltered.filter = None
    kp = np.ascontiguousarray(keypoints, np.float32)
    S = kp.shape[0]
    opt = seq.optimizer
    if state is None:
        t = opt.build_table()
        state = dict(last_qpos=np.tile(seq.joint_limits.mean(1).astype(np.float32), (S, 1)),
                     filter_state=np.zeros((S, t.dof), np.float32), filter_init=np.zeros(S, np.uint8),
                     projected=np.zeros((S, t.len_proj), np.uint8) if t.len_proj else None, damping=np.zeros(S, np.float32))
    entry = {k: (None if v is None else v.copy()) for k, v in state.items()}
    q, status, exit_state = emu_host.solve_sequences(unfiltered, kp, state={k: (None if v is None else v.copy())
                                                                           for k, v in state.items()})
    x = np.ascontiguousarray(q[:, :, opt.idx_pin2target])
    return x, q, status, entry, exit_state


def grad_sequences(seq, keypoints, qpos, last_qpos, filter_init=None, projected=None, status=None, grad_robot_qpos=None,
                   grad_last_qpos=None, grad_filter_state=None, lp_alpha=None):
    """Emulated dexr_grad_sequences.  Returns (grad keypoints [S,T,21,3], grad entry last_qpos [S,n], grad entry filter_state
    [S,dof], grad status [S,T], projected_ws [S,T,len_proj] or None)."""
    from dex_retargeting_b200 import _native as N

    lib = load()
    opt = seq.optimizer
    table = opt.build_table()
    prm = opt.params(clip_init=True, lp_alpha=seq.low_pass_alpha if lp_alpha is None else lp_alpha)
    assert table.n_fixed == 0, "streams with fixed joints: not wired in the emulation helper"

    def arr(a, dt):
        return None if a is None else np.ascontiguousarray(a, dtype=dt)

    kp, q, last = arr(keypoints, np.float32), arr(qpos, np.float32), arr(last_qpos, np.float32)
    finit, proj, st = arr(filter_init, np.uint8), arr(projected, np.uint8), arr(status, np.int32)
    gy, gl, gf = arr(grad_robot_qpos, np.float32), arr(grad_last_qpos, np.float32), arr(grad_filter_state, np.float32)
    S, T = kp.shape[:2]
    ws = np.full((S, T, table.len_proj), 255, np.uint8) if table.len_proj else None
    g_kp = np.full(kp.shape, np.nan, np.float32)
    g_last = np.full((S, table.n_var), np.nan, np.float32)
    g_fs = np.full((S, table.dof), np.nan, np.float32)
    g_st = np.full((S, T), -1, np.int32)

    def ptr(a):
        return None if a is None else a.ctypes.data

    io = N.DexrGradSequences()
    io.keypoints, io.last_qpos, io.projected, io.filter_init = ptr(kp), ptr(last), ptr(proj), ptr(finit)
    io.qpos, io.status, io.grad_robot_qpos, io.grad_last_qpos_out, io.grad_filter_state_out = ptr(q), ptr(st), ptr(gy), ptr(gl), ptr(gf)
    io.projected_ws = ptr(ws)
    io.grad_keypoints, io.grad_last_qpos, io.grad_filter_state, io.grad_status = ptr(g_kp), ptr(g_last), ptr(g_fs), ptr(g_st)
    err = C.create_string_buffer(600)
    rc = lib.emu_grad_sequences(C.byref(table), C.byref(prm), C.byref(io), C.c_longlong(S), C.c_longlong(T), err, C.c_int(600))
    if rc != 0:
        raise RuntimeError(f"stream backward host emulation failed ({rc}): {err.value.decode()}")
    return g_kp, g_last, g_fs, g_st, ws
