"""Autograd for `Optimizer.retarget_batch`: the implicit-function backward pass (libdexr_grad.so, include/dexr_grad.h).

The forward pass is the ordinary batched solve (`dexr_solve_frames`), bit for bit.  The backward pass differentiates each
frame's optimality condition at the returned minimiser x*: one exact-Hessian build, one Cholesky factorisation and two
triangular solves per frame on the GPU, giving dl/dkeypoints (or dl/dref_value) and dl/dlast_qpos.  Joints held at an active
bound get no sensitivity; the warm start's role as the starting point is not differentiable (only its role as the
regularisation anchor is).  Frames the forward solve flagged (max iterations, non-finite input) get a zero gradient.
"""
from __future__ import annotations

import ctypes as C

import torch
from torch.autograd.function import once_differentiable

from . import _native as N


def grad_frames(opt, qpos, grad_qpos, *, last_qpos, keypoints=None, ref_value=None, fixed_qpos=None, projected=None,
                status=None, clip_init=False, stream=None):
    """Launch the backward pass of `opt.retarget_batch` (all tensors contiguous, on the optimizer's device; `projected`: the
    DexPilot flags AFTER the forward call).  Returns (grad of keypoints / ref_value, grad of last_qpos, grad status int32 [B])."""
    eng = opt.engine()
    glib = N.load_grad()
    dev = torch.device("cuda", eng.device)
    B = qpos.shape[0]
    io = N.DexrGradFrames()

    def ptr(t):
        return None if t is None else t.data_ptr()

    io.keypoints, io.ref_value, io.fixed_qpos, io.last_qpos = ptr(keypoints), ptr(ref_value), ptr(fixed_qpos), ptr(last_qpos)
    io.projected, io.qpos, io.status, io.grad_qpos = ptr(projected), ptr(qpos), ptr(status), ptr(grad_qpos)
    g_in = torch.empty_like(keypoints if keypoints is not None else ref_value)
    g_last = torch.empty((B, opt.opt_dof), dtype=torch.float32, device=dev)
    g_status = torch.empty((B,), dtype=torch.int32, device=dev)
    if keypoints is not None:
        io.grad_keypoints = g_in.data_ptr()
    else:
        io.grad_ref_value = g_in.data_ptr()
    io.grad_last_qpos, io.grad_status = g_last.data_ptr(), g_status.data_ptr()
    s = stream if stream is not None else torch.cuda.current_stream(dev)
    p = opt.params(clip_init=clip_init)
    table_dev = eng.lib.dexr_robot_device_table(eng.handle)
    N.check_grad(glib.dexr_grad_frames(C.byref(eng.table), C.c_void_p(table_dev), C.byref(p), C.byref(io), B, eng.device,
                                       C.c_void_p(s.cuda_stream)), "dexr_grad_frames")
    return g_in, g_last, g_status


class RetargetFunction(torch.autograd.Function):
    """qpos = retarget(keypoints | ref_value, last_qpos); the side outputs of the call stay plain tensors."""

    @staticmethod
    def forward(ctx, opt, kwargs, inp, last_qpos):
        by_kp = kwargs.pop("_by_keypoints")
        fixed_qpos = kwargs.get("fixed_qpos")
        projected = kwargs.get("projected")
        status = kwargs.get("status_out")
        own_status = status is None
        if own_status:  # the backward pass needs the forward status words
            status = torch.empty((last_qpos.shape[0],), dtype=torch.int32, device=last_qpos.device)
            kwargs["status_out"] = status
        src = dict(keypoints=inp) if by_kp else dict(ref_value=inp)
        qpos = opt._retarget_batch_launch(last_qpos=last_qpos, **src, **kwargs)
        ctx.opt, ctx.by_kp, ctx.clip_init = opt, by_kp, kwargs.get("clip_init", False)
        # the caller's flag tensor is rewritten in place by its next frame before backward runs: keep this frame's flags
        flags = projected.clone() if projected is not None else None
        ctx.save_for_backward(inp, last_qpos, fixed_qpos, flags, qpos, status.clone() if not own_status else status)
        return qpos

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_qpos):  # (runs on the current stream, which autograd sets to the forward call's)
        inp, last_qpos, fixed_qpos, flags, qpos, status = ctx.saved_tensors
        src = dict(keypoints=inp) if ctx.by_kp else dict(ref_value=inp)
        g_in, g_last, g_status = grad_frames(ctx.opt, qpos, grad_qpos.contiguous(), last_qpos=last_qpos, fixed_qpos=fixed_qpos,
                                             projected=flags, status=status, clip_init=ctx.clip_init, **src)
        ctx.opt.last_grad_status = g_status
        return None, None, g_in if ctx.needs_input_grad[2] else None, g_last if ctx.needs_input_grad[3] else None


def retarget_batch_autograd(opt, *, keypoints=None, ref_value=None, last_qpos=None, **kwargs):
    """The autograd route of `Optimizer.retarget_batch` (see there for when it is taken and what it refuses)."""
    if kwargs.get("out") is not None:
        raise ValueError("retarget_batch: `out=` cannot be combined with inputs that require grad (the result must be a new "
                         "autograd tensor)")
    if kwargs.get("raw_hand") is not None:
        raise ValueError("retarget_batch: raw_hand is not differentiable (the wrist-frame estimate from landmarks 0/5/9 is "
                         "nonlinear); pre-process the keypoints in torch and pass them instead")
    fixed = kwargs.get("fixed_qpos")
    if fixed is not None and fixed.requires_grad:
        raise ValueError("retarget_batch: gradients with respect to fixed_qpos are not supported; detach it")
    by_kp = keypoints is not None
    kw = {k: v for k, v in kwargs.items() if k != "out"}
    kw["_by_keypoints"] = by_kp
    return RetargetFunction.apply(opt, kw, keypoints if by_kp else ref_value, last_qpos)
