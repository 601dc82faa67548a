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


# ---------------------------------------------------------------------------------------------------------- streams
def grad_sequences(seq, keypoints, qpos, *, last_qpos, filter_init=None, projected=None, fixed_qpos=None, status=None,
                   grad_robot_qpos=None, grad_last_qpos=None, grad_filter_state=None, lp_alpha=None, projected_ws=None,
                   stream=None):
    """Launch the backward pass of `seq.retarget_sequences` through S streams x T steps (all tensors contiguous, on the
    optimizer's device).  `qpos` [S,T,opt_dof]: the forward trace x*_t; `last_qpos` / `filter_init` / `projected`: the state the
    streams ENTERED the forward call with; `grad_*`: upstream gradients of the filtered robot qpos [S,T,dof], of the exit
    last_qpos [S,opt_dof] and of the exit filter_state [S,dof] (None: zero); `lp_alpha` defaults to the sequence's filter.
    Returns (grad keypoints [S,T,21,3], grad entry last_qpos [S,opt_dof], grad entry filter_state [S,dof],
    grad status int32 [S,T], projected_ws [S,T,len_proj] uint8 -- the DexPilot flags each step applied -- or None)."""
    opt = seq.optimizer
    eng = opt.engine()
    glib = N.load_grad()
    dev = torch.device("cuda", eng.device)
    S, T = int(keypoints.shape[0]), int(keypoints.shape[1])
    len_proj = int(eng.table.len_proj)
    io = N.DexrGradSequences()

    def ptr(t):
        return None if t is None else t.data_ptr()

    io.keypoints, io.fixed_qpos, io.last_qpos, io.projected = ptr(keypoints), ptr(fixed_qpos), ptr(last_qpos), ptr(projected)
    io.filter_init, io.qpos, io.status = ptr(filter_init), ptr(qpos), ptr(status)
    io.grad_robot_qpos, io.grad_last_qpos_out, io.grad_filter_state_out = ptr(grad_robot_qpos), ptr(grad_last_qpos), \
        ptr(grad_filter_state)
    if len_proj and projected_ws is None:
        projected_ws = torch.empty((S, T, len_proj), dtype=torch.uint8, device=dev)
    io.projected_ws = ptr(projected_ws)
    g_kp = torch.empty_like(keypoints)
    g_last = torch.empty((S, opt.opt_dof), dtype=torch.float32, device=dev)
    g_fs = torch.empty((S, opt.robot.dof), dtype=torch.float32, device=dev)
    g_status = torch.empty((S, T), dtype=torch.int32, device=dev)
    io.grad_keypoints, io.grad_last_qpos, io.grad_filter_state, io.grad_status = ptr(g_kp), ptr(g_last), ptr(g_fs), ptr(g_status)
    s = stream if stream is not None else torch.cuda.current_stream(dev)
    p = opt.params(clip_init=True, lp_alpha=seq.low_pass_alpha if lp_alpha is None else lp_alpha)
    table_dev = eng.lib.dexr_robot_device_table(eng.handle)
    N.check_grad(glib.dexr_grad_sequences(C.byref(eng.table), C.c_void_p(table_dev), C.byref(p), C.byref(io), S, T, eng.device,
                                          C.c_void_p(s.cuda_stream)), "dexr_grad_sequences")
    return g_kp, g_last, g_fs, g_status, projected_ws


def lowpass(q, y, filter_state, filter_init, alpha, stream):
    """dexr_grad_lowpass: the stream solver's low-pass filter over q [S,T,dof] -> y, state updated in place."""
    S, T, dof = (int(v) for v in q.shape)
    glib = N.load_grad()
    N.check_grad(glib.dexr_grad_lowpass(q.data_ptr(), y.data_ptr(), filter_state.data_ptr(), filter_init.data_ptr(),
                                        float(alpha), S, T, dof, q.device.index, C.c_void_p(stream.cuda_stream)),
                 "dexr_grad_lowpass")


class SequencesFunction(torch.autograd.Function):
    """(robot_qpos, exit last_qpos, exit filter_state) = retarget_sequences(keypoints, entry last_qpos, entry filter_state).
    filter_init, projected and damping are state without a gradient, updated in place."""

    @staticmethod
    def forward(ctx, seq, state, kw, keypoints, last_qpos, filter_state):
        opt = seq.optimizer
        eng = opt.engine()
        dev = torch.device("cuda", eng.device)
        S, T = int(keypoints.shape[0]), int(keypoints.shape[1])
        s = kw["stream"] if kw["stream"] is not None else torch.cuda.current_stream(dev)
        fixed_qpos = kw["fixed_qpos"]
        ctx.set_materialize_grads(False)
        # entry state the backward pass starts from (the flags and filter_init are rewritten in place below)
        last_in = last_qpos.detach().clone()
        finit_in = state.filter_init.clone()
        proj_in = state.projected.clone() if state.projected is not None else None
        exit_last = last_qpos.detach().clone()
        exit_fs = filter_state.detach().clone()
        status = kw["status_out"]
        own_status = status is None
        if own_status:
            status = torch.empty((S, T), dtype=torch.int32, device=dev)
        # 1. the solver with the filter off: robot_qpos_out is then the unfiltered q_t, and x*_t an exact gather of it
        trace_q = torch.empty((S, T, opt.robot.dof), dtype=torch.float32, device=dev)
        seq._launch_sequences(keypoints.detach(), state, fixed_qpos, trace_q, status, s, lp_alpha=-1.0, last_qpos=exit_last,
                              filter_state=exit_fs)
        # 2. the filter, with the fused kernel's expression (same bits as the filtered single launch)
        alpha = seq.low_pass_alpha
        if 0.0 <= alpha <= 1.0:
            robot_qpos = torch.empty_like(trace_q)
            lowpass(trace_q, robot_qpos, exit_fs, state.filter_init, alpha, s)
        else:
            robot_qpos = trace_q
        idx = torch.as_tensor(opt.idx_pin2target, dtype=torch.long, device=dev)
        trace = trace_q.index_select(2, idx).contiguous()
        ctx.seq, ctx.stream = seq, kw["stream"]
        ctx.save_for_backward(keypoints.detach(), fixed_qpos, last_in, proj_in, finit_in, trace,
                              status if own_status else status.clone())
        return robot_qpos, exit_last, exit_fs

    @staticmethod
    @once_differentiable
    def backward(ctx, g_robot, g_last, g_fs):  # (runs on the current stream, which autograd sets to the forward call's)
        keypoints, fixed_qpos, last_in, proj_in, finit_in, trace, status = ctx.saved_tensors
        S, T = int(keypoints.shape[0]), int(keypoints.shape[1])
        dev = keypoints.device
        if g_robot is None and g_last is None and g_fs is None:
            return None, None, None, None, None, None

        def c(t):
            return None if t is None else t.contiguous()

        if S == 0 or T == 0:  # nothing solved: the exit state is the entry state
            return (None, None, None, torch.zeros_like(keypoints) if ctx.needs_input_grad[3] else None,
                    (g_last if g_last is not None else torch.zeros_like(last_in)) if ctx.needs_input_grad[4] else None,
                    (g_fs if g_fs is not None else torch.zeros((S, ctx.seq.optimizer.robot.dof), device=dev))
                    if ctx.needs_input_grad[5] else None)
        g_kp, g_lq, g_fs_in, g_status, _ = grad_sequences(ctx.seq, keypoints, trace, last_qpos=last_in, filter_init=finit_in,
                                                          projected=proj_in, fixed_qpos=fixed_qpos, status=status,
                                                          grad_robot_qpos=c(g_robot), grad_last_qpos=c(g_last),
                                                          grad_filter_state=c(g_fs))
        ctx.seq.last_grad_status = g_status
        return (None, None, None, g_kp if ctx.needs_input_grad[3] else None, g_lq if ctx.needs_input_grad[4] else None,
                g_fs_in if ctx.needs_input_grad[5] else None)


def retarget_sequences_autograd(seq, keypoints, state, *, fixed_qpos=None, out=None, status_out=None, stream=None,
                                raw_hand=None):
    """The autograd route of `SeqRetargeting.retarget_sequences` (see there for when it is taken and what it refuses)."""
    if out is not None:
        raise ValueError("retarget_sequences: `out=` cannot be combined with inputs that require grad (the result must be a new "
                         "autograd tensor)")
    if raw_hand is not None:
        raise ValueError("retarget_sequences: raw_hand is not differentiable (the wrist-frame estimate from landmarks 0/5/9 is "
                         "nonlinear); pre-process the keypoints in torch and pass them instead")
    if fixed_qpos is not None and fixed_qpos.requires_grad:
        raise ValueError("retarget_sequences: gradients with respect to fixed_qpos are not supported; detach it")
    kw = dict(fixed_qpos=fixed_qpos, status_out=status_out, stream=stream)
    robot_qpos, last, fs = SequencesFunction.apply(seq, state, kw, keypoints, state.last_qpos, state.filter_state)
    state.last_qpos, state.filter_state = last, fs
    return robot_qpos, state
