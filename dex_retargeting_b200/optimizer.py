"""Position / Vector / DexPilot optimizers backed by the sm_100a solver (libdexr.so).

Drop-in for `dex_retargeting.optimizer` (reference: src/dex_retargeting/optimizer.py:15-577): same
class names, constructor arguments, attributes (`idx_pin2target`, `idx_pin2fixed`,
`target_link_human_indices`, `computed_link_indices`, `origin_link_indices`, ...), the same
`retarget(ref_value, fixed_qpos, last_qpos) -> float32 (n,)` entry, the same ValueErrors.

What changed underneath: there is no nlopt object and no Python objective closure.  `retarget()` ships
one frame through the C ABI (`dexr_solve_frames_host`); the new `retarget_batch()` takes torch CUDA
tensors `[B, ...]` and solves every frame of the batch in ONE kernel launch (`dexr_solve_frames`).
The solver minimises the objective whose gradient the reference hands to SLSQP, i.e.
    L(x) + norm_delta * |x - last_qpos|^2      inside [lower - 1e-3, upper + 1e-3]
to convergence (the reference stops SLSQP early at ftol_abs 1e-5 / 1e-6, optimizer.py:136,239,397).
There is no CPU fallback: without the CUDA library / a GPU these calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from abc import abstractmethod
from typing import List, Optional

import numpy as np

from . import _native as N
from .kinematics_adaptor import KinematicAdaptor, MimicJointKinematicAdaptor
from .robot_wrapper import RobotWrapper
from .table import ObjectiveSpec, compile_table, table_bytes


class _SolverStats:
    """Stand-in for the attributes of `nlopt.opt` that callers read (seq_retarget.py:147-152)."""

    def __init__(self):
        self._value = float("nan")

    def last_optimum_value(self):
        return self._value


class _Engine:
    """Owns one `dexr_robot_t` handle (device copy of a robot table)."""

    def __init__(self, table: N.DexrTable, device: int, table_dev_ptr: Optional[int] = None):
        self.lib = N.load()
        self.table = table
        self.device = int(device)
        h = C.c_void_p()
        if table_dev_ptr is None:
            N.check(self.lib.dexr_robot_create(C.byref(table), self.device, C.byref(h)), "dexr_robot_create")
        else:
            N.check(self.lib.dexr_robot_create_from_device(C.c_void_p(table_dev_ptr), C.sizeof(N.DexrTable), self.device,
                                                            C.byref(h)), "dexr_robot_create_from_device")
        self.handle = h

    def launch_info(self) -> dict:
        info = N.DexrLaunchInfo()
        N.check(self.lib.dexr_get_launch_info(self.handle, C.byref(info)), "dexr_get_launch_info")
        return {k: getattr(info, k) for k, _ in info._fields_}

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.dexr_robot_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def _default_device() -> int:
    import torch

    return torch.cuda.current_device() if torch.cuda.is_available() else 0


class Optimizer:
    retargeting_type = "BASE"

    def __init__(self, robot: RobotWrapper, target_joint_names: List[str], target_link_human_indices: np.ndarray,
                 device: Optional[int] = None):
        self.robot = robot
        self.num_joints = robot.dof

        joint_names = robot.dof_joint_names
        idx_pin2target = []
        for name in target_joint_names:
            if name not in joint_names:
                raise ValueError(f"Joint {name} given does not appear to be in robot XML.")
            idx_pin2target.append(joint_names.index(name))
        self.target_joint_names = list(target_joint_names)
        self.idx_pin2target = np.array(idx_pin2target)
        self.idx_pin2fixed = np.array([i for i in range(robot.dof) if i not in idx_pin2target], dtype=int)
        self.opt_dof = len(idx_pin2target)  # includes nothing but the optimised joints
        self.opt = _SolverStats()
        self.last_status = None  # int32 status words of the most recent host-path solve (iterations | flags)
        self.last_grad_status = None  # int32 DEXR_GRAD_STATUS_* words of the most recent retarget_batch backward pass

        self.target_link_human_indices = target_link_human_indices
        self.has_free_joint = len([n for n in robot.link_names if "dummy" in n]) >= 6
        self.adaptor: Optional[KinematicAdaptor] = None

        # bounds: "no limit" until set_joint_limit is called (SeqRetargeting does, seq_retarget.py:22-31)
        self._limits = np.tile(np.array([[-1e4, 1e4]]), (self.opt_dof, 1))
        self._epsilon = 1e-3
        self._device = device
        self._engine: Optional[_Engine] = None
        # solver knobs that have no counterpart in the reference
        self.max_iters = 64
        # DEXR_STEP_TOL overrides the default stopping step for A/B runs (INTEGRATION.md); the attribute stays settable
        self.step_tol = float(os.environ.get("DEXR_STEP_TOL", 1e-5))
        # initial Levenberg-Marquardt damping: 1e-2, and 1.0 once a mimic adaptor is set (set_kinematic_adaptor); DEXR_LAMBDA0
        # overrides both for A/B runs; the attribute stays settable
        self.lambda0 = float(os.environ.get("DEXR_LAMBDA0", 1e-2))

    # ---------------------------------------------------------------- reference API
    def set_joint_limit(self, joint_limits: np.ndarray, epsilon=1e-3):
        joint_limits = np.asarray(joint_limits)
        if joint_limits.shape != (self.opt_dof, 2):
            raise ValueError(f"Expect joint limits have shape: {(self.opt_dof, 2)}, but get {joint_limits.shape}")
        self._limits = joint_limits.astype(np.float64).copy()
        self._epsilon = float(epsilon)
        self._engine = None

    def get_link_indices(self, target_link_names):
        return [self.robot.get_link_index(n) for n in target_link_names]

    def set_kinematic_adaptor(self, adaptor: KinematicAdaptor):
        # The reference calls adaptor.forward_qpos / backward_jacobian inside its Python objective (optimizer.py:150-151,
        # 186-187); here the adaptor is compiled into the robot table, and the only adaptor the reference ships --
        # the mimic-joint affine map -- is the only one the kernel knows.  Anything else would be silently ignored.
        if not isinstance(adaptor, MimicJointKinematicAdaptor):
            raise NotImplementedError(f"{type(adaptor).__name__}: only MimicJointKinematicAdaptor can be compiled into the "
                                      "robot table of the CUDA solver")
        self.adaptor = adaptor
        mimic = set(int(i) for i in adaptor.idx_pin2mimic)  # mimic joints are driven, not supplied
        self.idx_pin2fixed = np.array([x for x in self.idx_pin2fixed if int(x) not in mimic], dtype=int)
        self._engine = None
        # Robots with mimic joints fold the kinematic curvature into the reduced Hessian (H_x = M^T H_q M), where the solver's
        # positive-definite fallback cannot take it out again: an indefinite Hessian is only cured by more damping, one
        # factor 10 per failed factorisation.  Measured on 512 seeded frames per hand (host emulation, warm start 0.05 rad):
        # teleop SVH / Inspire / Ability pay 3.3 / 4.6 / 4.0 rejected trials per frame from 1e-2 and 1.5 / 2.7 / 2.1 from 1.0,
        # at unchanged iteration counts and identical answers; 10 is better still for the vector hands but costs the position
        # configurations iterations (offline Inspire 5.85 -> 6.36).
        if "DEXR_LAMBDA0" not in os.environ and len(mimic) > 0:
            self.lambda0 = 1.0

    @property
    def fixed_joint_names(self):
        names = self.robot.dof_joint_names
        return [names[i] for i in self.idx_pin2fixed]

    def retarget(self, ref_value, fixed_qpos, last_qpos, damping=None):
        """One frame.  ref_value: (m,3); fixed_qpos: (len(idx_pin2fixed),); last_qpos: (opt_dof,) warm start
        and regularisation anchor.  Returns float32 (opt_dof,) in `target_joint_names` order.
        `damping` (not in the reference): float32 array of one element that a caller feeding a STREAM frame by frame keeps
        between calls -- the solver's carried damping (`dexr_frames_t.damping_io`), read and updated in place."""
        if len(fixed_qpos) != len(self.idx_pin2fixed):
            raise ValueError(
                f"Optimizer has {len(self.idx_pin2fixed)} joints but non_target_qpos {fixed_qpos} is given"
            )
        qpos, _ = self._solve_host(np.asarray(ref_value, dtype=np.float32)[None], np.asarray(fixed_qpos, dtype=np.float32)[None],
                                   np.asarray(last_qpos, dtype=np.float32)[None], clip_init=False, damping=damping)
        return qpos[0]

    # ---------------------------------------------------------------- engine
    @abstractmethod
    def _objective_spec(self) -> ObjectiveSpec:
        ...

    def _loss_params(self, p: N.DexrParams):
        """Fill the loss-specific fields of the parameter block."""

    def _mimic_tuple(self):
        a = self.adaptor
        if isinstance(a, MimicJointKinematicAdaptor):
            return (a.source_joint_names, a.mimic_joint_names, [float(v) for v in a.multipliers], [float(v) for v in a.offsets])
        return None

    def build_table(self) -> N.DexrTable:
        return compile_table(self.robot.kin, self.target_joint_names, self._objective_spec(), self._limits,
                             self._epsilon, self._mimic_tuple(), self.fixed_joint_names)

    @property
    def device_index(self) -> int:
        if self._device is None:
            self._device = _default_device()
        return int(self._device)

    def engine(self) -> _Engine:
        if self._engine is None:
            self._engine = _Engine(self.build_table(), self.device_index)
        return self._engine

    def adopt_device_table(self, table: N.DexrTable, table_dev_ptr: int, device: int):
        """Use a table that already lives on `device` (after an NCCL broadcast, see parallel.py)."""
        self._device = device
        self._engine = _Engine(table, device, table_dev_ptr)

    def params(self, clip_init: bool = False, lp_alpha: float = -1.0, raw_hand=None) -> N.DexrParams:
        """`raw_hand`: None = the keypoints are wrist-centred MANO-convention points; HandType.right / left (or "right" /
        "left", any case: single_hand_detector.py:47 spells them "Right" / "Left") = they are RAW detector landmarks of that hand and the kernel pre-processes them itself (fused
        single_hand_detector.py:100-103, 130-158)."""
        p = N.default_params()
        p.tol, p.lambda0, p.max_iters = self.step_tol, self.lambda0, int(self.max_iters)
        p.clip_init = 1 if clip_init else 0
        p.lp_alpha = float(lp_alpha)
        if raw_hand is not None:
            name = (raw_hand if isinstance(raw_hand, str) else raw_hand.name).lower()  # the detector's own spelling is "Right" / "Left"
            if name not in ("right", "left"):
                raise ValueError(f"raw_hand must be right or left, got {raw_hand!r}")
            p.preprocess = 1 if name == "right" else 2
        self._loss_params(p)
        return p

    @property
    def num_residuals(self) -> int:
        return len(self._objective_spec().res_task)

    # ---------------------------------------------------------------- host path (numpy, B small)
    def _solve_host(self, ref_value, fixed_qpos, last_qpos, clip_init, keypoints=None, projected=None,
                    want_robot_qpos=False, damping=None):
        eng = self.engine()
        B = last_qpos.shape[0]
        n = self.opt_dof
        m = self.num_residuals
        io = N.DexrFrames()
        keep = []

        def ptr(a):
            keep.append(a)
            return a.ctypes.data_as(C.c_void_p)

        if keypoints is not None:
            kp = np.ascontiguousarray(keypoints, dtype=np.float32).reshape(B, N.NUM_KEYPOINTS, 3)
            io.keypoints = ptr(kp)
        else:
            rv = np.ascontiguousarray(ref_value, dtype=np.float32)
            if rv.shape != (B, m, 3):
                raise ValueError(f"ref_value must have shape {(m, 3)}, got {rv.shape[1:]}")
            io.ref_value = ptr(rv)
        lq = np.ascontiguousarray(last_qpos, dtype=np.float32).reshape(B, n)
        io.last_qpos = ptr(lq)
        nf = len(self.idx_pin2fixed)
        if nf:
            io.fixed_qpos = ptr(np.ascontiguousarray(fixed_qpos, dtype=np.float32).reshape(B, nf))
        qpos = np.empty((B, n), dtype=np.float32)
        cost = np.empty((B,), dtype=np.float32)
        status = np.empty((B,), dtype=np.int32)
        io.qpos_out, io.cost_out, io.status_out = ptr(qpos), ptr(cost), ptr(status)
        rq = None
        if want_robot_qpos:
            rq = np.empty((B, self.robot.dof), dtype=np.float32)
            io.robot_qpos_out = ptr(rq)
        if projected is not None:
            io.projected = ptr(projected)
        if damping is not None:
            if not isinstance(damping, np.ndarray) or damping.dtype != np.float32 or damping.shape != (B,) or not damping.flags.c_contiguous:
                raise ValueError(f"damping must be a contiguous float32 array of shape ({B},) (updated in place)")
            io.damping_io = ptr(damping)
        p = self.params(clip_init=clip_init)
        N.check(eng.lib.dexr_solve_frames_host(eng.handle, C.byref(p), C.byref(io), B), "dexr_solve_frames_host")
        # nlopt's last_optimum_value() is the reference objective's VALUE, which leaves the regulariser out
        # (optimizer.py:166-167 vs :194); the kernel's cost includes norm_delta |x - x_last|^2, so take it back out
        reg = float(self.norm_delta) * float(((qpos[-1].astype(np.float64) - lq[-1].astype(np.float64)) ** 2).sum())
        self.opt._value = float(cost[-1]) - reg
        self.last_status = status
        return qpos, rq

    def retarget_batch_host(self, ref_value=None, fixed_qpos=None, last_qpos=None, *, keypoints=None, projected=None,
                            out=None, clip_init=False, raw_hand=None, damping=None):
        """Host-buffer twin of `retarget_batch`: float32 numpy arrays (or CPU torch tensors, ideally
        pinned) in, numpy out.  The library stages chunks through its own device buffers and overlaps the
        host->device copies, the solve and the device->host copies (`dexr_solve_frames_host`).  Returns
        when `out` [B,opt_dof] holds the results."""
        def as_np(a, dtype=np.float32):
            if a is None:
                return None
            if hasattr(a, "numpy") and not isinstance(a, np.ndarray):
                a = a.numpy()
            return np.ascontiguousarray(a, dtype=dtype)

        last = as_np(last_qpos)
        if last is None:
            raise ValueError("last_qpos is required")
        if (ref_value is None) == (keypoints is None):
            raise ValueError("give exactly one of ref_value / keypoints")
        B = last.shape[0]
        eng = self.engine()
        io = N.DexrFrames()
        keep = []

        def ptr(a, shape, name):
            if tuple(a.shape) != tuple(shape):
                raise ValueError(f"{name}: expected shape {tuple(shape)}, got {tuple(a.shape)}")
            keep.append(a)
            return a.ctypes.data_as(C.c_void_p)

        if keypoints is not None:
            io.keypoints = ptr(as_np(keypoints), (B, N.NUM_KEYPOINTS, 3), "keypoints")
        else:
            io.ref_value = ptr(as_np(ref_value), (B, self.num_residuals, 3), "ref_value")
        io.last_qpos = ptr(last, (B, self.opt_dof), "last_qpos")
        nf = len(self.idx_pin2fixed)
        if nf:
            if fixed_qpos is None:
                raise ValueError(f"Optimizer has {nf} joints but no fixed_qpos is given")
            io.fixed_qpos = ptr(as_np(fixed_qpos), (B, nf), "fixed_qpos")
        if projected is not None:
            pj = projected.numpy() if hasattr(projected, "numpy") and not isinstance(projected, np.ndarray) else projected
            if pj.dtype != np.uint8 or not pj.flags.c_contiguous:
                raise ValueError("projected must be a contiguous uint8 array (updated in place)")
            io.projected = ptr(pj, (B, self._objective_spec().len_proj), "projected")
        if damping is not None:  # per-frame carried damping of B streams fed frame by frame (dexr_frames_t.damping_io), in place
            dm = damping.numpy() if hasattr(damping, "numpy") and not isinstance(damping, np.ndarray) else damping
            if dm.dtype != np.float32 or not dm.flags.c_contiguous:
                raise ValueError("damping must be a contiguous float32 array (updated in place)")
            io.damping_io = ptr(dm, (B,), "damping")
        if out is None:
            out = np.empty((B, self.opt_dof), dtype=np.float32)
        out_np = out.numpy() if hasattr(out, "numpy") and not isinstance(out, np.ndarray) else out
        if out_np.dtype != np.float32 or not out_np.flags.c_contiguous:
            raise ValueError("out must be a contiguous float32 array")
        io.qpos_out = ptr(out_np, (B, self.opt_dof), "out")
        p = self.params(clip_init=clip_init, raw_hand=raw_hand)
        N.check(eng.lib.dexr_solve_frames_host(eng.handle, C.byref(p), C.byref(io), B), "dexr_solve_frames_host")
        return out

    # ---------------------------------------------------------------- device path (torch, B large)
    def retarget_batch(self, ref_value=None, fixed_qpos=None, last_qpos=None, *, keypoints=None, projected=None,
                       out=None, robot_qpos_out=None, status_out=None, cost_out=None, clip_init=False, stream=None, raw_hand=None,
                       damping=None):
        """Solve B independent frames in one launch.  All arguments are float32 CUDA tensors on this
        optimizer's device (projected: uint8, status_out: int32), contiguous:
          ref_value [B,m,3]  OR  keypoints [B,21,3] (the human-index gather is done in the kernel)
          fixed_qpos [B,len(idx_pin2fixed)] (omit when there are none), last_qpos [B,opt_dof]
        `raw_hand` (HandType): `keypoints` are raw detector landmarks of that hand; the wrist-frame estimate and the MANO
        rotation of the reference's detector are applied inside the solver (see `params`).
        `damping` [B] float32, in/out: the carried damping of B STREAMS that are fed frame by frame through this call
        (`StreamState.damping`, `dexr_frames_t.damping_io`); omit for independent frames.
        Returns qpos [B,opt_dof] (= `out` if given).  Nothing is synchronised.
        Autograd: when grad mode is on and `keypoints`, `ref_value` or `last_qpos` requires grad, the result carries a `grad_fn`
        whose backward is the implicit-function gradient of each frame's minimiser (dex_retargeting_b200/grad.py; the forward
        results are the same bits).  That route refuses `out=`, `raw_hand` and a `fixed_qpos` that requires grad; the per-frame
        status of the last backward pass is left in `last_grad_status`."""
        import torch

        if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (keypoints, ref_value, last_qpos)):
            from .grad import retarget_batch_autograd

            return retarget_batch_autograd(self, keypoints=keypoints, ref_value=ref_value, last_qpos=last_qpos,
                                           fixed_qpos=fixed_qpos, projected=projected, out=out, robot_qpos_out=robot_qpos_out,
                                           status_out=status_out, cost_out=cost_out, clip_init=clip_init, stream=stream,
                                           raw_hand=raw_hand, damping=damping)
        return self._retarget_batch_launch(ref_value, fixed_qpos, last_qpos, keypoints=keypoints, projected=projected, out=out,
                                           robot_qpos_out=robot_qpos_out, status_out=status_out, cost_out=cost_out,
                                           clip_init=clip_init, stream=stream, raw_hand=raw_hand, damping=damping)

    def _retarget_batch_launch(self, ref_value=None, fixed_qpos=None, last_qpos=None, *, keypoints=None, projected=None, out=None,
                               robot_qpos_out=None, status_out=None, cost_out=None, clip_init=False, stream=None, raw_hand=None,
                               damping=None):
        """The one `dexr_solve_frames` launch behind `retarget_batch` (no autograd)."""
        import torch

        eng, io, p, out, B = self._prepare_batch(ref_value, fixed_qpos, last_qpos, keypoints=keypoints, projected=projected, out=out,
                                                 robot_qpos_out=robot_qpos_out, status_out=status_out, cost_out=cost_out,
                                                 clip_init=clip_init, raw_hand=raw_hand, damping=damping)
        s = stream if stream is not None else torch.cuda.current_stream(torch.device("cuda", eng.device))
        N.check(eng.lib.dexr_solve_frames(eng.handle, C.byref(p), C.byref(io), B, C.c_void_p(s.cuda_stream)),
                "dexr_solve_frames")
        return out

    def _prepare_batch(self, ref_value=None, fixed_qpos=None, last_qpos=None, *, keypoints=None, projected=None, out=None,
                       robot_qpos_out=None, status_out=None, cost_out=None, clip_init=False, raw_hand=None, stream=None,
                       damping=None):
        """Validate the tensors of one batch and lay them out as `dexr_frames_t` (shared by the single-robot and the
        mixed-robot launch).  Returns (engine, io, params, out, B)."""
        import torch

        eng = self.engine()
        if last_qpos is None:
            raise ValueError("last_qpos is required")
        B = last_qpos.shape[0]
        dev = torch.device("cuda", eng.device)

        def chk(t, shape, dtype, name):
            if t.device != dev or t.dtype != dtype or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
                raise ValueError(f"{name}: expected contiguous {dtype} tensor of shape {tuple(shape)} on {dev}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")
            return t.data_ptr()

        io = N.DexrFrames()
        m = self.num_residuals
        if (ref_value is None) == (keypoints is None):
            raise ValueError("give exactly one of ref_value / keypoints")
        if keypoints is not None:
            io.keypoints = chk(keypoints, (B, N.NUM_KEYPOINTS, 3), torch.float32, "keypoints")
        else:
            io.ref_value = chk(ref_value, (B, m, 3), torch.float32, "ref_value")
        io.last_qpos = chk(last_qpos, (B, self.opt_dof), torch.float32, "last_qpos")
        nf = len(self.idx_pin2fixed)
        if nf:
            if fixed_qpos is None:
                raise ValueError(f"Optimizer has {nf} joints but no fixed_qpos is given")
            io.fixed_qpos = chk(fixed_qpos, (B, nf), torch.float32, "fixed_qpos")
        if out is None:
            out = torch.empty((B, self.opt_dof), dtype=torch.float32, device=dev)
        io.qpos_out = chk(out, (B, self.opt_dof), torch.float32, "out")
        if robot_qpos_out is not None:
            io.robot_qpos_out = chk(robot_qpos_out, (B, self.robot.dof), torch.float32, "robot_qpos_out")
        if status_out is not None:
            io.status_out = chk(status_out, (B,), torch.int32, "status_out")
        if cost_out is not None:
            io.cost_out = chk(cost_out, (B,), torch.float32, "cost_out")
        if projected is not None:
            io.projected = chk(projected, (B, self._objective_spec().len_proj), torch.uint8, "projected")
        if damping is not None:
            io.damping_io = chk(damping, (B,), torch.float32, "damping")
        if raw_hand is not None and keypoints is None:
            raise ValueError("raw_hand needs `keypoints` (raw landmarks), not ref_value")
        return eng, io, self.params(clip_init=clip_init, raw_hand=raw_hand), out, B


def retarget_batch_mixed(jobs, stream=None):
    """Several robots, ONE call (`dexr_solve_frames_multi`): `jobs` is a list of `(optimizer, kwargs)` where `kwargs` are the
    arguments of `Optimizer.retarget_batch` for that robot's batch (every optimizer on the same device, at most 16 groups).
    The reference builds one optimizer per robot and would run them back to back (retargeting_config.py:167-257); here the
    library forks one standalone persistent kernel per robot onto its own side streams and joins them on the caller's stream
    with events, so the groups share the SMs and small per-robot batches do not each wait for the previous group's tail
    (`DEXR_MULTI_MODE=persistent` selects the alternative, one kernel whose CTAs walk the groups; measured slower at every
    size, profiles/r02/mixed_launch_sweep.txt).  Returns the list of result tensors, bit-identical to per-robot launches."""
    import torch

    if len(jobs) > N.MAX_GROUPS:
        raise ValueError(f"at most {N.MAX_GROUPS} robot groups per launch, got {len(jobs)}")
    groups = (N.DexrGroup * max(len(jobs), 1))()
    keep, outs, dev_index = [], [], None
    for i, (opt, kw) in enumerate(jobs):
        eng, io, p, out, B = opt._prepare_batch(**kw)
        if dev_index is None:
            dev_index = eng.device
        elif eng.device != dev_index:
            raise ValueError("all robots of a mixed launch must live on the same device")
        keep.append((eng, p))
        groups[i].robot, groups[i].params, groups[i].io, groups[i].num_frames = eng.handle, C.pointer(p), io, B
        outs.append(out)
    if not jobs:
        return outs
    s = stream if stream is not None else torch.cuda.current_stream(torch.device("cuda", dev_index))
    N.check(N.load().dexr_solve_frames_multi(groups, len(jobs), C.c_void_p(s.cuda_stream)), "dexr_solve_frames_multi")
    return outs


class PositionOptimizer(Optimizer):
    retargeting_type = "POSITION"

    def __init__(self, robot: RobotWrapper, target_joint_names: List[str], target_link_names: List[str],
                 target_link_human_indices: np.ndarray, huber_delta=0.02, norm_delta=4e-3, device=None):
        super().__init__(robot, target_joint_names, target_link_human_indices, device)
        self.body_names = target_link_names
        self.huber_delta = huber_delta
        self.norm_delta = norm_delta
        self.target_link_indices = self.get_link_indices(target_link_names)  # also the name check
        # The per-coordinate Huber loss is solved with its positive-semidefinite majoriser throughout, so the Newton model needs
        # less initial damping than the norm-Huber losses: 1e-3 instead of 1e-2 (host emulation, 512 seeded frames per hand,
        # warm start 0.05 rad: Shadow 3.98 -> 3.26 iterations, LEAP 3.11 -> 2.74, Allegro 3.08 -> 2.90, identical answers; cold
        # starts 0.5 rad: iterations unchanged, +0.1-0.2 rejected trials per frame).  Hands with mimic joints override it with 1.0
        # (set_kinematic_adaptor); DEXR_LAMBDA0 overrides everything.
        if "DEXR_LAMBDA0" not in os.environ:
            self.lambda0 = 1e-3

    def _objective_spec(self) -> ObjectiveSpec:
        idx = [int(i) for i in np.asarray(self.target_link_human_indices).reshape(-1)]
        m = len(self.body_names)
        if len(idx) != m:
            raise ValueError("Position retargeting link names and link indices dim mismatch")
        return ObjectiveSpec(N.LOSS_POSITION, list(self.body_names), list(range(m)), [-1] * m, idx, [-1] * m)

    def _loss_params(self, p):
        p.huber_delta, p.norm_delta, p.scaling = self.huber_delta, self.norm_delta, 1.0


def _link_cache(origin_names, task_names):
    """Positions of a link shared by several vectors are computed once (optimizer.py:224-234)."""
    computed = list(dict.fromkeys(list(origin_names) + list(task_names)))
    return computed, [computed.index(n) for n in origin_names], [computed.index(n) for n in task_names]


class VectorOptimizer(Optimizer):
    retargeting_type = "VECTOR"

    def __init__(self, robot: RobotWrapper, target_joint_names: List[str], target_origin_link_names: List[str],
                 target_task_link_names: List[str], target_link_human_indices: np.ndarray, huber_delta=0.02,
                 norm_delta=4e-3, scaling=1.0, device=None):
        super().__init__(robot, target_joint_names, target_link_human_indices, device)
        self.origin_link_names = target_origin_link_names
        self.task_link_names = target_task_link_names
        self.huber_delta = huber_delta
        self.norm_delta = norm_delta
        self.scaling = scaling
        self.computed_link_names, origin_idx, task_idx = _link_cache(target_origin_link_names, target_task_link_names)
        self.origin_link_indices = np.array(origin_idx)
        self.task_link_indices = np.array(task_idx)
        self.computed_link_indices = self.get_link_indices(self.computed_link_names)

    def _objective_spec(self) -> ObjectiveSpec:
        hi = np.asarray(self.target_link_human_indices)
        return ObjectiveSpec(N.LOSS_VECTOR, list(self.computed_link_names), [int(i) for i in self.task_link_indices],
                             [int(i) for i in self.origin_link_indices], [int(i) for i in hi[1]], [int(i) for i in hi[0]])

    def _loss_params(self, p):
        p.huber_delta, p.norm_delta, p.scaling = self.huber_delta, self.norm_delta, self.scaling


class DexPilotOptimizer(Optimizer):
    """DexPilot-style retargeting (https://arxiv.org/abs/1910.03135) for 2 to 5 fingers: finger-pair
    vectors are pulled together once the human thumb/finger distance drops below `project_dist` and
    released above `escape_dist`; wrist-to-tip vectors carry a larger weight."""

    retargeting_type = "DEXPILOT"

    def __init__(self, robot: RobotWrapper, target_joint_names: List[str], finger_tip_link_names: List[str],
                 wrist_link_name: str, target_link_human_indices: Optional[np.ndarray] = None, huber_delta=0.03,
                 norm_delta=4e-3, project_dist=0.03, escape_dist=0.05, eta1=1e-4, eta2=3e-2, scaling=1.0, device=None):
        if len(finger_tip_link_names) < 2 or len(finger_tip_link_names) > 5:
            raise ValueError(
                f"DexPilot optimizer can only be applied to hands with 2 to 5 fingers, but got "
                f"{len(finger_tip_link_names)} fingers."
            )
        self.num_fingers = len(finger_tip_link_names)
        origin_link_index, task_link_index = self.generate_link_indices(self.num_fingers)
        if target_link_human_indices is None:
            target_link_human_indices = (np.stack([origin_link_index, task_link_index], axis=0) * 4).astype(int)
        link_names = [wrist_link_name] + list(finger_tip_link_names)
        origin_names = [link_names[i] for i in origin_link_index]
        task_names = [link_names[i] for i in task_link_index]

        super().__init__(robot, target_joint_names, target_link_human_indices, device)
        self.origin_link_names = origin_names
        self.task_link_names = task_names
        self.scaling = scaling
        self.huber_delta = huber_delta
        self.norm_delta = norm_delta
        self.project_dist = project_dist
        self.escape_dist = escape_dist
        self.eta1 = eta1
        self.eta2 = eta2
        self.computed_link_names, origin_idx, task_idx = _link_cache(origin_names, task_names)
        self.origin_link_indices = np.array(origin_idx)
        self.task_link_indices = np.array(task_idx)
        self.computed_link_indices = self.get_link_indices(self.computed_link_names)
        (self.projected, self.s2_project_index_origin, self.s2_project_index_task, self.projected_dist) = (
            self.set_dexpilot_cache(self.num_fingers, eta1, eta2)
        )

    @staticmethod
    def generate_link_indices(num_fingers):
        """
        >>> DexPilotOptimizer.generate_link_indices(4)
        ([2, 3, 4, 3, 4, 4, 0, 0, 0, 0], [1, 1, 1, 2, 2, 3, 1, 2, 3, 4])
        """
        pairs = [(j, i) for i in range(1, num_fingers) for j in range(i + 1, num_fingers + 1)]
        pairs += [(0, i) for i in range(1, num_fingers + 1)]  # wrist (0) -> every finger tip
        return [o for o, _ in pairs], [t for _, t in pairs]

    @staticmethod
    def set_dexpilot_cache(num_fingers, eta1, eta2):
        """
        >>> DexPilotOptimizer.set_dexpilot_cache(4, 0.1, 0.2)
        (array([False, False, False, False, False, False]), [1, 2, 2], [0, 0, 1], array([0.1, 0.1, 0.1, 0.2, 0.2, 0.2]))
        """
        n_s1 = num_fingers - 1
        s2 = [(j, i) for i in range(0, num_fingers - 2) for j in range(i + 1, num_fingers - 1)]
        projected = np.zeros(n_s1 + len(s2), dtype=bool)
        projected_dist = np.array([eta1] * n_s1 + [eta2] * len(s2))
        return projected, [o for o, _ in s2], [t for _, t in s2], projected_dist

    def _objective_spec(self) -> ObjectiveSpec:
        hi = np.asarray(self.target_link_human_indices)
        len_proj = len(self.projected)
        len_s2 = len(self.s2_project_index_task)
        return ObjectiveSpec(
            N.LOSS_DEXPILOT, list(self.computed_link_names), [int(i) for i in self.task_link_indices],
            [int(i) for i in self.origin_link_indices], [int(i) for i in hi[1]], [int(i) for i in hi[0]],
            num_fingers=self.num_fingers, len_proj=len_proj, len_s1=len_proj - len_s2,
            s2_origin=list(self.s2_project_index_origin), s2_task=list(self.s2_project_index_task),
        )

    def _loss_params(self, p):
        p.huber_delta, p.norm_delta, p.scaling = self.huber_delta, self.norm_delta, self.scaling
        p.project_dist, p.escape_dist, p.eta1, p.eta2 = self.project_dist, self.escape_dist, self.eta1, self.eta2

    def retarget(self, ref_value, fixed_qpos, last_qpos, damping=None):
        if len(fixed_qpos) != len(self.idx_pin2fixed):
            raise ValueError(
                f"Optimizer has {len(self.idx_pin2fixed)} joints but non_target_qpos {fixed_qpos} is given"
            )
        flags = np.ascontiguousarray(self.projected, dtype=np.uint8)[None]  # hysteresis state, updated in place
        qpos, _ = self._solve_host(np.asarray(ref_value, dtype=np.float32)[None], np.asarray(fixed_qpos, dtype=np.float32)[None],
                                   np.asarray(last_qpos, dtype=np.float32)[None], clip_init=False, projected=flags, damping=damping)
        self.projected = flags[0].astype(bool)
        return qpos[0]
