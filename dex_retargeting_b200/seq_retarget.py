"""Sequence wrapper: temporal state around the optimizer.

Drop-in for `dex_retargeting.seq_retarget.SeqRetargeting` (reference:
src/dex_retargeting/seq_retarget.py:12-161): `retarget()` clips the previous solution to the joint
limits, solves, keeps the UNFILTERED solution as the next warm start, scatters it into the full
pinocchio-ordered qpos, applies mimic joints and the low-pass filter, returns float64 (robot.dof,).

New, batched: `retarget_sequences()` runs S independent streams x T frames with exactly that recurrence
inside ONE kernel launch (`dexr_solve_sequences`): a group of lanes owns a stream and walks its frames,
`last_qpos`, the DexPilot hysteresis flags and the filter state never leave the SM between frames.
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _native as N
from .constants import OPERATOR2MANO, HandType
from .optimizer import Optimizer
from .optimizer_utils import LPFilter
from .urdf import DUMMY_JOINT_NAMES


@dataclass
class StreamState:
    """Device-resident state of S streams (torch tensors); resumable / checkpointable."""

    last_qpos: "torch.Tensor"     # [S, opt_dof] float32, unfiltered previous solution
    filter_state: "torch.Tensor"  # [S, dof] float32
    filter_init: "torch.Tensor"   # [S] uint8
    projected: Optional["torch.Tensor"]  # [S, len_proj] uint8 (DexPilot) or None
    damping: Optional["torch.Tensor"] = None  # [S] float32: the solver's carried damping (dexr_sequences_t.damping_state)

    _FIELDS = ("last_qpos", "filter_state", "filter_init", "projected", "damping")

    def state_dict(self) -> dict:
        """Host copies of every tensor (None stays None): what a checkpoint of S running streams has to hold.  A run resumed
        from it continues bit-identically (the state is complete: tests/test_gpu_parity.py splits a call in two)."""
        return {k: (None if getattr(self, k) is None else getattr(self, k).detach().cpu().clone()) for k in self._FIELDS}

    @classmethod
    def from_state_dict(cls, state: dict, device=None) -> "StreamState":
        """Inverse of `state_dict` (tensors moved to `device`); a checkpoint written before `damping` existed resumes with the
        solver's default damping."""
        import torch

        missing = [k for k in cls._FIELDS[:3] if state.get(k) is None]
        if missing:
            raise ValueError(f"stream state checkpoint lacks {missing}")
        S = int(state["last_qpos"].shape[0])
        for k in cls._FIELDS[1:]:
            t = state.get(k)
            if t is not None and int(t.shape[0]) != S:
                raise ValueError(f"stream state checkpoint: {k} holds {int(t.shape[0])} streams, last_qpos {S}")

        def put(t):
            return None if t is None else torch.as_tensor(t).to(device if device is not None else t.device).contiguous()

        st = cls(**{k: put(state.get(k)) for k in cls._FIELDS})
        if st.damping is None:
            st.damping = torch.zeros((S,), dtype=torch.float32, device=st.last_qpos.device)
        return st


def _quat_to_matrix(q):
    w, x, y, z = (float(v) for v in q)
    n = (w * w + x * x + y * y + z * z) ** 0.5
    w, x, y, z = w / n, x / n, y / n, z / n
    return np.array([
        [1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
        [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
        [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)],
    ])


def _intrinsic_xyz_from_matrix(R):
    """Angles (a, b, c) with R = Rx(a) Ry(b) Rz(c) (intrinsic x-y'-z'')."""
    sb = float(np.clip(R[0, 2], -1.0, 1.0))
    b = np.arcsin(sb)
    if abs(sb) < 1 - 1e-10:
        a = np.arctan2(-R[1, 2], R[2, 2])
        c = np.arctan2(-R[0, 1], R[0, 0])
    else:  # gimbal lock: put everything into the first angle
        a = np.arctan2(R[2, 1], R[1, 1])
        c = 0.0
    return np.array([a, b, c])


class SeqRetargeting:
    def __init__(self, optimizer: Optimizer, has_joint_limits=True, lp_filter: Optional[LPFilter] = None):
        self.optimizer = optimizer
        robot = optimizer.robot

        self.has_joint_limits = has_joint_limits
        joint_limits = np.ones_like(robot.joint_limits)
        joint_limits[:, 0] = -1e4  # a large value is equivalent to no limit
        joint_limits[:, 1] = 1e4
        if has_joint_limits:
            joint_limits[:] = robot.joint_limits[:]
            optimizer.set_joint_limit(joint_limits[optimizer.idx_pin2target])
        self.joint_limits = joint_limits[optimizer.idx_pin2target]

        self.last_qpos = joint_limits.mean(1)[optimizer.idx_pin2target].astype(np.float32)
        self._damping = np.zeros(1, dtype=np.float32)  # the stream's carried solver damping (Optimizer.retarget, `damping`)
        self.accumulated_time = 0
        self.num_retargeting = 0
        self.filter = lp_filter
        self.is_warm_started = False
        self.last_grad_status = None  # int32 [S,T] DEXR_GRAD_STATUS_* words of the most recent retarget_sequences backward pass

    # ------------------------------------------------------------------------------ single stream
    def warm_start(self, wrist_pos: np.ndarray, wrist_quat: np.ndarray, hand_type: HandType = HandType.right,
                   is_mano_convention: bool = False):
        """Analytic initialisation of the 6 dummy free joints from a wrist pose (position retargeting
        with a flying hand; seq_retarget.py:45-110).  wrist_quat is (w, x, y, z)."""
        if len(wrist_pos) != 3:
            raise ValueError(f"Wrist pos: {wrist_pos} is not a 3-dim vector.")
        if len(wrist_quat) != 4:
            raise ValueError(f"Wrist quat: {wrist_quat} is not a 4-dim vector.")
        operator2mano = OPERATOR2MANO[hand_type] if is_mano_convention else np.eye(3)
        robot = self.optimizer.robot
        target_wrist_pose = np.eye(4)
        target_wrist_pose[:3, :3] = _quat_to_matrix(wrist_quat) @ operator2mano.T
        target_wrist_pose[:3, 3] = wrist_pos

        wrist_link_id = robot.get_joint_parent_child_frames(DUMMY_JOINT_NAMES[5])[1]
        qpos = robot.q0.copy()
        for num, name in enumerate(self.optimizer.target_joint_names):
            if name in DUMMY_JOINT_NAMES:
                qpos[num] = 0
        robot.compute_forward_kinematics(qpos)
        root2wrist = robot.get_link_pose_inv(wrist_link_id)
        target_root_pose = target_wrist_pose @ root2wrist
        pose_vec = np.concatenate([target_root_pose[:3, 3], _intrinsic_xyz_from_matrix(target_root_pose[:3, :3])])
        for num, name in enumerate(self.optimizer.target_joint_names):
            if name in DUMMY_JOINT_NAMES:
                self.last_qpos[num] = pose_vec[DUMMY_JOINT_NAMES.index(name)]
        self.is_warm_started = True

    def warm_start_batch(self, last_qpos, wrist_pos, wrist_quat, hand_type: HandType = HandType.right,
                         is_mano_convention: bool = False):
        """Batched `warm_start` (seq_retarget.py:45-110) for S streams: writes the analytic 6-D dummy-joint
        pose into `last_qpos` [S, opt_dof] (a torch tensor on any device, e.g. `StreamState.last_qpos`) from
        wrist positions [S,3] and quaternions [S,4] (w, x, y, z).  Pure tensor algebra, no host round trip."""
        import torch

        if wrist_pos.shape[-1] != 3 or wrist_quat.shape[-1] != 4:
            raise ValueError("wrist_pos must be [S,3] and wrist_quat [S,4]")
        robot = self.optimizer.robot
        names = self.optimizer.target_joint_names
        cols = [names.index(n) if n in names else -1 for n in DUMMY_JOINT_NAMES]
        if min(cols) < 0:
            raise ValueError("warm_start needs the 6 dummy free joints among the optimised joints")
        dt, dev = last_qpos.dtype, last_qpos.device
        # constant of the robot: root -> wrist transform with the dummy joints at zero
        qpos = robot.q0.copy()
        for num, name in enumerate(names):
            if name in DUMMY_JOINT_NAMES:
                qpos[num] = 0
        robot.compute_forward_kinematics(qpos)
        wrist_link_id = robot.get_joint_parent_child_frames(DUMMY_JOINT_NAMES[5])[1]
        root2wrist = torch.as_tensor(robot.get_link_pose_inv(wrist_link_id), dtype=torch.float64, device=dev)
        o2m = torch.as_tensor(OPERATOR2MANO[hand_type] if is_mano_convention else np.eye(3), dtype=torch.float64, device=dev)
        q = wrist_quat.to(torch.float64)
        q = q / q.norm(dim=-1, keepdim=True)
        w, x, y, z = q.unbind(-1)
        Rw = torch.stack([
            torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], -1),
            torch.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], -1),
            torch.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1)], -2) @ o2m.T
        R = Rw @ root2wrist[:3, :3]
        t = (Rw @ root2wrist[:3, 3]) + wrist_pos.to(torch.float64)
        sb = R[..., 0, 2].clamp(-1.0, 1.0)
        b = torch.asin(sb)
        regular = sb.abs() < 1 - 1e-10
        a = torch.where(regular, torch.atan2(-R[..., 1, 2], R[..., 2, 2]), torch.atan2(R[..., 2, 1], R[..., 1, 1]))
        c = torch.where(regular, torch.atan2(-R[..., 0, 1], R[..., 0, 0]), torch.zeros_like(b))
        pose = torch.cat([t, torch.stack([a, b, c], -1)], dim=-1).to(dt)
        last_qpos[:, cols] = pose
        self.is_warm_started = True
        return last_qpos

    def retarget(self, ref_value, fixed_qpos=np.array([])):
        tic = time.perf_counter()
        qpos = self.optimizer.retarget(
            ref_value=np.asarray(ref_value).astype(np.float32),
            fixed_qpos=np.asarray(fixed_qpos).astype(np.float32),
            last_qpos=np.clip(self.last_qpos, self.joint_limits[:, 0], self.joint_limits[:, 1]),
            damping=self._damping,
        )
        self.accumulated_time += time.perf_counter() - tic
        self.num_retargeting += 1
        self.last_qpos = qpos
        robot_qpos = np.zeros(self.optimizer.robot.dof)
        robot_qpos[self.optimizer.idx_pin2fixed] = fixed_qpos
        robot_qpos[self.optimizer.idx_pin2target] = qpos
        if self.optimizer.adaptor is not None:
            robot_qpos = self.optimizer.adaptor.forward_qpos(robot_qpos)
        if self.filter is not None:
            robot_qpos = self.filter.next(robot_qpos)
        return robot_qpos

    def set_qpos(self, robot_qpos: np.ndarray):
        self.last_qpos = np.asarray(robot_qpos)[self.optimizer.idx_pin2target]
        self._damping[:] = 0  # a new warm start: the solver's default damping again

    def get_qpos(self, fixed_qpos: Optional[np.ndarray] = None):
        robot_qpos = np.zeros(self.optimizer.robot.dof)
        robot_qpos[self.optimizer.idx_pin2target] = self.last_qpos
        if fixed_qpos is not None:
            robot_qpos[self.optimizer.idx_pin2fixed] = fixed_qpos
        return robot_qpos

    def verbose(self):
        print(f"Retargeting {self.num_retargeting} times takes: {self.accumulated_time}s")
        print(f"Last distance: {self.optimizer.opt.last_optimum_value()}")

    def reset(self):
        self.last_qpos = self.joint_limits.mean(1).astype(np.float32)
        self._damping[:] = 0
        self.num_retargeting = 0
        self.accumulated_time = 0

    @property
    def joint_names(self):
        return self.optimizer.robot.dof_joint_names

    # ------------------------------------------------------------------------------ batched streams
    @property
    def low_pass_alpha(self) -> float:
        return float(self.filter.alpha) if self.filter is not None else -1.0

    def make_stream_state(self, num_streams: int) -> StreamState:
        """Initial state of S fresh streams: mid-range warm start (seq_retarget.py:33-35), filter not
        initialised, no DexPilot projection."""
        import torch

        opt = self.optimizer
        dev = torch.device("cuda", opt.device_index)
        last = torch.from_numpy(np.ascontiguousarray(self.joint_limits.mean(1), dtype=np.float32)).to(dev)
        len_proj = opt._objective_spec().len_proj
        return StreamState(
            last_qpos=last[None].repeat(num_streams, 1).contiguous(),
            filter_state=torch.zeros((num_streams, opt.robot.dof), dtype=torch.float32, device=dev),
            filter_init=torch.zeros((num_streams,), dtype=torch.uint8, device=dev),
            projected=torch.zeros((num_streams, len_proj), dtype=torch.uint8, device=dev) if len_proj else None,
            damping=torch.zeros((num_streams,), dtype=torch.float32, device=dev),
        )

    def retarget_sequences(self, keypoints, state: Optional[StreamState] = None, fixed_qpos=None, out=None,
                           status_out=None, stream=None, raw_hand=None):
        """keypoints: float32 CUDA tensor [S,T,21,3] (raw 21-point hand frames).  Runs every stream
        through T SeqRetargeting.retarget() steps in one launch.  Returns (robot_qpos [S,T,dof] float32
        in pinocchio joint order, filtered; state) -- `state` is updated in place and can be passed
        to the next call to continue the streams.  `raw_hand` (HandType): the keypoints are raw detector landmarks of that
        hand, pre-processed inside the kernel (Optimizer.params).

        Autograd: when grad mode is on and `keypoints`, `state.last_qpos` or `state.filter_state` requires grad, the result
        carries a `grad_fn` whose backward walks every stream back in time (dex_retargeting_b200/grad.py: the implicit gradient
        of each step's minimiser, chained through the warm-start anchor, the mimic fold and the low-pass filter).  The forward
        results and exit state are the same bits as without autograd.  On that route `state.last_qpos` and
        `state.filter_state` are REBOUND to new tensors (the exit state, part of the graph) instead of being written in place,
        so a state passed to the next call carries the graph through the whole video, and `.detach()` on them truncates it;
        `filter_init`, `projected` and `damping` are still updated in place.  The route refuses `out=`, `raw_hand` and a
        `fixed_qpos` that requires grad; the [S,T] status words of the last backward pass are left in `last_grad_status`."""
        import torch

        if keypoints.dim() != 4 or tuple(keypoints.shape[2:]) != (N.NUM_KEYPOINTS, 3):
            raise ValueError(f"keypoints must have shape [S,T,21,3], got {tuple(keypoints.shape)}")
        S, T = int(keypoints.shape[0]), int(keypoints.shape[1])
        if state is None:
            state = self.make_stream_state(S)
        if torch.is_grad_enabled() and any(t is not None and t.requires_grad
                                           for t in (keypoints, state.last_qpos, state.filter_state)):
            from .grad import retarget_sequences_autograd

            return retarget_sequences_autograd(self, keypoints, state, fixed_qpos=fixed_qpos, out=out, status_out=status_out,
                                               stream=stream, raw_hand=raw_hand)
        dev = torch.device("cuda", self.optimizer.device_index)
        if out is None:
            out = torch.empty((S, T, self.optimizer.robot.dof), dtype=torch.float32, device=dev)
        self._launch_sequences(keypoints, state, fixed_qpos, out, status_out, stream, lp_alpha=self.low_pass_alpha,
                               raw_hand=raw_hand)
        return out, state

    def _launch_sequences(self, keypoints, state, fixed_qpos, out, status_out, stream, lp_alpha, raw_hand=None, last_qpos=None,
                          filter_state=None):
        """The one `dexr_solve_sequences` launch.  `last_qpos` / `filter_state`: the state buffers written in place (default:
        the state's own)."""
        import torch

        opt = self.optimizer
        eng = opt.engine()
        dev = torch.device("cuda", eng.device)
        S, T = int(keypoints.shape[0]), int(keypoints.shape[1])
        last_qpos = state.last_qpos if last_qpos is None else last_qpos
        filter_state = state.filter_state if filter_state is None else filter_state

        def chk(t, shape, dtype, name):
            if t.device != dev or t.dtype != dtype or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
                raise ValueError(f"{name}: expected contiguous {dtype} tensor of shape {tuple(shape)} on {dev}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")
            return t.data_ptr()

        io = N.DexrSequences()
        io.keypoints = chk(keypoints, (S, T, N.NUM_KEYPOINTS, 3), torch.float32, "keypoints")
        nf = len(opt.idx_pin2fixed)
        if nf:
            if fixed_qpos is None:
                raise ValueError(f"Optimizer has {nf} joints but no fixed_qpos is given")
            io.fixed_qpos = chk(fixed_qpos, (S, T, nf), torch.float32, "fixed_qpos")
        io.last_qpos = chk(last_qpos, (S, opt.opt_dof), torch.float32, "state.last_qpos")
        io.filter_state = chk(filter_state, (S, opt.robot.dof), torch.float32, "state.filter_state")
        io.filter_init = chk(state.filter_init, (S,), torch.uint8, "state.filter_init")
        if state.projected is not None:
            io.projected = chk(state.projected, (S, state.projected.shape[1]), torch.uint8, "state.projected")
        if state.damping is not None:
            io.damping_state = chk(state.damping, (S,), torch.float32, "state.damping")
        io.robot_qpos_out = chk(out, (S, T, opt.robot.dof), torch.float32, "out")
        if status_out is not None:
            io.status_out = chk(status_out, (S, T), torch.int32, "status_out")
        s = stream if stream is not None else torch.cuda.current_stream(dev)
        p = opt.params(clip_init=True, lp_alpha=lp_alpha, raw_hand=raw_hand)
        N.check(eng.lib.dexr_solve_sequences(eng.handle, C.byref(p), C.byref(io), S, T, C.c_void_p(s.cuda_stream)),
                "dexr_solve_sequences")
