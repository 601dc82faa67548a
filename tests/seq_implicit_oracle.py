"""Float64 reference of the stream backward pass (TEST INFRASTRUCTURE): tests/implicit_oracle.py's per-frame implicit gradient
chained through time with the low-pass filter and mimic adjoints in numpy.

Per stream, backwards over t: ybar += Ybar_t; qbar_t = alpha ybar and ybar *= 1 - alpha if the filter was initialised before
step t (else qbar_t = ybar, ybar = 0); xbar_t = M^T qbar_t + carry with M = dq/dx (scatter + mimic, fixed joints dropped);
implicit_grad at x*_t with the anchor clip32(x*_{t-1}) (x*_{-1}: the entry last_qpos) and the flags step t applied (replayed
from the entry flags) gives dl/dkp_t and the anchor adjoint, which is the next carry.  Shares nothing with the kernel but the
definitions: M comes from the adaptor (oracle), the flags from OracleOptimizer.prepare."""
import numpy as np

from implicit_oracle import implicit_grad, keypoint_grad, post_flags


def compose64(o, x, fixed=None):
    """Robot qpos (pinocchio order) of the optimised joints x: scatter, fixed joints, mimic (the oracle's adaptor)."""
    q = np.zeros(o.robot.dof)
    q[o.idx_pin2target] = x
    if fixed is not None and len(o.idx_pin2fixed):
        q[o.idx_pin2fixed] = fixed
    return o.adaptor.forward_qpos(q) if o.adaptor is not None else q


def mimic_matrix(o):
    """M = dq/dx [dof, n] (compose64 is affine: columns of differences)."""
    n = len(o.idx_pin2target)
    q0 = compose64(o, np.zeros(n))
    return np.stack([compose64(o, np.eye(n)[i]) - q0 for i in range(n)], 1)


def at_bounds64(o, x):
    """A float32 trace row in float64, with the joints the solver holds at a (float32) bound put exactly on the float64 bound,
    so that the reference sees the kernel's active set."""
    x32 = np.asarray(x, np.float32)
    x64 = x32.astype(np.float64)
    x64 = np.where(x32 == o.lower.astype(np.float32), o.lower, x64)
    return np.where(x32 == o.upper.astype(np.float32), o.upper, x64)


def replay_flags(o, refs, flags0):
    """The DexPilot flags each step applies, from the entry flags [len_proj] over refs [T,m,3]."""
    out, f = [], np.asarray(flags0, bool)
    for r in refs:
        f = post_flags(o, r, f)
        out.append(f.copy())
    return np.array(out)


def seq_grad(o, kp, x, last0, gy, g_last_out=None, g_fs_out=None, flags0=None, finit0=False, alpha=-1.0):
    """kp [T,21,3], trace x [T,n] (float32 values), entry last_qpos [n], upstream gy [T,dof] (+ exit last_qpos [n] and exit
    filter_state [dof]).  Returns (dl/dkp [T,21,3], dl/d entry last_qpos [n], dl/d entry filter_state [dof], flags [T,len_proj])."""
    T, n = x.shape
    dof = o.robot.dof
    M = mimic_matrix(o)
    refs = np.array([o.ref_from_keypoints(k) for k in kp], np.float32)
    flags = replay_flags(o, refs, flags0 if flags0 is not None else np.zeros(len(o.projected), bool)) \
        if o.type == "dexpilot" else [None] * T
    use_filter = 0.0 <= alpha <= 1.0
    ybar = np.zeros(dof) if g_fs_out is None else np.asarray(g_fs_out, np.float64).copy()
    carry = np.zeros(n) if g_last_out is None else np.asarray(g_last_out, np.float64).copy()
    gkp = np.zeros((T, 21, 3))
    for t in range(T - 1, -1, -1):
        Y = np.asarray(gy[t], np.float64)
        if use_filter:
            ybar = ybar + Y
            if t > 0 or finit0:
                qbar, ybar = alpha * ybar, (1 - alpha) * ybar
            else:
                qbar, ybar = ybar, np.zeros(dof)
        else:
            qbar = Y
        xbar = M.T @ qbar + carry
        last = x[t - 1] if t > 0 else last0
        rb, ab, _, _ = implicit_grad(o, refs[t], np.zeros(0), last, at_bounds64(o, x[t]), xbar, flags=flags[t], clip_init=True)
        gkp[t] = keypoint_grad(o, rb)
        carry = ab
    return gkp, carry, (ybar if use_filter else ybar), (np.array(flags) if o.type == "dexpilot" else None)
