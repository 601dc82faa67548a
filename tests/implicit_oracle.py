"""Float64 reference of the implicit-function gradient of a frame's minimiser (TEST INFRASTRUCTURE).

At a minimiser x of F(x; t, a) on the box, with the upstream gradient gbar:
    free joints F = not (x at lower with g > 0 or x at upper with g < 0)     (the rule of oracle.solvers.polish)
    H_FF v_F = gbar_F, v = 0 elsewhere                                       (H: oracle.solvers._ggn_hessian, the exact Hessian)
    theta_bar = -(dg/dtheta)_F^T v_F
The mixed partials dg/dtheta are taken by CENTRAL DIFFERENCES -- of FrameObjective.value_and_grad w.r.t. the target array and
the anchor, and of a float64 restatement of OracleOptimizer.prepare w.r.t. ref_value with the DexPilot flags frozen (prepare
itself rounds DexPilot targets to float32, which finite differences cannot see through) -- so this derivation shares nothing
with the kernel's analytic one (dexr_grad_kernels.cuh) but the Hessian's definition.
"""
import numpy as np

from oracle.solvers import _ggn_hessian


def targets64(o, ref_value, flags):
    """OracleOptimizer.prepare in float64 with the DexPilot flags given (post-update, held fixed): (targets [m,3], weights)."""
    ref_value = np.asarray(ref_value, np.float64)
    if o.type == "position":
        return ref_value.copy(), None
    if o.type == "vector":
        return ref_value * o.scaling, np.ones(o.m)
    len_proj = len(o.projected)
    len_s1 = len_proj - len(o.s2_task)
    proj = np.asarray(flags, bool)
    dist = np.linalg.norm(ref_value[:len_proj], axis=1)
    w = np.where(proj, np.array([200.0] * len_s1 + [400.0] * (len_proj - len_s1)), 1.0)
    w = np.concatenate([w, np.full(o.num_fingers, float(len_proj + o.num_fingers))])
    ref = ref_value * o.scaling
    pv = ref_value[:len_proj] / (dist[:, None] + 1e-6) * o.projected_dist[:, None]
    ref[:len_proj] = np.where(proj[:, None], pv, ref[:len_proj])
    return ref, w


def clip32(o, last_qpos):
    """SeqRetargeting's warm-start clip with the limits rounded to float32 (as the robot table holds them), float64 out."""
    lim = o.joint_limits.astype(np.float32)
    return np.clip(np.asarray(last_qpos, np.float32), lim[:, 0], lim[:, 1]).astype(np.float64)


def post_flags(o, ref_value, flags_in):
    """The DexPilot flags a frame applies (prepare's hysteresis update from `flags_in`)."""
    saved = o.projected.copy()
    o.projected[:] = np.asarray(flags_in, bool)
    o.prepare(np.asarray(ref_value, np.float32), update_state=True)
    out = o.projected.copy()
    o.projected[:] = saved
    return out


def implicit_grad(o, ref_value, fixed_qpos, last_qpos, x, gbar, flags=None, clip_init=False, h=1e-6):
    """dl/dref_value [m,3], dl/dlast_qpos [n], free mask [n], cond(H_FF) at the minimiser x.  `flags`: DexPilot flags after
    the frame (None: derived from the distances alone, as for a frame without carried flags)."""
    if o.type == "dexpilot" and flags is None:
        flags = post_flags(o, ref_value, np.zeros(len(o.projected), bool))
    x = np.asarray(x, np.float64)
    last = np.asarray(last_qpos, np.float32).astype(np.float64)
    # the clip limits are float32 table values: a warm start ON a limit is left alone (gradient passes), as in the solver
    anchor = clip32(o, last) if clip_init else last
    ref = np.asarray(ref_value, np.float64)
    target, weights = targets64(o, ref, flags)
    obj = o.make_objective(np.asarray(ref_value, np.float32), fixed_qpos, anchor, update_state=False)
    obj.target, obj.weights, obj.last = target, weights, anchor

    def grad_at(target_=None, last_=None):
        saved = obj.target, obj.last
        if target_ is not None:
            obj.target = target_
        if last_ is not None:
            obj.last = last_
        g = obj.value_and_grad(x)[1]
        obj.target, obj.last = saved
        return g

    g = grad_at()
    act = ((x <= o.lower) & (g > 0)) | ((x >= o.upper) & (g < 0))
    free = ~act
    H = _ggn_hessian(obj, x)
    Hff = H[np.ix_(free, free)]
    v = np.zeros_like(x)
    v[free] = np.linalg.solve(Hff, np.asarray(gbar, np.float64)[free])
    cond = float(np.linalg.cond(Hff)) if free.any() else 1.0

    # dg/dtarget by central differences, then the chain through t(ref) (also central differences, flags frozen)
    m = target.shape[0]
    tbar = np.zeros((m, 3))
    for k in range(m):
        for c in range(3):
            tp, tm = target.copy(), target.copy()
            tp[k, c] += h
            tm[k, c] -= h
            dg = (grad_at(target_=tp) - grad_at(target_=tm)) / (2 * h)
            tbar[k, c] = -dg @ v
    rbar = np.zeros((m, 3))
    for k in range(m):
        for c in range(3):
            rp, rm = ref.copy(), ref.copy()
            rp[k, c] += h
            rm[k, c] -= h
            dt = (targets64(o, rp, flags)[0] - targets64(o, rm, flags)[0]) / (2 * h)
            rbar[k, c] = (dt * tbar).sum()
    # anchor: dg/da by central differences; clip_init passes the gradient only where the clip left the warm start alone
    abar = np.zeros_like(x)
    for i in range(len(x)):
        ap, am = anchor.copy(), anchor.copy()
        ap[i] += h
        am[i] -= h
        abar[i] = -((grad_at(last_=ap) - grad_at(last_=am)) / (2 * h)) @ v
    if clip_init:
        abar = np.where(anchor == last, abar, 0.0)
    return rbar, abar, free, cond


def keypoint_grad(o, rbar):
    """Adjoint of the keypoint gather ref_from_keypoints: [m,3] -> [21,3]."""
    out = np.zeros((21, 3))
    idx = np.asarray(o.target_link_human_indices)
    if o.type == "position":
        np.add.at(out, idx.reshape(-1), rbar)
    else:
        np.add.at(out, idx[1], rbar)
        np.add.at(out, idx[0], -rbar)
    return out
