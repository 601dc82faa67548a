"""Writes tests/golden/grad_seq_vectors.npz: float64 oracle traces of short streams and their reference gradients
(tests/seq_implicit_oracle.py), for the stream backward pass (dexr_grad_sequences).

Per workload tag: S streams of T steps from tools/workloads.streams (the recorded trajectory, per-stream 2 mm offsets), solved by
the float64 converged oracle (OracleSeqRetargeting's recurrence: clipped warm start, unfiltered solution carried, DexPilot flags
carried; each solution rounded to float32 as the stream passes it on), seeded upstream gradients on all three outputs.
  leap_dexpilot     config 4's hand (LEAP DexPilot, 16 lanes), its filter, a window where the flags switch
  allegro           Allegro vector with the filter; the last stream enters with a warm start outside the joint limits
  allegro_nofilter  the same streams without the filter
  allegro_finit     the filter initialised at entry
  ability           a mimic hand (Ability vector, filter)
  shadow            a 32-lane hand (Shadow teleop vector, filter)
Stored: keys, alpha, entry last_qpos / flags / filter_init, trace x [S,T,n], forward status, upstream gradients, reference
gradients (keypoints [S,T,21,3], entry last_qpos [S,n], entry filter_state [S,dof]) and the replayed flags [S,T,len_proj].

Usage: python tests/tools/gen_grad_seq_vectors.py
"""
import multiprocessing as mp
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
import workloads as W  # noqa: E402

S, T = 8, 12
SEED = 2031
# tag: (config key, alpha override or None, filter_init at entry, stream seed, first frame of the trajectory)
CASES = {
    # frames 248..259 of config 4's streams: the DexPilot flags switch at frames 252-258
    "leap_dexpilot": (W.LEAP_DEXPILOT_KEY, None, False, W.STREAM_SEED, 248),
    "allegro": ("teleop/allegro_hand_right", None, False, W.STREAM_SEED + 1, 0),
    "allegro_nofilter": ("teleop/allegro_hand_right", -1.0, False, W.STREAM_SEED + 1, 0),
    "allegro_finit": ("teleop/allegro_hand_right", None, True, W.STREAM_SEED + 1, 0),
    "ability": ("teleop/ability_hand_right", None, False, W.STREAM_SEED + 2, 0),
    "shadow": ("teleop/shadow_hand_right", None, False, W.STREAM_SEED + 3, 0),
}


def oracle_stream(o, kp, last0, flags0):
    """Trace x [T,n] float32 of one stream (float64 converged solves, OracleSeqRetargeting's recurrence)."""
    from implicit_oracle import clip32
    from oracle.solvers import solve_converged

    if o.type == "dexpilot":
        o.projected[:] = flags0
    last, xs = np.asarray(last0, np.float32), []
    for t in range(len(kp)):
        ref = o.ref_from_keypoints(kp[t])
        x, _, _ = solve_converged(o, ref, np.zeros(0), clip32(o, last).astype(np.float32), update_state=True)
        last = x.astype(np.float32)
        xs.append(last)
    return np.array(xs)


def _one(args):
    from helpers import build_oracle
    from seq_implicit_oracle import seq_grad

    key, kp, last0, gy, gl, gf, finit, alpha = args
    o = build_oracle(key)
    flags0 = np.zeros(len(o.projected), bool) if o.type == "dexpilot" else None
    x = oracle_stream(o, kp, last0, flags0)
    gkp, glast, gfs, flags = seq_grad(o, kp, x, last0, gy, gl, gf, flags0=flags0, finit0=finit, alpha=alpha)
    return x, gkp, glast, gfs, (flags if flags is not None else np.zeros((len(kp), 0), bool))


def case(pool, key, alpha, finit, seed, first):
    seq = W.build(key)
    opt = seq.optimizer
    a = seq.low_pass_alpha if alpha is None else alpha
    kp = np.ascontiguousarray(W.streams(S, first + T, seed=seed)[:, first:])
    last0 = np.tile(seq.joint_limits.mean(1).astype(np.float32), (S, 1))
    if key.startswith("teleop/allegro"):  # the last stream's entry warm start lies outside the limits: clipped anchor at t = 0
        span = (seq.joint_limits[:, 1] - seq.joint_limits[:, 0]).astype(np.float32)
        last0[-1, ::3] = seq.joint_limits[::3, 1] + 0.3 * span[::3]
    rng = np.random.RandomState(seed + SEED)
    n, dof = opt.opt_dof, opt.robot.dof
    gy = rng.randn(S, T, dof).astype(np.float32)
    gl = rng.randn(S, n).astype(np.float32)
    gf = rng.randn(S, dof).astype(np.float32)
    parts = pool.map(_one, [(key, kp[s], last0[s], gy[s], gl[s], gf[s], finit, a) for s in range(S)])
    x, gkp, glast, gfs, flags = (np.array([p[i] for p in parts]) for i in range(5))
    return dict(key=np.array(key), alpha=np.array(a, np.float32), keypoints=kp, last_qpos=last0,
                filter_init=np.full(S, int(finit), np.uint8), x=x.astype(np.float32), grad_robot_qpos=gy, grad_last_qpos_out=gl,
                grad_filter_state_out=gf, grad_keypoints=gkp.astype(np.float32), grad_last_qpos=glast.astype(np.float32),
                grad_filter_state=gfs.astype(np.float32), flags=flags.astype(np.uint8))


def main():
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    dst = ROOT / "tests" / "golden" / "grad_seq_vectors.npz"
    out = {}
    t0 = time.time()
    with mp.get_context("fork").Pool(8) as pool:
        for tag, (key, alpha, finit, seed, first) in CASES.items():
            rec = case(pool, key, alpha, finit, seed, first)
            for k, v in rec.items():
                out[f"{tag}/{k}"] = v
            print(f"{tag}: {S} x {T}, alpha {float(rec['alpha'])}, {time.time() - t0:.0f} s", flush=True)
    np.savez_compressed(dst, **out)
    print("wrote", dst, dst.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
