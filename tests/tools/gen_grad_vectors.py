"""Writes tests/golden/grad_vectors.npz: float64 implicit-function gradients (tests/implicit_oracle.py) of the oracle minimisers
of bench frames, for the backward pass of retarget_batch (dexr_grad_frames).

Per workload tag, the first N frames that tools/workloads.py regenerates from its seeds (the same frames as
tests/golden/bench_parity.npz, whose minimisers are polished to float64 here):
  metric         Vector Allegro right (16 lanes)                      shadow_narrow  Position Shadow, free-flying base (32 lanes)
  leap_frames    DexPilot LEAP right (flags start cleared)           mixed/<robot>  the six teleop vector hands (mimic: Ability, SVH, Inspire)
  metric_clip    the cold-start Allegro frames solved with clip_init (the anchor is the warm start clipped to the joint limits)
Stored: digest of the inputs, seeded upstream gradient gbar [N,n], oracle minimiser x [N,n], gradients w.r.t. keypoints
[N,21,3], ref_value [N,m,3] and last_qpos [N,n], free-joint mask [N,n], cond(H_FF) [N], DexPilot flags after the frame.

Usage: python tests/tools/gen_grad_vectors.py [N]
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

GBAR_SEED = 2024
_O = {}


def _oracle(key):
    if key not in _O:
        from helpers import build_oracle

        _O[key] = build_oracle(key)
    return _O[key]


def _grad_chunk(args):
    from implicit_oracle import clip32, implicit_grad, keypoint_grad, post_flags
    from oracle.solvers import polish, solve_converged

    key, kp, x0, fixed, xs, gbar, clip = args
    o = _oracle(key)
    rec = {k: [] for k in ("x", "grad_keypoints", "grad_ref_value", "grad_last_qpos", "free", "cond", "flags")}
    for i in range(kp.shape[0]):
        if o.type == "dexpilot":
            o.projected[:] = False
        ref = o.ref_from_keypoints(kp[i])
        fx = fixed[i] if fixed is not None else np.zeros(0)
        anchor = clip32(o, x0[i]).astype(np.float32) if clip else x0[i]
        if xs is None:
            x, _, _ = solve_converged(o, ref, fx, anchor, update_state=False)
        else:
            x, _ = polish(o.make_objective(ref, fx, anchor, update_state=False), xs[i].astype(np.float64), o.lower, o.upper)
        flags = post_flags(o, ref, np.zeros(len(o.projected), bool)) if o.type == "dexpilot" else np.zeros(0, bool)
        rb, ab, free, cond = implicit_grad(o, ref, fx, x0[i], x, gbar[i], flags=flags if o.type == "dexpilot" else None,
                                           clip_init=clip)
        for k, v in (("x", x), ("grad_keypoints", keypoint_grad(o, rb)), ("grad_ref_value", rb), ("grad_last_qpos", ab),
                     ("free", free), ("cond", cond), ("flags", flags)):
            rec[k].append(v)
    return {k: np.array(v) for k, v in rec.items()}


def case(pool, key, kp, x0, fixed, xs, n, seed, clip=False):
    kp, x0 = kp[:n], x0[:n]
    fixed = fixed[:n] if fixed is not None else None
    gbar = np.random.RandomState(seed).randn(n, x0.shape[1]).astype(np.float32)
    chunks = np.array_split(np.arange(n), min(n, 32))
    parts = pool.map(_grad_chunk, [(key, kp[c], x0[c], fixed[c] if fixed is not None else None,
                                    xs[c] if xs is not None else None, gbar[c], clip) for c in chunks])
    out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    for k in ("x", "grad_keypoints", "grad_ref_value", "grad_last_qpos", "cond"):  # float32 keeps ~1e-7: ample for the tests
        out[k] = out[k].astype(np.float32)
    out.update(gbar=gbar, digest=np.array(W.digest(kp, x0, fixed)), n=np.array(n), key=np.array(key), clip_init=np.array(clip))
    return out


def main():
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    dst = ROOT / "tests" / "golden" / "grad_vectors.npz"
    par = np.load(ROOT / "tests" / "golden" / "bench_parity.npz")
    out = {}
    t0 = time.time()
    with mp.get_context("fork").Pool(8) as pool:
        def add(tag, rec):
            for k, v in rec.items():
                out[f"{tag}/{k}"] = v
            print(f"{tag}: {int(rec['n'])} frames, active frames {int((~rec['free']).any(1).sum())}, cond max {rec['cond'].max():.1e}, "
                  f"{time.time() - t0:.0f} s", flush=True)

        seq = W.build(W.METRIC_KEY)
        kp, x0, fixed, _ = W.frames(seq, 65536, W.METRIC_SEED)
        add("metric", case(pool, W.METRIC_KEY, kp, x0, fixed, par["metric/q"], n, GBAR_SEED))
        kp, x0, fixed, _ = W.frames(seq, 65536, W.METRIC_SEED, sigma=0.5)
        add("metric_clip", case(pool, W.METRIC_KEY, kp, x0, fixed, None, min(n, 64), GBAR_SEED + 1, clip=True))
        seq = W.build(W.SHADOW_POS_KEY)
        kp, x0, fixed, _ = W.frames(seq, 65536, W.SHADOW_SEED, narrow_dummy=True)
        add("shadow_narrow", case(pool, W.SHADOW_POS_KEY, kp, x0, fixed, par["shadow_narrow/q"], n, GBAR_SEED + 2))
        seq = W.build(W.LEAP_DEXPILOT_KEY)
        kp, x0, fixed, _ = W.frames(seq, 65536, W.SHADOW_SEED)
        add("leap_frames", case(pool, W.LEAP_DEXPILOT_KEY, kp, x0, fixed, par["leap_frames/q"], n, GBAR_SEED + 3))
        for i, key in enumerate(W.MIXED_KEYS):
            seq = W.build(key)
            kp, x0, fixed, _ = W.frames(seq, 16384, W.MIXED_SEED + i)
            tag = "mixed/" + key.split("/")[1]
            add(tag, case(pool, key, kp, x0, fixed, par[tag + "/q"], n, GBAR_SEED + 4 + i))
    np.savez_compressed(dst, **out)
    print("wrote", dst, dst.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
