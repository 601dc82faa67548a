"""Forward vs backward kernel time of retarget_batch on 65 536 frames (CUDA events, L2 flushed between timed launches).

Workloads: Allegro vector (the metric workload), Shadow position config 3 (narrowed dummy range) and LEAP DexPilot.  Records
the card name and power limit of the same run.  Writes profiles/grad/grad_bench.json (or the path given).
Usage: python tools/grad_bench.py [--reps R] [out.json]
"""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import workloads as W  # noqa: E402

from dex_retargeting_b200 import _native as N  # noqa: E402
from dex_retargeting_b200.grad import grad_frames  # noqa: E402

B = 65536


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return out or None
    except Exception:
        return None


def timed(fn, flush, reps):
    ts = []
    for _ in range(reps):
        flush.zero_()  # evict L2 (the 256 MB buffer is larger than the B200's L2)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 20
    args = [a for i, a in enumerate(sys.argv[1:]) if not a.startswith("--") and sys.argv[i] != "--reps"]
    out = Path(args[0]) if args else ROOT / "profiles" / "grad" / "grad_bench.json"
    d = torch.device("cuda", 0)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=d)
    rec = dict(card=torch.cuda.get_device_name(0), power_limit=power_limit(), frames=B, reps=reps,
               grad_build_id=N.load_grad().dexr_grad_build_id().decode(), solver_build_id=N.build_id(), workloads={})
    cases = [("allegro_vector", W.METRIC_KEY, dict(seed=W.METRIC_SEED)),
             ("shadow_position_config3", W.SHADOW_POS_KEY, dict(seed=W.SHADOW_SEED, narrow_dummy=True)),
             ("leap_dexpilot", W.LEAP_DEXPILOT_KEY, dict(seed=W.SHADOW_SEED))]
    for name, key, kw in cases:
        seq = W.build(key, device=0)
        opt = seq.optimizer
        kp, x0, fixed, _ = W.frames(seq, B, kw["seed"], narrow_dummy=kw.get("narrow_dummy", False))
        kpt, x0t = torch.tensor(kp, device=d), torch.tensor(x0, device=d)
        fx = torch.tensor(fixed, device=d) if fixed is not None else None
        lp = len(opt.projected) if opt.retargeting_type == "DEXPILOT" else 0
        pj0 = torch.zeros((B, lp), dtype=torch.uint8, device=d) if lp else None
        pj = pj0.clone() if lp else None
        q = torch.empty((B, opt.opt_dof), dtype=torch.float32, device=d)
        st = torch.empty((B,), dtype=torch.int32, device=d)

        def fwd():
            if pj is not None:
                pj.copy_(pj0)
            opt.retarget_batch(keypoints=kpt, fixed_qpos=fx, last_qpos=x0t, projected=pj, out=q, status_out=st)

        fwd()
        torch.cuda.synchronize()
        gq = torch.tensor(np.random.RandomState(0).randn(B, opt.opt_dof).astype(np.float32), device=d)

        def bwd():
            grad_frames(opt, q, gq, last_qpos=x0t, keypoints=kpt, fixed_qpos=fx, projected=pj, status=st)

        bwd()
        torch.cuda.synchronize()
        gin, gl, gs = grad_frames(opt, q, gq, last_qpos=x0t, keypoints=kpt, fixed_qpos=fx, projected=pj, status=st)
        torch.cuda.synchronize()
        gs = gs.cpu().numpy()
        f_med, f_min = timed(fwd, flush, reps)
        b_med, b_min = timed(bwd, flush, reps)
        r = dict(key=key, forward_ms_median=f_med, forward_ms_min=f_min, backward_ms_median=b_med, backward_ms_min=b_min,
                 backward_over_forward=b_med / f_med, forward_mean_iters=float((st.cpu().numpy() & 0xffff).mean()),
                 grad_status_shifted=int(((gs & N.GRAD_STATUS_SHIFTED) != 0).sum()),
                 grad_status_zeroed=int(((gs & 0b11100) != 0).sum()), grad_finite=bool(torch.isfinite(gin).all().item()))
        rec["workloads"][name] = r
        print(name, json.dumps(r), flush=True)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
