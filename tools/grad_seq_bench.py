"""Forward vs backward time of SeqRetargeting.retarget_sequences (CUDA events, L2 flushed between timed launches).

Per workload: the no-grad forward (one fused launch), the autograd route's forward (the stream solver with the filter off, the
dexr_grad_lowpass filter, the trace gather and the state clones) and the backward pass (dexr_grad_sequences: flag replay and
reverse sweep).  Workloads: config 4 (LEAP DexPilot 2048 x 300), its one-GPU shard 256 x 300, Allegro vector 2048 x 300.
Records the card name and power limit of the same run and the library build ids.  Writes profiles/grad/grad_seq_bench.json
(or the path given).
Usage: python tools/grad_seq_bench.py [--reps R] [out.json]
"""
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import workloads as W  # noqa: E402
from grad_bench import power_limit, timed  # noqa: E402

from dex_retargeting_b200 import _native as N  # noqa: E402
from dex_retargeting_b200.grad import grad_sequences  # noqa: E402


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 10
    args = [a for i, a in enumerate(sys.argv[1:]) if not a.startswith("--") and sys.argv[i] != "--reps"]
    out = Path(args[0]) if args else ROOT / "profiles" / "grad" / "grad_seq_bench.json"
    d = torch.device("cuda", 0)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=d)
    rec = dict(card=torch.cuda.get_device_name(0), power_limit=power_limit(), reps=reps,
               grad_build_id=N.load_grad().dexr_grad_build_id().decode(), solver_build_id=N.build_id(), workloads={})
    cases = [("leap_dexpilot_config4", W.LEAP_DEXPILOT_KEY, 2048, 300), ("leap_dexpilot_shard", W.LEAP_DEXPILOT_KEY, 256, 300),
             ("allegro_vector", W.METRIC_KEY, 2048, 300)]
    for name, key, S, T in cases:
        seq = W.build(key, device=0)
        kp = torch.tensor(W.streams(S, T), device=d)
        st0 = seq.make_stream_state(S)
        st = seq.make_stream_state(S)
        status = torch.empty((S, T), dtype=torch.int32, device=d)
        robot = torch.empty((S, T, seq.optimizer.robot.dof), dtype=torch.float32, device=d)

        def reset():
            for k in st._FIELDS:
                if getattr(st0, k) is not None:
                    setattr(st, k, getattr(st0, k).clone())

        def fwd():
            reset()
            seq.retarget_sequences(kp, st, out=robot, status_out=status)

        kpg = kp.clone().requires_grad_(True)
        holder = {}

        def fwd_ag():
            reset()
            holder["out"] = seq.retarget_sequences(kpg, st, status_out=status)[0]

        fwd_ag()
        torch.cuda.synchronize()
        fn = holder["out"].grad_fn
        keypoints, fixed_qpos, last_in, proj_in, finit_in, trace, status_saved = fn.saved_tensors
        gy = torch.tensor(np.random.RandomState(0).randn(S, T, seq.optimizer.robot.dof).astype(np.float32), device=d)

        def bwd():
            holder["g"] = grad_sequences(seq, keypoints, trace, last_qpos=last_in, filter_init=finit_in, projected=proj_in,
                                         status=status_saved, grad_robot_qpos=gy)

        bwd()
        torch.cuda.synchronize()
        gs = holder["g"][3].cpu().numpy()
        st_f = status_saved.cpu().numpy()
        f_med, f_min = timed(fwd, flush, reps)
        a_med, a_min = timed(fwd_ag, flush, reps)
        b_med, b_min = timed(bwd, flush, reps)
        r = dict(key=key, streams=S, steps=T, forward_ms_median=f_med, forward_ms_min=f_min, autograd_forward_ms_median=a_med,
                 autograd_forward_ms_min=a_min, backward_ms_median=b_med, backward_ms_min=b_min,
                 backward_over_forward=b_med / f_med, forward_mean_iters=float((st_f & 0xffff).mean()),
                 forward_flagged_steps=int(((st_f >> 24) != 0).sum()),
                 grad_status_shifted=int(((gs & N.GRAD_STATUS_SHIFTED) != 0).sum()),
                 grad_status_zeroed=int(((gs & 0b11100) != 0).sum()), grad_finite=bool(torch.isfinite(holder["g"][0]).all().item()))
        rec["workloads"][name] = r
        print(name, json.dumps(r), flush=True)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
