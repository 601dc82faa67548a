#!/usr/bin/env python
"""Throughput benchmark of the retargeting hot path (hand-frames/s), one process per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference-side CPU path, same metric / config
    python bench.py ... --dump-outputs DIR    # also save the last timed step's qpos as DIR/qpos.npy (seeded inputs)

Headline (BASELINE.json metric: "hand-frames/sec (21-kpt -> Allegro 16-DoF), batch 65536"): VectorOptimizer, Allegro
right hand, the shipped teleop config (scaling 1.6, huber 0.02, norm_delta 4e-3), one step = one batch of 65 536 synthetic
21-keypoint frames PER GPU -> 16 joint angles each (weak scaling: every rank its own frames, no data-path collective).
Workloads are generated on the host by tools/workloads.py (seeded numpy: q* ~ U(limits), FK, wrist / tips written at keypoints
{0,4,8,12,16} divided by the scale, warm start q* + 0.05 N(0,1) clipped) and built from the PACKAGED config + URDF.

One JSON line on stdout (rank 0):
  value      device-timed throughput of the headline, inputs resident in HBM, CUDA events, max over ranks
  e2e        the same batch through the host-buffer C-ABI call (pinned host memory in and out, copies inside the timed region);
             `e2e.staged_pageable` = the same call on pageable numpy buffers (chunked H2D -> solve -> D2H pipeline);
             `e2e.ref_value_form` = the same call fed ref_value [B,m,3], the form Optimizer.retarget receives (secondary: the
             headline form is the 21 keypoints north_star names)
  roofline   algorithmic HBM bytes / measured launch time vs the measured copy peak (the contract figure), plus what
             actually bounds the solver: `issue` (warp instructions per second vs 4 issue slots x SMs x clock) and `fp32`
             (executed FP32 operations per second vs 2 x 128 lanes x SMs x clock), both from the committed ncu capture of the
             SAME library build (profiles/roofline_traffic.json carries `build_id`; a mismatch voids them)
  sustained  the headline launch looped for >= 1 s (clocks under a long load)
  parity     |dq|_inf of THESE frames against the committed oracle fixture (tests/golden/bench_parity.npz, mode B)
  configs    one record per BASELINE.json configuration and arm, same timing discipline (L2 flushed between timed launches):
             2 (Allegro 4096), cold-start and real-trajectory arms of the metric config, 3 (Shadow position 65 536, STRONG
             scaling: the global batch is split over the ranks; shipped and narrowed dummy-joint ranges), 4 (DexPilot LEAP
             2048 streams x 300, streams split over the ranks), 5 (six robots x 16 384, every group split over the ranks)
  cpu_baseline   the oracle's reference-faithful CPU path (or the real reference when pinocchio + nlopt import) on this box's
             host cores, bounded sample, plus its one-core rate
"""
import argparse
import json
import math
import os
import statistics
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import workloads as W  # noqa: E402

FRAMES_PER_GPU = 65536
N_INPUT_SETS = 8  # rotating input batches: 8 x 20.7 MB of inputs > 126 MB L2
FP32_LANES_PER_SM = 128


def bytes_per_frame(opt, streams=False):
    """Algorithmic HBM bytes per hand-frame (SURVEY.md 8d): keypoints in + warm start in + qpos out; streams carry the warm
    start in registers and write the full filtered qpos."""
    if streams:
        return 252 + 4 * opt.robot.dof
    return 252 + 4 * opt.opt_dof + 4 * opt.opt_dof + 4 * len(opt.idx_pin2fixed)


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML): a background thread polls every
    2 ms, and the main thread adds one sample right after the launches are enqueued (GPU still busy), so even
    a timed region of a few milliseconds is covered."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.reasons, self._stop = [], set(), threading.Event()
        self.max_mhz, self._h, self._nv = None, None, None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")
        self._t = threading.Thread(target=self._run, daemon=True)

    def sample_now(self):
        if self._h is None:
            return
        nv = self._nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            for bit, nm in self.REASONS.items():
                if r & bit:
                    self.reasons.add(nm)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def _run(self):
        while not self._stop.is_set():
            self.sample_now()
            time.sleep(0.002)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=2)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------- CPU baseline
_WORKER = {}


def _cpu_worker_init(kind):
    sys.path.insert(0, str(ROOT / "tests"))
    _WORKER["kind"] = kind
    if kind == "reference":  # the real thing: the reference's own SeqRetargeting over nlopt + pinocchio
        from reference_probe import probe

        probe()  # puts the reference package on sys.path
        from dex_retargeting.retargeting_config import RetargetingConfig as RefConfig

        from dex_retargeting_b200.constants import config_root
        from dex_retargeting_b200.retargeting_config import RetargetingConfig

        RefConfig.set_default_urdf_dir(str(RetargetingConfig.packaged_urdf_dir()))
        _WORKER["ref"] = RefConfig.load_from_file(config_root() / (W.METRIC_KEY + ".yml")).build()
    else:
        from helpers import build_oracle

        _WORKER["o"] = build_oracle(W.METRIC_KEY)


def _cpu_worker(args):
    kp, x0 = args
    out = []
    if _WORKER["kind"] == "reference":
        ref = _WORKER["ref"]
        opt = ref.optimizer
        idx = np.asarray(opt.target_link_human_indices)
        for i in range(kp.shape[0]):
            rv = kp[i][idx[1]] - kp[i][idx[0]]
            out.append(opt.retarget(rv.astype(np.float32), np.zeros(0, np.float32), x0[i]))  # optimizer.py:77-102
        return np.array(out)
    from oracle.solvers import solve_reference

    o = _WORKER["o"]
    for i in range(kp.shape[0]):
        ref = o.ref_from_keypoints(kp[i]).astype(np.float32)
        lastc = np.clip(x0[i], o.joint_limits[:, 0], o.joint_limits[:, 1])
        q, _ = solve_reference(o, ref, np.zeros(0, np.float32), lastc)
        out.append(q)
    return np.array(out)


class CpuReferencePool:
    """The reference CPU path on `cores` single-threaded worker processes: the real reference (nlopt + pinocchio) when it
    imports, else the oracle's mode A (C FK / Jacobians like pinocchio's, loss in numpy, scipy SLSQP at the reference's ftol,
    value without / gradient with the regulariser)."""

    def __init__(self, cores, kp, x0, kind):
        import multiprocessing as mp

        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[var] = "1"  # inherited by the spawned workers: one thread each, no oversubscription
        self.cores = cores
        self.pool = mp.get_context("spawn").Pool(cores, initializer=_cpu_worker_init, initargs=(kind,))
        self.pool.map(_cpu_worker, [(kp[:1], x0[:1])] * cores)  # imports + first call outside any timing

    def frames_per_second(self, kp, x0, workers=None):
        w = workers or self.cores
        chunks = [(kp[i::w], x0[i::w]) for i in range(w)]
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker, chunks, chunksize=1)
        return kp.shape[0] / (time.perf_counter() - t0)

    def close(self):
        self.pool.close()
        self.pool.join()


def reference_kind():
    from reference_probe import probe

    found = probe()
    return ("reference" if found["reference"] else "port"), found


def host_cores():
    """Usable host cores: scheduler affinity, capped by the cgroup CPU quota when there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


KIND_NOTE = {"port": "restated reference path (C FK/Jacobian + numpy loss + scipy SLSQP at the reference's ftol); pinocchio/nlopt "
                     "do not import on this box",
             "reference": "the reference's own Optimizer.retarget (nlopt LD_SLSQP + pinocchio), one process per core"}


# --------------------------------------------------------------------------------------- main
def load_captures(build_id, path=None):
    """profiles/roofline_traffic.json -> {(bench record name, frames per launch): capture} for the captures taken from THIS library
    build, plus a note when the file belongs to another build (then nothing derived from it is reported)."""
    captures, cap_note = {}, None
    tpath = Path(path) if path else ROOT / "profiles" / "roofline_traffic.json"
    if tpath.exists():
        tj = json.loads(tpath.read_text())
        tj = tj if "captures" in tj else {"captures": {"metric": tj}}
        for name, c in tj["captures"].items():
            if c.get("build_id") == build_id:
                captures[(name.split("@")[0], c.get("frames_per_launch"))] = c
        if not captures:
            cap_note = f"profiles/roofline_traffic.json was captured from another library build (loaded build {build_id}): traffic / issue / fp32 withheld"
    return captures, cap_note


def roofline_record(c, cap_note, frames_per_launch, ms, bpf, iters, peak, peak_src, peak_issue, peak_fp32):
    """One `roofline` object: the contract figure (algorithmic HBM bytes / launch time vs the measured copy peak) and, from the
    ncu capture `c` of the same build, DRAM traffic and the two fractions that actually bind (issue slots, FP32)."""
    ach = bpf * frames_per_launch / (ms * 1e-3) / 1e9
    r = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
         "peak_source": peak_src, "bytes_per_frame": bpf, "launch_ms": ms}
    it_cap = c.get("iterations_mean_at_capture") if c else None
    if c and it_cap and iters and abs(iters / it_cap - 1.0) > 0.02:
        # the per-launch instruction / flop counts belong to another iteration count (solver parameters changed since the
        # capture, e.g. the initial damping): DRAM traffic is input-bound and stays valid, the two derived fractions do not
        r["traffic"] = c.get("dram_bytes_per_launch")
        r["note"] = (f"issue / fp32 withheld: captured at {it_cap:.3f} iterations per frame, this run solves at {iters:.3f} "
                     "(same library build, other solver parameters); profiles/r02/prof_*.md hold the capture")
    elif c:
        r["traffic"] = c.get("dram_bytes_per_launch")
        if c.get("warp_inst_per_launch"):
            a = c["warp_inst_per_launch"] / (ms * 1e-3)
            r["issue"] = {"achieved": a, "peak": peak_issue, "unit": "warp-inst/s", "frac": a / peak_issue,
                          "warp_inst_per_frame": c["warp_inst_per_launch"] / frames_per_launch}
        if c.get("fp32_flop_per_launch"):
            a = c["fp32_flop_per_launch"] / (ms * 1e-3)
            r["fp32"] = {"flops_per_frame": c["fp32_flop_per_launch"] / frames_per_launch, "achieved": a / 1e12, "peak": peak_fp32 / 1e12,
                         "unit": "TFLOP/s", "frac": a / peak_fp32,
                         "counted": "executed FFMA x 2 + FADD + FMUL thread instructions (ncu smsp__sass_thread_inst_executed_op_*), same capture"}
        r["capture"] = {"build_id": c.get("build_id"), "source": c.get("source")}
    elif cap_note:
        r["note"] = cap_note
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU per step (headline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only (skip the per-configuration records)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the qpos the last timed headline step computed to DIR/qpos.npy "
                    "(float32 [frames, 16]; qpos_rank<r>.npy per rank when several GPUs run), to compare two builds output for output")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    config = {"workload": "VectorOptimizer Allegro right 16-DoF, teleop config (scaling 1.6, huber 0.02, norm_delta 4e-3), "
                          "21-keypoint frames -> qpos, independent frames",
              "frames_per_gpu_per_step": args.frames, "global_frames_per_step": args.frames * world,
              "parallelism": f"frames sharded over {world} GPU(s), no data-path collective",
              "warm_start": "q* + 0.05 N(0,1) clipped", "l2": f"{N_INPUT_SETS} rotating input batches "
              f"({N_INPUT_SETS * args.frames * 316 / 1e6:.0f} MB > 126 MB L2); per-configuration records flush L2 "
              "(256 MB write) before every timed launch",
              "built_from": "dex_retargeting_b200/configs/teleop/allegro_hand_right.yml + packaged URDF"}

    if args.impl == "reference":
        if rank != 0:
            return
        seq = W.build(W.METRIC_KEY)
        cores = host_cores()
        kind, found = reference_kind()
        per_step = min(args.frames, max(cores * 64, 64))
        kp, x0, _, _ = W.frames(seq, args.frames, W.METRIC_SEED)  # the frames rank 0's first device batch holds
        pool = CpuReferencePool(cores, kp, x0, kind)
        rates = []
        for s in range(args.warmup + args.steps):
            lo = (s * per_step) % max(args.frames - per_step + 1, 1)
            r = pool.frames_per_second(kp[lo:lo + per_step], x0[lo:lo + per_step])
            if s >= args.warmup:
                rates.append(r)
        one_core = pool.frames_per_second(kp[:64], x0[:64], workers=1)
        pool.close()
        total = per_step * args.steps
        dt = sum(per_step / r for r in rates)
        value = total / dt
        sample = f"{per_step} frames/step x {args.steps} steps of the same synthetic workload (a rate: the 65 536-frame batch is sampled)"
        line = {"impl": "reference", "metric": "hand_frames_per_sec", "value": value, "unit": "frames/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "frames_per_step_actual": per_step,
                "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample,
                                 "one_core": one_core, "found": found, "note": KIND_NOTE[kind]},
                "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    import torch
    import torch.distributed as dist

    import parity as P
    from dex_retargeting_b200 import _native as NATIVE
    from dex_retargeting_b200.parallel import shard_range

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    seq = W.build(W.METRIC_KEY, device=local_rank)
    opt = seq.optimizer
    if world > 1:
        from dex_retargeting_b200.parallel import broadcast_table

        broadcast_table(opt, src=0)  # the only collective of the path: 8 KB robot table at init
    B = args.frames
    sets = [W.frames(seq, B, W.METRIC_SEED + rank + 1000 * s) for s in range(N_INPUT_SETS)]
    kp_sets = [torch.from_numpy(s[0]).to(dev) for s in sets]
    x0_sets = [torch.from_numpy(s[1]).to(dev) for s in sets]
    out = torch.empty((B, opt.opt_dof), dtype=torch.float32, device=dev)
    status = torch.zeros((B,), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def run(s):
        opt.retarget_batch(keypoints=kp_sets[s % N_INPUT_SETS], last_qpos=x0_sets[s % N_INPUT_SETS], out=out, status_out=status)

    # ---- device-resident arm (headline) -----------------------------------------------------------
    for s in range(args.warmup):
        run(s)
    barrier()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    with ClockSampler(local_rank) as clk:
        evs[0].record()
        for s in range(args.steps):
            run(s)
            evs[s + 1].record()
        clk.sample_now()  # launches are enqueued, the GPU is still working through them
        barrier()
    total_ms = evs[0].elapsed_time(evs[-1])
    launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    if args.dump_outputs:  # `out` is reused by every later arm: save the last timed step's answers now
        dump = Path(args.dump_outputs)
        dump.mkdir(parents=True, exist_ok=True)
        np.save(dump / ("qpos.npy" if world == 1 else f"qpos_rank{rank}.npy"), out.cpu().numpy())

    # ---- sustained: the same launch looped for >= 1 s ---------------------------------------------
    n_sus = max(args.steps, int(math.ceil(1.1e3 / max(statistics.mean(launch_ms), 1e-3))))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk_sus:
        e0.record()
        for s in range(n_sus):
            run(s)
        e1.record()
        clk_sus.sample_now()
        barrier()
    sus_ms = e0.elapsed_time(e1)

    # ---- parity of the headline frames (set 0 = the fixture's frames on rank 0) ---------------------
    run(0)
    torch.cuda.synchronize(dev)
    st = status.cpu().numpy()
    iters_mean = float((st & 0xffff).mean())
    flagged = int(((st >> 24) != 0).sum())
    parity = []
    if rank == 0 and B == FRAMES_PER_GPU:
        n = int(P.fixture()["metric/n"])
        parity.append(P.compare("metric", out[:n].cpu().numpy(), W.digest(sets[0][0][:n], sets[0][1][:n], None), st[:n]))

    # ---- end-to-end arm: pinned host buffers through the host C-ABI call -------------------------
    kp_pin = [torch.from_numpy(sets[i][0]).pin_memory() for i in range(2)]
    x0_pin = [torch.from_numpy(sets[i][1]).pin_memory() for i in range(2)]
    out_pin = torch.empty((B, opt.opt_dof), dtype=torch.float32).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))
    for s in range(2):
        opt.retarget_batch_host(keypoints=kp_pin[s % 2], last_qpos=x0_pin[s % 2], out=out_pin)
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        opt.retarget_batch_host(keypoints=kp_pin[s % 2], last_qpos=x0_pin[s % 2], out=out_pin)
    torch.cuda.synchronize(dev)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    checksum = float(out_pin.double().sum())
    # the same call on pageable buffers: staged H2D -> solve -> D2H pipeline through library-owned device buffers
    out_page = np.empty((B, opt.opt_dof), dtype=np.float32)
    opt.retarget_batch_host(keypoints=sets[0][0], last_qpos=sets[0][1], out=out_page)
    barrier()
    t0 = time.perf_counter()
    for s in range(3):
        opt.retarget_batch_host(keypoints=sets[s % 2][0], last_qpos=sets[s % 2][1], out=out_page)
    staged_ms = (time.perf_counter() - t0) * 1e3 / 3
    # the same frames in the form Optimizer.retarget() itself receives (optimizer.py:47): ref_value [B,m,3] = the caller-side
    # gather keypoints[task] - keypoints[origin] (example/vector_retargeting/single_hand_detector usage), 48 B instead of 252 B
    hi = np.asarray(opt.target_link_human_indices)
    rv_pin = [torch.from_numpy(np.ascontiguousarray(sets[i][0][:, hi[1]] - sets[i][0][:, hi[0]])).pin_memory() for i in range(2)]
    out_rv = torch.empty((B, opt.opt_dof), dtype=torch.float32).pin_memory()
    for s in range(2):
        opt.retarget_batch_host(ref_value=rv_pin[s % 2], last_qpos=x0_pin[s % 2], out=out_rv)
    rv_same = float((out_rv - out_pin).abs().max()) if e2e_steps % 2 == 0 else float("nan")
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        opt.retarget_batch_host(ref_value=rv_pin[s % 2], last_qpos=x0_pin[s % 2], out=out_rv)
    torch.cuda.synchronize(dev)
    rv_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    rv_bytes = int(rv_pin[0][0].numel()) * 4

    times = {"total_ms": total_ms, "e2e_ms": e2e_ms, "sus_ms": sus_ms, "staged_ms": staged_ms, "rv_ms": rv_ms}

    # ---- per-configuration records ---------------------------------------------------------------
    records = []  # (record dict, time key)

    def timed(fn, reps, warm=2):
        """Mean device time per launch (ms): L2 flushed before every timed launch, CUDA events around the launch only."""
        for i in range(warm):
            fn(i)
        barrier()
        ms = 0.0
        for i in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(i)
            b.record()
            b.synchronize()
            ms += a.elapsed_time(b)
        return ms / reps

    def frames_record(name, base_cfg, seqx, data_sets, global_n, scaling, tag=None, reps=8, note=None):
        """data_sets: list of (kp, x0, fixed) host arrays of the GLOBAL batch; this rank solves its contiguous shard."""
        o = seqx.optimizer
        b, e = shard_range(global_n, rank, world) if scaling == "strong" else (0, global_n)
        dsets = [(torch.from_numpy(k[b:e]).to(dev), torch.from_numpy(x[b:e]).to(dev),
                  torch.from_numpy(f[b:e]).to(dev) if f is not None else None) for k, x, f in data_sets]
        n = e - b
        q = torch.empty((n, o.opt_dof), dtype=torch.float32, device=dev)
        stt = torch.zeros((n,), dtype=torch.int32, device=dev)
        proj = torch.zeros((n, o._objective_spec().len_proj), dtype=torch.uint8, device=dev) if o.retargeting_type == "DEXPILOT" else None

        def fn(i):
            k, x, f = dsets[i % len(dsets)]
            if proj is not None:
                proj.zero_()
            o.retarget_batch(keypoints=k, last_qpos=x, fixed_qpos=f, out=q, status_out=stt, projected=proj)

        ms = timed(fn, reps)
        fn(0)
        torch.cuda.synchronize(dev)
        s_np = stt.cpu().numpy()
        rec = {"name": name, "baseline_config": base_cfg, "scaling": scaling, "global_frames": global_n * (1 if scaling == "strong" else world),
               "frames_per_gpu": n, "type": o.retargeting_type, "n_var": o.opt_dof, "dof": o.robot.dof,
               "iterations_mean": float((s_np & 0xffff).mean()), "flagged": int(((s_np >> 24) != 0).sum()),
               "bytes_per_frame": bytes_per_frame(o), "launch": o.engine().launch_info(), "reps": reps}
        if note:
            rec["note"] = note
        if tag and rank == 0:
            nfx = min(int(P.fixture()[f"{tag}/n"]), n)
            k, x, f = data_sets[0]
            rec["parity"] = P.compare(tag, q[:nfx].cpu().numpy(), W.digest(k[:nfx], x[:nfx], f[:nfx] if f is not None else None)
                                      if nfx == int(P.fixture()[f"{tag}/n"]) else None, s_np[:nfx])
        times[name] = ms
        records.append(rec)

    if not args.no_configs:
        # config 2: Vector Allegro, batch 4096 (its frames are the prefix of the metric batch)
        k0, x0_, _, _ = W.frames(seq, FRAMES_PER_GPU, W.METRIC_SEED)
        frames_record("allegro_vector_b4096", 2, seq, [(k0[:4096], x0_[:4096], None)], 4096, "strong", tag="metric", reps=20)
        # arms of the metric config: cold start (tests/test_optimizer.py:28-42) and the recorded trajectory
        kc, xc, _, _ = W.frames(seq, FRAMES_PER_GPU, W.METRIC_SEED, sigma=0.5)
        frames_record("allegro_vector_cold_start", "metric-arm", seq, [(kc, xc, None)], FRAMES_PER_GPU, "weak", tag="metric_cold",
                      note="warm start q* + 0.5 N(0,1) clipped")
        kr, xr = W.real_frames(seq, FRAMES_PER_GPU)
        frames_record("allegro_vector_real_trajectory", "metric-arm", seq, [(kr, xr, None)], FRAMES_PER_GPU, "weak", tag="metric_real",
                      note="621 recorded frames tiled with 2 mm offsets, every frame started from the mid-range pose")
        # config 3: Position Shadow (24 + 6 dummy = 30 DoF), 65 536 frames in total, strong scaling
        sh = W.build(W.SHADOW_POS_KEY, device=local_rank)
        for narrow, nm, tg in ((True, "shadow_position_narrowed", "shadow_narrow"), (False, "shadow_position_shipped", "shadow_ship")):
            ds = [W.frames(sh, FRAMES_PER_GPU, W.SHADOW_SEED + s, narrow_dummy=narrow)[:3] for s in range(2)]
            frames_record(nm, 3, sh, ds, FRAMES_PER_GPU, "strong", tag=tg, reps=5,
                          note="dummy joints drawn from " + ("+-0.5 m / +-pi" if narrow else "the shipped +-5 m / +-2 pi"))
        # config 4: DexPilot LEAP, 2048 streams x 300 frames in total, streams split over the ranks
        lp = W.build(W.LEAP_DEXPILOT_KEY, device=local_rank)
        kd, xd, _, _ = W.frames(lp, FRAMES_PER_GPU, W.SHADOW_SEED)
        frames_record("leap_dexpilot_frames", "config-4-arm", lp, [(kd, xd, None)], FRAMES_PER_GPU, "weak", tag="leap_frames", reps=5,
                      note="the config-4 objective on independent frames (hysteresis flags start cleared)")
        S, T = 2048, 300
        kps = W.streams(S, T)
        b, e = shard_range(S, rank, world)
        tk = torch.from_numpy(kps[b:e]).to(dev)
        rq = torch.empty((e - b, T, lp.optimizer.robot.dof), dtype=torch.float32, device=dev)
        sst = torch.zeros((e - b, T), dtype=torch.int32, device=dev)

        def fn_streams(i):
            lp.retarget_sequences(tk, out=rq, status_out=sst)

        ms = timed(fn_streams, 3, warm=1)
        fn_streams(0)
        torch.cuda.synchronize(dev)
        s_np = sst.cpu().numpy()
        rec = {"name": "leap_dexpilot_streams", "baseline_config": 4, "scaling": "strong", "global_streams": S, "steps": T,
               "streams_per_gpu": e - b, "global_frames": S * T, "type": "DEXPILOT", "n_var": 16, "dof": 16,
               "iterations_mean": float((s_np & 0xffff).mean()), "flagged": int(((s_np >> 24) != 0).sum()),
               "bytes_per_frame": bytes_per_frame(lp.optimizer, streams=True), "launch": lp.optimizer.engine().launch_info(), "reps": 3,
               "us_per_frame_per_stream": None}
        if rank == 0:
            nS = min(int(P.fixture()["leap_streams/n"]) // T, e - b)
            rec["parity"] = P.compare("leap_streams", rq[:nS].cpu().numpy(), W.digest(kps[:nS]) if nS * T == int(P.fixture()["leap_streams/n"]) else None,
                                      s_np[:nS])
        times["leap_dexpilot_streams"] = ms
        records.append(rec)
        # config 5: six robots x 16 384 frames, every robot group split over the ranks, one launch per robot on its own stream
        jobs = []
        per = 16384
        b, e = shard_range(per, rank, world)
        for i, key in enumerate(W.MIXED_KEYS):
            sq = W.build(key, device=local_rank)
            k, x, f, _ = W.frames(sq, per, W.MIXED_SEED + i)
            jobs.append((sq.optimizer, torch.from_numpy(k[b:e]).to(dev), torch.from_numpy(x[b:e]).to(dev),
                         torch.from_numpy(f[b:e]).to(dev) if f is not None else None,
                         torch.empty((e - b, sq.optimizer.opt_dof), dtype=torch.float32, device=dev), torch.cuda.Stream(dev),
                         key.split("/")[1], (k, x, f)))
        main_stream = torch.cuda.current_stream(dev)
        from dex_retargeting_b200.optimizer import retarget_batch_mixed

        mixed_jobs = [(o, dict(keypoints=k, last_qpos=x, fixed_qpos=f, out=q)) for o, k, x, f, q, s, _, _ in jobs]

        def fn_mixed(i):  # ONE persistent launch over the six robot groups (dexr_solve_frames_multi)
            retarget_batch_mixed(mixed_jobs)

        def fn_six_launches(i):  # round 1's way: one launch per robot, six CUDA streams
            for o, k, x, f, q, s, _, _ in jobs:
                s.wait_stream(main_stream)
                o.retarget_batch(keypoints=k, last_qpos=x, fixed_qpos=f, out=q, stream=s)
            for *_, s, _, _ in jobs:
                main_stream.wait_stream(s)

        ms_six = timed(fn_six_launches, 5)
        ms = timed(fn_mixed, 5)
        fn_mixed(0)
        torch.cuda.synchronize(dev)
        rec = {"name": "mixed_robots", "baseline_config": 5, "scaling": "strong", "global_frames": per * len(jobs), "frames_per_gpu": (e - b) * len(jobs),
               "robots": [j[6] for j in jobs], "bytes_per_frame": sum(bytes_per_frame(j[0]) for j in jobs) / len(jobs), "reps": 5,
               "launches_per_step": 1 if os.environ.get("DEXR_MULTI_MODE") == "persistent" else len(jobs),
               "note": "ONE call, dexr_solve_frames_multi: the six robot groups run as concurrent standalone kernels forked onto library side "
                       "streams and joined by events (default), or as one persistent kernel with DEXR_MULTI_MODE=persistent (measured slower, "
                       "profiles/r02/mixed_launch_sweep.txt)",
               "six_launches_ms_this_rank": ms_six}
        if rank == 0:
            pr = []
            for o, k, x, f, q, s, nm, host in jobs:
                nfx = min(int(P.fixture()[f"mixed/{nm}/n"]), e - b)
                hk, hx, hf = host
                pr.append(P.compare(f"mixed/{nm}", q[:nfx].cpu().numpy(),
                                    W.digest(hk[:nfx], hx[:nfx], hf[:nfx] if hf is not None else None) if nfx == int(P.fixture()[f"mixed/{nm}/n"]) else None))
            rec["parity"] = pr
        times["mixed_robots"] = ms
        records.append(rec)

    # ---- max over ranks of every time ----------------------------------------------------------------
    keys = sorted(times)
    t = torch.tensor([times[k] for k in keys], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    times = {k: float(v) for k, v in zip(keys, t.tolist())}
    total_ms, e2e_ms, sus_ms, staged_ms = times["total_ms"], times["e2e_ms"], times["sus_ms"], times["staged_ms"]
    rv_ms = times["rv_ms"]

    if rank == 0:
        peaks_path = ROOT / "MEASURED_PEAKS.json"
        if peaks_path.exists():
            peak, peak_src = json.loads(peaks_path.read_text())["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        props = torch.cuda.get_device_properties(dev)
        sm_mhz = (clk.summary() or {}).get("sm_max_mhz") or 1965
        peak_issue = 4 * props.multi_processor_count * sm_mhz * 1e6
        peak_fp32 = 2 * FP32_LANES_PER_SM * props.multi_processor_count * sm_mhz * 1e6
        build_id = NATIVE.build_id()
        captures, cap_note = load_captures(build_id)

        def roof(name, frames_per_launch, ms, bpf, iters=None):
            return roofline_record(captures.get((name, frames_per_launch)), cap_note, frames_per_launch, ms, bpf, iters,
                                   peak, peak_src, peak_issue, peak_fp32)

        mean_launch_ms = statistics.mean(launch_ms)
        value = B * world * args.steps / (total_ms * 1e-3)
        rl = roof("metric", B, mean_launch_ms, bytes_per_frame(opt), iters_mean)
        rl.update(launch_ms_mean=mean_launch_ms, launch_ms_min=min(launch_ms), launch_ms_max=max(launch_ms),
                  note="latency / FP32-issue bound solver: `issue` and `fp32` are the rooflines that bind (DESIGN.md 3.4)")
        for rec in records:
            ms = times[rec["name"]]
            units = rec.get("global_frames")
            per_gpu = rec.get("frames_per_gpu", rec.get("streams_per_gpu", 0) * rec.get("steps", 1))
            rec["ms_per_step"] = ms
            rec["value"] = units / (ms * 1e-3)
            rec["unit"] = "frames/s"
            rec["n_gpus"] = world
            if rec["name"] == "leap_dexpilot_streams":
                rec["us_per_frame_per_stream"] = ms * 1e3 / rec["steps"]
            rec["roofline"] = roof(rec["name"], per_gpu, ms, rec["bytes_per_frame"], rec.get("iterations_mean"))
        line = {
            "metric": "hand_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "roofline": rl,
            "sustained": {"value": B * world * n_sus / (sus_ms * 1e-3), "unit": "frames/s", "seconds": sus_ms * 1e-3, "steps": n_sus,
                          "clocks": clk_sus.summary()},
            "e2e": {"value": B * world / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": B * (252 + 64),
                    "d2h_bytes_per_step": B * 64, "ms_per_step": e2e_ms, "steps": e2e_steps, "checksum": checksum,
                    "api": "Optimizer.retarget_batch_host -> dexr_solve_frames_host, pinned host buffers in and out; zero-copy: the "
                           "kernel's TMA producer pulls the input tiles from host memory over PCIe and the results are "
                           "stored straight to host memory, all inside the timed region",
                    "staged_pageable": {"value": B * world / (staged_ms * 1e-3), "unit": "frames/s", "ms_per_step": staged_ms, "steps": 3,
                                        "api": "same call, pageable numpy buffers: 4-chunk H2D -> solve -> D2H pipeline on two internal streams"},
                    "ref_value_form": {"value": B * world / (rv_ms * 1e-3), "unit": "frames/s", "ms_per_step": rv_ms, "steps": e2e_steps,
                                       "h2d_bytes_per_step": B * (rv_bytes + 64), "d2h_bytes_per_step": B * 64,
                                       "max_abs_diff_vs_keypoint_form_rad": rv_same,
                                       "api": "same call with ref_value [B,m,3] (what Optimizer.retarget receives, the gather done by "
                                              "the caller outside the timed region) instead of the 21 keypoints; NOT the headline form"}},
            "gpu_launches": args.steps, "clocks": clk.summary(),
            "solver": {"mean_iterations": iters_mean, "frames_flagged": flagged, "launch": opt.engine().launch_info(), "build_id": build_id},
            "parity": parity, "configs": records,
        }
        if not args.no_cpu_baseline:
            cores = host_cores()
            kind, found = reference_kind()
            n_s = int(min(16384, max(64, cores * 64)))
            pool = CpuReferencePool(cores, sets[0][0], sets[0][1], kind)
            r = pool.frames_per_second(sets[0][0][:n_s], sets[0][1][:n_s])
            one = pool.frames_per_second(sets[0][0][:64], sets[0][1][:64], workers=1)
            pool.close()
            line["cpu_baseline"] = {"value": r, "unit": "frames/s", "cores": cores, "kind": kind, "one_core": one,
                                    "sample": f"first {n_s} frames of rank 0's first input batch, {cores} processes; one_core = first 64 frames, 1 process",
                                    "note": KIND_NOTE[kind]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
