"""Backward pass of retarget_batch (dexr_grad_kernels.cuh), checked without a GPU.

1. The float64 implicit gradient (tests/implicit_oracle.py) against central differences of converged float64 minimisers
   (oracle mode B) -- the reference of everything below is itself checked against the definition of a derivative.
2. The kernel SOURCE run through the host emulation (tests/emu_grad_host.py: the same warp shim as the forward solver's
   emulation) against that reference: on the committed fixture frames (tests/golden/grad_vectors.npz) and on synthetic robots
   with fixed joints.  The forward solution comes from the emulated forward solver; frames whose x* differs from the oracle's
   by more than 1e-4 or whose active sets differ are counted, not compared.  Error levels are printed (pytest -s).
"""
import sys

import numpy as np
import pytest

import emu_grad_host
import emu_host
from helpers import GOLDEN, build_oracle, build_product, synth_problems
from implicit_oracle import implicit_grad, keypoint_grad, post_flags, targets64

sys.path.insert(0, str(GOLDEN.parent.parent / "tools"))  # tools/workloads.py regenerates the fixture's frames
FIXTURE = GOLDEN / "grad_vectors.npz"
EMU_FRAMES = 24  # per workload (the emulation runs one warp at a time)
TAGS = ["metric", "metric_clip", "shadow_narrow", "leap_frames", "mixed/allegro_hand_right", "mixed/shadow_hand_right",
        "mixed/leap_hand_right", "mixed/ability_hand_right", "mixed/schunk_svh_hand_right", "mixed/inspire_hand_right"]
# relative error of a frame's whole gradient (input and last_qpos parts together), frames with cond(H_FF) < 1e5; measured
# levels: median <= 1.1e-6, p99 <= 6e-5 (shadow_narrow, the worst workload)
TOL_MEDIAN, TOL_P99 = 1e-5, 5e-4


def fixture_frames(tag, n):
    import workloads as W
    from dex_retargeting_b200 import _native  # noqa: F401

    fx = np.load(FIXTURE)
    key = str(fx[f"{tag}/key"])
    seq = W.build(key)
    if tag.startswith("mixed/"):
        kp, x0, fixed, _ = W.frames(seq, 16384, W.MIXED_SEED + W.MIXED_KEYS.index(key))
    elif tag == "metric":
        kp, x0, fixed, _ = W.frames(seq, 65536, W.METRIC_SEED)
    elif tag == "metric_clip":
        kp, x0, fixed, _ = W.frames(seq, 65536, W.METRIC_SEED, sigma=0.5)
    elif tag == "shadow_narrow":
        kp, x0, fixed, _ = W.frames(seq, 65536, W.SHADOW_SEED, narrow_dummy=True)
    else:
        kp, x0, fixed, _ = W.frames(seq, 65536, W.SHADOW_SEED)
    N = int(fx[f"{tag}/n"])
    n = min(n, N)
    assert str(fx[f"{tag}/digest"]) == W.digest(kp[:N], x0[:N], fixed[:N] if fixed is not None else None), "workload drifted"
    rec = {k.split("/")[-1]: fx[k][:n] for k in fx.files if k.startswith(tag + "/") and fx[k].ndim > 0}
    return seq, key, kp[:n], x0[:n], (fixed[:n] if fixed is not None else None), rec, bool(fx[f"{tag}/clip_init"])


def rel_errors(got_in, got_last, want_in, want_last):
    ref = np.concatenate([want_in.reshape(len(want_in), -1), want_last], 1).astype(np.float64)
    got = np.concatenate([got_in.reshape(len(got_in), -1), got_last], 1).astype(np.float64)
    return np.abs(got - ref).max(1) / np.maximum(np.abs(ref).max(1), 1e-30)


def compare(tag, q, gst, rec, g_in, g_last, mode):
    """`gst`: the kernel's grad status words; their ACTIVE bit against the oracle's active set stands in for the active sets."""
    same = (np.abs(q - rec["x"]).max(1) < 1e-4) & (((gst & 1) != 0) == (~rec["free"]).any(1))
    ok = same & (rec["cond"] < 1e5)
    want = rec["grad_keypoints"] if mode == "keypoints" else rec["grad_ref_value"]
    err = rel_errors(g_in, g_last, want, rec["grad_last_qpos"])
    for i in range(len(err)):  # every frame, also the ones not held to the tolerance
        print(f"  {tag} {mode} frame {i}: rel err {err[i]:.2e} cond {rec['cond'][i]:.1e} same basin {bool(same[i])}")
    e = err[ok]
    print(f"{tag} {mode}: {ok.sum()}/{len(ok)} frames compared ({(~same).sum()} other basin / active set), "
          f"rel err median {np.median(e):.2e} p99 {np.quantile(e, 0.99):.2e} max {e.max():.2e}")
    assert ok.sum() >= 0.9 * len(ok)
    assert np.median(e) < TOL_MEDIAN and np.quantile(e, 0.99) < TOL_P99


@pytest.mark.parametrize("mode", ["keypoints", "ref_value"])
@pytest.mark.parametrize("tag", TAGS)
def test_emulated_gradient_matches_fixture(tag, mode):
    """Both group widths (16: Allegro, LEAP, mimic hands; 32: Shadow), every loss, mimic folds, active bounds, clip_init."""
    seq, key, kp, x0, fixed, rec, clip = fixture_frames(tag, EMU_FRAMES)
    opt = seq.optimizer
    o = build_oracle(key)
    n = len(kp)
    proj = np.zeros((n, len(o.projected)), np.uint8) if o.type == "dexpilot" else None
    q, st, _ = emu_host.solve_frames(opt, x0, keypoints=kp, fixed_qpos=fixed, projected=proj, clip_init=clip)
    assert np.all((st >> 24) == 0)
    if proj is not None:
        np.testing.assert_array_equal(proj.astype(bool), rec["flags"])
    src = dict(keypoints=kp) if mode == "keypoints" else dict(ref_value=np.array([o.ref_from_keypoints(k) for k in kp], np.float32))
    g_in, g_last, gst = emu_grad_host.grad_frames(opt, x0, q, rec["gbar"], fixed_qpos=fixed, projected=proj, status=st,
                                                  clip_init=clip, **src)
    assert np.all((gst & 0b11100) == 0), gst
    compare(tag, q, gst, rec, g_in, g_last, mode)


def test_fixture_covers_the_cases():
    fx = np.load(FIXTURE)
    for tag in TAGS:
        assert int(fx[f"{tag}/n"]) >= 64
    assert (~fx["metric/free"]).any(1).sum() >= 10, "frames with active bounds"
    assert bool(fx["metric_clip/clip_init"])
    assert fx["leap_frames/flags"].any(), "DexPilot frames with projected rows"


def test_oracle_matches_finite_differences_of_minimisers():
    """The reference gradient is a derivative: directional central differences (h = 1e-5) of polished float64 minimisers,
    position (Shadow, dummy free joints), vector (Ability: mimic) and DexPilot (LEAP).  Frames whose active set or flags
    change inside the window are skipped; active joints get exactly 0."""
    from oracle.solvers import polish, solve_converged

    h = 1e-5
    checked = 0
    for key in ("offline/shadow_hand_right", "teleop/ability_hand_right", "teleop/leap_hand_right_dexpilot"):
        o = build_oracle(key)
        refs, fixed, x0, _ = synth_problems(o, 3, np.random.RandomState(11), init_noise=0.05, target_noise=0.01)
        rng = np.random.RandomState(12)
        for i in range(3):
            zero = np.zeros(len(o.projected), bool) if o.type == "dexpilot" else None
            flags = post_flags(o, refs[i], zero) if zero is not None else None

            def solve(ref, last):
                if zero is not None:
                    o.projected[:] = False
                return solve_converged(o, ref, fixed[i], last, x_init=x0[i], update_state=False)[0]

            x = solve(refs[i].astype(np.float64), x0[i])
            gbar = rng.randn(len(x))
            rb, ab, free, _ = implicit_grad(o, refs[i], fixed[i], x0[i], x, gbar, flags=flags)
            assert np.all(ab[~free] == 0.0) or np.allclose(ab[~free], 0.0, atol=1e-12)
            d = rng.randn(*refs[i].shape)
            def moved(ref):  # float64 targets (prepare rounds DexPilot targets to float32), flags frozen, polished from x
                obj = o.make_objective(refs[i], fixed[i], x0[i], update_state=False)
                obj.target, obj.weights = targets64(o, ref, flags)
                return polish(obj, x, o.lower, o.upper)[0]

            xp, xm = moved(refs[i] + h * d), moved(refs[i] - h * d)
            if zero is not None and not (np.array_equal(post_flags(o, refs[i] + h * d, zero), flags) and
                                         np.array_equal(post_flags(o, refs[i] - h * d, zero), flags)):
                continue
            if not (np.array_equal(xp <= o.lower, x <= o.lower) and np.array_equal(xp >= o.upper, x >= o.upper)):
                continue
            fd = gbar @ (xp - xm) / (2 * h)
            an = (rb * d).sum()
            print(f"{key} frame {i}: d(gbar.x)/d(ref) along d: fd {fd:.6e} implicit {an:.6e}")
            assert an == pytest.approx(fd, rel=1e-4, abs=1e-7)
            # anchor: re-polish x in float64 with the anchor moved (make_objective would round a moved anchor to float32)
            da = rng.randn(len(x))
            xs = []
            for sgn in (1, -1):
                if zero is not None:
                    o.projected[:] = False
                obj = o.make_objective(refs[i], fixed[i], x0[i], update_state=False)
                obj.last = obj.last + sgn * h * da
                xs.append(polish(obj, x, o.lower, o.upper)[0])
            fd_a = gbar @ (xs[0] - xs[1]) / (2 * h)
            print(f"{key} frame {i}: d(gbar.x)/d(last_qpos) along d: fd {fd_a:.6e} implicit {ab @ da:.6e}")
            assert ab @ da == pytest.approx(fd_a, rel=1e-4, abs=1e-7)
            checked += 1
    assert checked >= 6


def test_fixed_joints_synthetic_chain(tmp_path):
    """A 16-joint serial chain (prismatic joints mixed in) with four joints supplied per frame (fixed_qpos)."""
    from synthetic_robots import write_chain

    from dex_retargeting_b200.retargeting_config import RetargetingConfig
    from oracle.objectives import OracleOptimizer
    from oracle.solvers import solve_converged

    p, cfg = write_chain(tmp_path, 16, prismatic_every=5)
    cfg["target_joint_names"] = [f"j{i:02d}" for i in range(16) if i not in (2, 7, 11, 13)]
    seq = RetargetingConfig.from_dict(dict(cfg)).build()
    o = OracleOptimizer(dict(cfg), str(tmp_path))
    refs, fixed, x0, _ = synth_problems(o, 6, np.random.RandomState(4), init_noise=0.05, target_noise=0.002)
    q, st, _ = emu_host.solve_frames(seq.optimizer, x0, ref_value=refs, fixed_qpos=fixed)
    gbar = np.random.RandomState(5).randn(*x0.shape).astype(np.float32)
    g_in, g_last, gst = emu_grad_host.grad_frames(seq.optimizer, x0, q, gbar, ref_value=refs, fixed_qpos=fixed, status=st)
    errs = []
    for i in range(len(q)):
        x, _, _ = solve_converged(o, refs[i], fixed[i], x0[i], update_state=False)
        if np.abs(x - q[i]).max() > 1e-4:
            continue
        rb, ab, free, cond = implicit_grad(o, refs[i], fixed[i], x0[i], x, gbar[i])
        errs.append(rel_errors(g_in[i:i + 1], g_last[i:i + 1], rb[None], ab[None])[0])
        kg = keypoint_grad(o, rb)
        assert kg.shape == (21, 3)
    print("synthetic chain with fixed joints: rel err", ["%.1e" % e for e in errs])
    assert len(errs) >= 4 and max(errs) < TOL_P99


def test_flagged_frames_get_zero_gradient():
    """Forward status max-iterations / non-finite, and non-finite inputs: zero gradient and a status bit."""
    from dex_retargeting_b200 import _native as N

    seq, key, kp, x0, fixed, rec, _ = fixture_frames("metric", 4)
    opt = seq.optimizer
    q = rec["x"].astype(np.float32)
    st = np.array([0, N.STATUS_MAXITER | 7, N.STATUS_NONFINITE, 0], np.int32)
    kp = kp.copy()
    kp[3, 8, 1] = np.nan
    g_in, g_last, gst = emu_grad_host.grad_frames(opt, x0, q, rec["gbar"], keypoints=kp, fixed_qpos=fixed, status=st)
    assert gst[1] & N.GRAD_STATUS_SKIPPED and gst[2] & N.GRAD_STATUS_SKIPPED and gst[3] & N.GRAD_STATUS_NONFINITE
    assert not (gst[0] & 0b11100)
    for i in (1, 2, 3):
        assert np.all(g_in[i] == 0) and np.all(g_last[i] == 0)
    assert np.abs(g_in[0]).max() > 0
