"""Backward pass of SeqRetargeting.retarget_sequences on the B200 (libdexr_grad.so) -- needs a GPU.

The autograd route's forward bits against the no-grad call, the flag replay, the GPU gradients against the float64 fixture
(tests/golden/grad_seq_vectors.npz) and against the host emulation, against a Python composition of T dexr_grad_frames calls,
directional finite differences through full stream solves, chained calls, stream-position independence, the unchanged no-grad
path, refusals and a side stream.  Error levels are printed (pytest -s)."""
import copy
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from helpers import GOLDEN, build_oracle  # noqa: E402

sys.path.insert(0, str(GOLDEN.parent.parent / "tools"))
pytestmark = pytest.mark.gpu
FIXTURE = GOLDEN / "grad_seq_vectors.npz"
KEYS = {"leap": "teleop/leap_hand_right_dexpilot", "allegro": "teleop/allegro_hand_right", "ability": "teleop/ability_hand_right"}


def dev():
    return torch.device("cuda", 0)


def build(name, filt=True):
    import workloads as W

    seq = W.build(KEYS[name], device=0)
    if not filt:
        seq = copy.copy(seq)
        seq.filter = None
    return seq


def streams(S, T, seed=7):
    import workloads as W

    return torch.tensor(W.streams(S, T, seed=seed), device=dev())


def state_of(st):
    return {k: (None if getattr(st, k) is None else getattr(st, k).detach().clone()) for k in st._FIELDS}


def loss_of(seq, out, st, seed=3):
    """A seeded linear loss on all three outputs; returns (loss, (gy, gl, gf))."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    gy = torch.randn(out.shape, generator=g).to(dev())
    gl = torch.randn(st.last_qpos.shape, generator=g).to(dev())
    gf = torch.randn(st.filter_state.shape, generator=g).to(dev())
    return (out * gy).sum() + (st.last_qpos * gl).sum() + (st.filter_state * gf).sum(), (gy, gl, gf)


def grad_run(seq, kp, st=None, seed=3, **kw):
    """Autograd route: gradients of loss_of w.r.t. keypoints and the entry last_qpos / filter_state."""
    S = kp.shape[0]
    st = st or seq.make_stream_state(S)
    kp = kp.clone().requires_grad_(True)
    st.last_qpos.requires_grad_(True)
    st.filter_state.requires_grad_(True)
    last0, fs0 = st.last_qpos, st.filter_state
    out, st = seq.retarget_sequences(kp, st, **kw)
    loss, ups = loss_of(seq, out, st, seed)
    loss.backward()
    torch.cuda.synchronize()
    return out.detach(), st, kp.grad, last0.grad, fs0.grad, ups


@pytest.mark.parametrize("name,filt", [("leap", True), ("leap", False), ("allegro", True), ("allegro", False), ("ability", True)])
def test_autograd_forward_is_bitwise_the_no_grad_call(name, filt):
    seq = build(name, filt)
    kp = streams(64, 30)
    st_ref = seq.make_stream_state(64)
    ref, _ = seq.retarget_sequences(kp, st_ref)
    st = seq.make_stream_state(64)
    st.last_qpos.requires_grad_(True)
    out, st = seq.retarget_sequences(kp.clone().requires_grad_(True), st)
    assert out.grad_fn is not None and st.last_qpos.grad_fn is not None
    assert torch.equal(out.detach(), ref)
    for k in st._FIELDS:
        a, b = getattr(st, k), getattr(st_ref, k)
        assert (a is None) == (b is None)
        if a is not None:
            assert torch.equal(a.detach(), b), k
    # the exit last_qpos is the trace's last row: the unfiltered solution of the last step
    raw = copy.copy(seq)
    raw.filter = None
    q, _ = raw.retarget_sequences(kp, seq.make_stream_state(64))
    idx = torch.as_tensor(seq.optimizer.idx_pin2target, device=dev())
    assert torch.equal(st.last_qpos.detach(), q[:, -1].index_select(1, idx))


def test_flag_replay_ends_at_the_forward_flags():
    from dex_retargeting_b200.grad import grad_sequences

    seq = build("leap")
    # the recorded trajectory's DexPilot flags switch on from frame 252 and off again by frame 281: the forward pass is split
    # at frame 260, where flags are set, so that the replay is checked there as well as at the end
    kp = streams(128, 300)
    mid = 260
    st = seq.make_stream_state(128)
    entry = state_of(st)
    raw = copy.copy(seq)
    raw.filter = None
    q1, st = raw.retarget_sequences(kp[:, :mid].contiguous(), st)
    flags_mid = st.projected.clone()
    q2, st = raw.retarget_sequences(kp[:, mid:].contiguous(), st)
    q = torch.cat([q1, q2], 1)
    idx = torch.as_tensor(seq.optimizer.idx_pin2target, device=dev())
    trace = q.index_select(2, idx).contiguous()
    gy = torch.ones_like(q)
    *_, ws = grad_sequences(seq, kp, trace, last_qpos=entry["last_qpos"], filter_init=entry["filter_init"],
                            projected=entry["projected"], grad_robot_qpos=gy)
    torch.cuda.synchronize()
    assert ws.shape == (128, 300, st.projected.shape[1])
    assert bool(flags_mid.any()), "flags are set at the split"
    assert torch.equal(ws[:, mid - 1], flags_mid)
    assert torch.equal(ws[:, -1], st.projected)
    assert bool((ws[:, 1:] != ws[:, :-1]).any()), "flags switch inside the streams"


def fixture(tag):
    fx = np.load(FIXTURE)
    return {k.split("/", 1)[1]: fx[k] for k in fx.files if k.startswith(tag + "/")}


def fixture_grads(tag, runner):
    import workloads as W

    rec = fixture(tag)
    seq = W.build(str(rec["key"]), device=0)
    t = lambda a: torch.tensor(a, device=dev())  # noqa: E731
    proj = torch.zeros((rec["x"].shape[0], seq.optimizer.engine().table.len_proj), dtype=torch.uint8, device=dev())
    g = runner(seq, t(rec["keypoints"]), t(rec["x"]), last_qpos=t(rec["last_qpos"]), filter_init=t(rec["filter_init"]),
               projected=proj if proj.shape[1] else None, grad_robot_qpos=t(rec["grad_robot_qpos"]),
               grad_last_qpos=t(rec["grad_last_qpos_out"]), grad_filter_state=t(rec["grad_filter_state_out"]),
               lp_alpha=float(rec["alpha"]))
    torch.cuda.synchronize()
    return seq, rec, [v.cpu().numpy() if v is not None else None for v in g]


TAGS = ["leap_dexpilot", "allegro", "allegro_nofilter", "allegro_finit", "ability", "shadow"]


@pytest.mark.parametrize("tag", TAGS)
def test_gpu_gradient_matches_fixture(tag):
    from dex_retargeting_b200.grad import grad_sequences
    from test_grad_seq_emulation import compare

    seq, rec, (g_kp, g_last, g_fs, g_st, ws) = fixture_grads(tag, grad_sequences)
    assert np.all((g_st & 0b11100) == 0)
    if ws is not None:
        np.testing.assert_array_equal(ws, rec["flags"])
    compare(tag, rec, g_kp, g_last, g_fs)


@pytest.mark.parametrize("tag", ["leap_dexpilot", "allegro", "ability", "shadow"])
def test_gpu_matches_emulation(tag):
    import emu_grad_seq_host
    from dex_retargeting_b200.grad import grad_sequences
    from test_grad_seq_emulation import rel_errors

    seq, rec, (g_kp, g_last, g_fs, g_st, _) = fixture_grads(tag, grad_sequences)
    e_kp, e_last, e_fs, e_st, _ = emu_grad_seq_host.grad_sequences(
        seq, rec["keypoints"], rec["x"], rec["last_qpos"], filter_init=rec["filter_init"],
        projected=np.zeros((len(rec["x"]), rec["flags"].shape[2]), np.uint8), grad_robot_qpos=rec["grad_robot_qpos"],
        grad_last_qpos=rec["grad_last_qpos_out"], grad_filter_state=rec["grad_filter_state_out"], lp_alpha=float(rec["alpha"]))
    np.testing.assert_array_equal(e_st, g_st)
    err = rel_errors(g_kp, g_last, g_fs, e_kp, e_last, e_fs)
    print(f"{tag}: GPU vs emulation rel err median {np.median(err):.2e} max {err.max():.2e}")
    # (measured on a B200: median <= 4.7e-6 everywhere; max 7.8e-4 on LEAP DexPilot, <= 1e-5 on the vector hands)
    assert err.max() < (2e-3 if tag == "leap_dexpilot" else 1e-4) and np.median(err) < 1e-5


def compose_frames(seq, kp, trace, entry, status, ws, gy, gl, gf):
    """The stream backward written out in torch: T dexr_grad_frames calls chained by the float32 filter and fold adjoints."""
    from dex_retargeting_b200.grad import grad_frames

    opt = seq.optimizer
    t_ = opt.engine().table
    S, T = kp.shape[:2]
    dof, n = opt.robot.dof, opt.opt_dof
    alpha = seq.low_pass_alpha
    M = torch.zeros((n, dof), device=dev())  # x-bar = M q-bar, the table's variable groups
    for c in range(dof):
        v = t_.var_index[c]
        if v >= 0:
            for f in range(t_.group_count[c]):
                M[v, t_.group_lane[c][f]] = t_.group_mult[c][f]
    ybar = gf.clone()
    carry = gl.clone()
    g_kp = torch.empty_like(kp)
    for t in reversed(range(T)):
        if 0 <= alpha <= 1:
            ybar = ybar + gy[:, t]
            if t > 0 or bool(entry["filter_init"].all()):
                qbar, ybar = alpha * ybar, (1.0 - alpha) * ybar
            else:
                qbar, ybar = ybar, torch.zeros_like(ybar)
        else:
            qbar = gy[:, t]
        xbar = (qbar @ M.T if t_.has_mimic else qbar.index_select(1, torch.as_tensor(opt.idx_pin2target, device=dev()))) + carry
        last = trace[:, t - 1] if t > 0 else entry["last_qpos"]
        gi, carry, _ = grad_frames(opt, trace[:, t].contiguous(), xbar.contiguous(), last_qpos=last.contiguous(),
                                   keypoints=kp[:, t].contiguous(), projected=ws[:, t].contiguous() if ws is not None else None,
                                   status=status[:, t].contiguous(), clip_init=True)
        g_kp[:, t] = gi
    return g_kp, carry, ybar


@pytest.mark.parametrize("name,filt", [("allegro", False), ("allegro", True), ("leap", True), ("ability", True)])
def test_matches_composition_of_frame_calls(name, filt):
    from dex_retargeting_b200.grad import grad_sequences

    seq = build(name, filt)
    S, T = 48, 16
    kp = streams(S, T)
    st = seq.make_stream_state(S)
    entry = state_of(st)
    status = torch.empty((S, T), dtype=torch.int32, device=dev())
    raw = copy.copy(seq)
    raw.filter = None
    q, _ = raw.retarget_sequences(kp, st, status_out=status)
    trace = q.index_select(2, torch.as_tensor(seq.optimizer.idx_pin2target, device=dev())).contiguous()
    g = torch.Generator(device="cpu").manual_seed(5)
    gy = torch.randn(q.shape, generator=g).to(dev())
    gl = torch.randn(trace[:, 0].shape, generator=g).to(dev())
    gf = torch.randn(q[:, 0].shape, generator=g).to(dev())
    g_kp, g_last, g_fs, g_st, ws = grad_sequences(seq, kp, trace, last_qpos=entry["last_qpos"], filter_init=entry["filter_init"],
                                                  projected=entry["projected"], status=status, grad_robot_qpos=gy,
                                                  grad_last_qpos=gl, grad_filter_state=gf)
    c_kp, c_last, c_fs = compose_frames(seq, kp, trace, entry, status, ws, gy, gl, gf)
    torch.cuda.synchronize()
    if name == "allegro" and not filt:
        assert torch.equal(g_kp, c_kp) and torch.equal(g_last, c_last) and torch.equal(g_fs, c_fs)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))  # noqa: E731
    errs = rel(g_kp, c_kp), rel(g_last, c_last), rel(g_fs, c_fs) if 0 <= seq.low_pass_alpha <= 1 else 0.0
    print(f"{name} filter={filt}: stream kernel vs composed frames rel diff kp {errs[0]:.1e} last {errs[1]:.1e} fs {errs[2]:.1e}")
    assert max(errs) <= 1e-6


@pytest.mark.parametrize("name", ["allegro", "ability"])
def test_directional_finite_difference_through_stream_solves(name):
    """d loss / d kp along d from two full GPU stream solves at kp +- h d (h = 1e-3); streams whose active sets (at any step)
    or DexPilot flags change between the two are skipped."""
    from dex_retargeting_b200.grad import grad_sequences

    seq = build(name)
    o = build_oracle(KEYS[name])
    S, T = 128, 12
    kp = streams(S, T, seed=21)
    out, st, g_kp, _, _, (gy, gl, gf) = grad_run(seq, kp)
    d_ = torch.randn(kp.shape, generator=torch.Generator(device="cpu").manual_seed(9)).to(dev())
    d_[:, :, 0] = 0
    h = 1e-3
    raw = copy.copy(seq)
    raw.filter = None
    idx = torch.as_tensor(seq.optimizer.idx_pin2target, device=dev())
    lo, hi = torch.tensor(o.lower, dtype=torch.float32, device=dev()), torch.tensor(o.upper, dtype=torch.float32, device=dev())

    def solve(k):
        s1 = seq.make_stream_state(S)
        y, s1 = seq.retarget_sequences(k, s1)
        q, s2 = raw.retarget_sequences(k, seq.make_stream_state(S))
        x = q.index_select(2, idx)
        l_ = (y.double() * gy).sum((1, 2)) + (s1.last_qpos.double() * gl).sum(1) + (s1.filter_state.double() * gf).sum(1)
        ws = None
        if s2.projected is not None:
            *_, ws = grad_sequences(seq, k, x.contiguous(), last_qpos=seq.make_stream_state(S).last_qpos,
                                    filter_init=s1.filter_init * 0, projected=seq.make_stream_state(S).projected,
                                    grad_robot_qpos=torch.zeros_like(y))
        return l_, (x <= lo).flatten(1), (x >= hi).flatten(1), ws

    base, pl = solve(kp), solve(kp + h * d_)
    mi = solve(kp - h * d_)
    keep = torch.ones(S, dtype=torch.bool, device=dev())
    for i in (1, 2):
        keep &= (pl[i] == base[i]).all(1) & (mi[i] == base[i]).all(1)
    if base[3] is not None:
        keep &= (pl[3] == base[3]).flatten(1).all(1) & (mi[3] == base[3]).flatten(1).all(1)
    fd = (pl[0] - mi[0]) / (2 * h)
    an = (g_kp.double() * d_).sum((1, 2, 3))
    err = ((fd - an).abs() / an.abs().clamp_min(1e-3))[keep].cpu().numpy()
    print(f"{name}: {int(keep.sum())}/{S} streams kept, directional FD rel err median {np.median(err):.2e} "
          f"p90 {np.quantile(err, 0.9):.2e}")
    assert keep.sum() >= 0.25 * S
    assert np.median(err) < 1e-2


@pytest.mark.parametrize("name", ["allegro", "leap", "ability"])
def test_two_chained_calls_equal_one_call(name):
    seq = build(name)
    S, T = 32, 20
    kp = streams(S, T)
    out, st, g_kp, g_last, g_fs, (gy, gl, gf) = grad_run(seq, kp)
    k1 = kp[:, : T // 2].contiguous().requires_grad_(True)
    k2 = kp[:, T // 2:].contiguous().requires_grad_(True)
    st2 = seq.make_stream_state(S)
    st2.last_qpos.requires_grad_(True)
    st2.filter_state.requires_grad_(True)
    last0, fs0 = st2.last_qpos, st2.filter_state
    o1, st2 = seq.retarget_sequences(k1, st2)
    o2, st2 = seq.retarget_sequences(k2, st2)
    both = torch.cat([o1, o2], 1)
    assert torch.equal(both.detach(), out)
    loss = (both * gy).sum() + (st2.last_qpos * gl).sum() + (st2.filter_state * gf).sum()
    loss.backward()
    torch.cuda.synchronize()
    assert torch.equal(torch.cat([k1.grad, k2.grad], 1), g_kp)
    assert torch.equal(last0.grad, g_last) and torch.equal(fs0.grad, g_fs)
    # .detach() on the state truncates the graph at the call boundary
    st3 = seq.make_stream_state(S)
    k3 = kp[:, : T // 2].contiguous().requires_grad_(True)
    _, st3 = seq.retarget_sequences(k3, st3)
    st3.last_qpos, st3.filter_state = st3.last_qpos.detach(), st3.filter_state.detach()
    o4, st3 = seq.retarget_sequences(kp[:, T // 2:].contiguous(), st3)
    assert o4.grad_fn is None


def test_stream_gradient_independent_of_batch_size_and_position():
    from dex_retargeting_b200.grad import grad_sequences

    seq = build("leap")
    S, T = 2048, 10
    kp = streams(S, T)
    st = seq.make_stream_state(S)
    entry = state_of(st)
    status = torch.empty((S, T), dtype=torch.int32, device=dev())
    raw = copy.copy(seq)
    raw.filter = None
    q, _ = raw.retarget_sequences(kp, st, status_out=status)
    trace = q.index_select(2, torch.as_tensor(seq.optimizer.idx_pin2target, device=dev())).contiguous()
    gy = torch.randn(q.shape, generator=torch.Generator(device="cpu").manual_seed(1)).to(dev())

    def run(sel):
        return grad_sequences(seq, kp[sel].contiguous(), trace[sel].contiguous(), last_qpos=entry["last_qpos"][sel].contiguous(),
                              filter_init=entry["filter_init"][sel].contiguous(), projected=entry["projected"][sel].contiguous(),
                              status=status[sel].contiguous(), grad_robot_qpos=gy[sel].contiguous())[:4]

    full = run(torch.arange(S, device=dev()))
    perm = torch.randperm(S, generator=torch.Generator(device="cpu").manual_seed(2))[:37].to(dev())
    part = run(perm)
    for a, b in zip(full, part):
        assert torch.equal(a[perm], b)
    for i in (0, 1000, S - 1):
        one = run(torch.tensor([i], device=dev()))
        for a, b in zip(full, one):
            assert torch.equal(a[i:i + 1], b)


def test_no_grad_path_is_one_launch_in_place():
    import ctypes as C

    from dex_retargeting_b200 import _native as N

    seq = build("leap")
    eng = seq.optimizer.engine()
    kp = streams(16, 8).requires_grad_(True)
    st = seq.make_stream_state(16)
    ptrs = {k: getattr(st, k).data_ptr() for k in ("last_qpos", "filter_state")}
    before = st.last_qpos.clone()
    info = N.DexrLaunchInfo()
    N.check(eng.lib.dexr_get_launch_info(eng.handle, C.byref(info)), "info")
    n0 = info.kernels_launched
    with torch.no_grad():
        out, st2 = seq.retarget_sequences(kp, st)
    N.check(eng.lib.dexr_get_launch_info(eng.handle, C.byref(info)), "info")
    assert info.kernels_launched == n0 + 1
    assert st2 is st and out.grad_fn is None
    assert {k: getattr(st, k).data_ptr() for k in ptrs} == ptrs and not torch.equal(before, st.last_qpos)


def test_refusals_side_stream_and_grad_status():
    seq = build("allegro")
    kp = streams(8, 6)
    st = seq.make_stream_state(8)
    k = kp.clone().requires_grad_(True)
    with pytest.raises(ValueError, match="out="):
        seq.retarget_sequences(k, st, out=torch.empty((8, 6, seq.optimizer.robot.dof), device=dev()))
    with pytest.raises(ValueError, match="raw_hand"):
        seq.retarget_sequences(k, st, raw_hand="right")
    with pytest.raises(ValueError, match="fixed_qpos"):
        seq.retarget_sequences(k, st, fixed_qpos=torch.zeros((8, 6, 0), device=dev(), requires_grad=True))
    ref = grad_run(seq, kp)
    side = torch.cuda.Stream(device=dev())
    with torch.cuda.stream(side):
        got = grad_run(seq, kp, stream=side)
    torch.cuda.synchronize()
    for a, b in zip(ref[2:5], got[2:5]):
        assert torch.equal(a, b)
    gs = seq.last_grad_status
    assert gs.shape == (8, 6) and gs.dtype == torch.int32
    assert not bool((gs & 0b11100).any())
