"""C ABI of the stream backward pass (include/dexr_grad.h: dexr_grad_sequences, dexr_grad_lowpass): struct layout, exports and
argument validation without a GPU."""
import ctypes as C

from dex_retargeting_b200 import _native as N


def test_struct_mirror_and_exports():
    lib = N.load_grad()
    assert lib.dexr_grad_sequences_sizeof() == C.sizeof(N.DexrGradSequences) == 15 * 8
    assert lib.dexr_grad_frames_sizeof() == 96
    for name in ("dexr_grad_sequences_sizeof", "dexr_grad_sequences", "dexr_grad_lowpass"):
        assert name in N.GRAD_EXPORTS and getattr(lib, name) is not None
    assert lib.dexr_grad_version() == 1


def _setup(key):
    from helpers import build_product

    seq = build_product(key)
    opt = seq.optimizer
    return N.load_grad(), opt.build_table(), opt.params(clip_init=True, lp_alpha=seq.low_pass_alpha), opt


def test_invalid_arguments_are_rejected_without_gpu():
    lib, t, p, opt = _setup("teleop/allegro_hand_right")
    dev = C.c_void_p(0x1000)  # never dereferenced: validation happens before any CUDA call
    io = N.DexrGradSequences()

    def call(table=t, table_dev=dev, params=p, seqs=io, S=4, T=3):
        return lib.dexr_grad_sequences(C.byref(table) if table is not None else None, table_dev,
                                       C.byref(params) if params is not None else None,
                                       C.byref(seqs) if seqs is not None else None, S, T, 0, None)

    err = lambda: lib.dexr_grad_last_error()  # noqa: E731
    assert call(table=None) == -1 and b"null" in err()
    assert call(table_dev=None) == -1 and b"null" in err()
    assert call(params=None) == -1 and call(seqs=None) == -1
    assert call(table=N.DexrTable()) == -1 and b"magic" in err()
    assert call() == -1 and b"required" in err()
    io.keypoints = io.last_qpos = io.qpos = 0x2000
    assert call() == -1 and b"upstream gradient" in err()
    io.grad_robot_qpos = 0x3000
    assert p.lp_alpha >= 0
    assert call() == -1 and b"filter_init" in err()  # a filter without filter_init
    io.filter_init = 0x4000
    assert call(S=-1) == -1 and call(T=-1) == -1
    assert call(S=0) == 0 and call(T=0) == 0  # nothing to do
    raw = N.DexrParams.from_buffer_copy(p)
    raw.preprocess = 1
    assert call(params=raw) == -1 and b"preprocess" in err()
    # the gradient inputs pair with the upstream gradients: any one of the three is enough
    io.grad_robot_qpos, io.grad_filter_state_out = None, 0x5000
    assert call(S=0) == 0
    io.grad_filter_state_out, io.grad_last_qpos_out = None, 0x6000
    assert call(S=0) == 0


def test_dexpilot_needs_the_flag_workspace():
    lib, t, p, opt = _setup("teleop/leap_hand_right_dexpilot")
    assert t.len_proj > 0
    io = N.DexrGradSequences()
    io.keypoints = io.last_qpos = io.qpos = io.grad_robot_qpos = io.filter_init = 0x2000
    rc = lib.dexr_grad_sequences(C.byref(t), C.c_void_p(0x1000), C.byref(p), C.byref(io), 4, 3, 0, None)
    assert rc == -1 and b"projected_ws" in lib.dexr_grad_last_error()


def test_lowpass_arguments():
    lib = N.load_grad()
    x = 0x1000
    assert lib.dexr_grad_lowpass(None, x, x, x, 0.5, 4, 3, 16, 0, None) == -1 and b"null" in lib.dexr_grad_last_error()
    assert lib.dexr_grad_lowpass(x, x, x, x, 1.5, 4, 3, 16, 0, None) == -1 and b"alpha" in lib.dexr_grad_last_error()
    assert lib.dexr_grad_lowpass(x, x, x, x, 0.5, 4, 3, 33, 0, None) == -1 and b"dof" in lib.dexr_grad_last_error()
    assert lib.dexr_grad_lowpass(x, x, x, x, 0.5, -1, 3, 16, 0, None) == -1
    assert lib.dexr_grad_lowpass(x, x, x, x, 0.5, 0, 3, 16, 0, None) == 0
    assert lib.dexr_grad_lowpass(x, x, x, x, 0.5, 4, 0, 16, 0, None) == 0
