"""C ABI of libdexr_grad.so (include/dexr_grad.h): exports, struct layout, argument validation without a GPU."""
import ctypes as C
import re
from pathlib import Path

from dex_retargeting_b200 import _native as N

ROOT = Path(__file__).resolve().parent.parent


def test_header_symbols_equal_grad_exports():
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "dexr_grad.h").read_text(), flags=re.S)
    names = sorted(set(re.findall(r"\b(dexr_grad_[a-z_]+)\s*\(", text)))
    assert set(names) == set(N.GRAD_EXPORTS)
    lib = N.load_grad()
    for n in names:
        assert getattr(lib, n) is not None
    assert not set(N.GRAD_EXPORTS) & set(N.EXPORTS)


def test_struct_layout_and_constants():
    lib = N.load_grad()
    assert lib.dexr_grad_version() == 1
    assert lib.dexr_grad_frames_sizeof() == C.sizeof(N.DexrGradFrames) == 96
    consts = dict(re.findall(r"#define\s+(DEXR_GRAD_STATUS_[A-Z]+)\s+\(1 << (\d+)\)", (ROOT / "include" / "dexr_grad.h").read_text()))
    assert {k: 1 << int(v) for k, v in consts.items()} == {
        "DEXR_GRAD_STATUS_ACTIVE": N.GRAD_STATUS_ACTIVE, "DEXR_GRAD_STATUS_SHIFTED": N.GRAD_STATUS_SHIFTED,
        "DEXR_GRAD_STATUS_SINGULAR": N.GRAD_STATUS_SINGULAR, "DEXR_GRAD_STATUS_SKIPPED": N.GRAD_STATUS_SKIPPED,
        "DEXR_GRAD_STATUS_NONFINITE": N.GRAD_STATUS_NONFINITE}
    from dex_retargeting_b200.build import grad_source_id

    assert lib.dexr_grad_build_id().decode() == grad_source_id()


def test_invalid_arguments_are_rejected_without_gpu():
    from helpers import build_product

    lib = N.load_grad()
    opt = build_product("teleop/allegro_hand_right").optimizer
    t, p = opt.build_table(), opt.params()
    dev = C.c_void_p(0x1000)  # never dereferenced: validation happens before any CUDA call
    io = N.DexrGradFrames()

    def call(table=t, table_dev=dev, params=p, frames=io, n=4):
        return lib.dexr_grad_frames(C.byref(table) if table is not None else None, table_dev,
                                    C.byref(params) if params is not None else None, C.byref(frames), n, 0, None)

    assert call(table=None) == -1 and b"null" in lib.dexr_grad_last_error()
    assert call(table_dev=None) == -1
    bad = N.DexrTable()
    assert call(table=bad) == -1 and b"magic" in lib.dexr_grad_last_error()
    assert call() == -1 and b"exactly one" in lib.dexr_grad_last_error()
    io.keypoints = io.ref_value = 0x2000
    assert call() == -1
    io.ref_value = None
    io.grad_ref_value = 0x3000
    assert call() == -1 and b"input gradient" in lib.dexr_grad_last_error()
    io.grad_ref_value = None
    assert call() == -1 and b"required" in lib.dexr_grad_last_error()
    io.last_qpos = io.qpos = io.grad_qpos = 0x4000
    assert call(n=-1) == -1
    assert call(n=0) == 0  # empty batch: nothing to do
    raw = opt.params(raw_hand="right")
    assert call(params=raw) == -1 and b"preprocess" in lib.dexr_grad_last_error()
