"""Motion (Laplace) with chroma attenuation 0: the synthesis runs on the L planes only.

With chroma 0 the a and b planes of the motion image are multiplied by 0 before input + motion (MagnifyCore.hpp:140-148),
so the output's a and b are the input's, bit for bit (DESIGN.md §4).  The collapse and egress kernels then skip the a and b
planes; the state kernels keep updating them.  These tests hold that path to the general one (chroma 1e-30, a normal float
that takes the three-channel kernels), to a run whose chroma changes between frames, and, on the CUDA-on-CPU emulation
(MC_EMU=1), to the oracle with every device allocation filled with NaN, so that a kernel reading an a or b plane that this
frame did not write would show up in the output."""
import os

import numpy as np
import pytest

import lvm_b200 as L
from lvm_b200.synth import synth_frame
from oracle import livim_oracle as O
from common import make_cfgs, u8_diff

pytestmark = pytest.mark.gpu

F32_TOL = 1e-4


def params(levels, chroma):
    """Laplace parameters of the UI defaults (alpha 20, wavelength 50, 0.4-3 Hz) with chromAttenuation set directly."""
    cfg, _ = make_cfgs(O.MODE_LAPLACE, 20, 50.0, 0.4, 3.0, 0, levels)
    cfg.magnification.chromAttenuation = chroma
    return cfg


def clip(t, w, h, lanes):
    return np.stack([np.roll(synth_frame(t, w, h, 3), (3 * k, 7 * k), axis=(0, 1)) for k in range(lanes)])


def processor(lanes, strip, groups, band_from_state=1):
    p = L.MagnificationProcessor(0, lanes=lanes)
    p.set_option("egress_strip", strip)
    p.set_option("lane_groups", groups)
    p.set_option("band_from_state", band_from_state)
    p.set_option("keep_float_output", 1)
    return p


@pytest.mark.parametrize("groups", [1, 2])
@pytest.mark.parametrize("strip", [20, 0])
@pytest.mark.parametrize("w,h,levels", [(1920, 1080, 6), (321, 243, 2), (321, 243, 3), (321, 243, 6)])
def test_chroma_zero_equals_general_path(w, h, levels, strip, groups):
    """chroma 0 (L-only synthesis) and chroma 1e-30 (all three channels, the a and b motion scaled to ~1e-32 and lost in
    the add) give identical u8 frames and float taps, over both egress forms, one and two lane groups and both band
    sources."""
    lanes, frames = 2, 4 if w < 1000 else 3
    for band_from_state in ((1, 0) if w < 1000 else (1,)):
        a, b = processor(lanes, strip, groups, band_from_state), processor(lanes, strip, groups, band_from_state)
        ca, cb = params(levels, 0.0), params(levels, 1e-30)
        for t in range(frames):
            f = clip(t, w, h, lanes)
            _, oa = a.process_image(f, ca)
            _, ob = b.process_image(f, cb)
            assert np.array_equal(oa, ob), (t, band_from_state, int(u8_diff(oa, ob).max()))
            fa, fb = a.float_output(w, h, 3), b.float_output(w, h, 3)
            assert np.array_equal(fa, fb), (t, band_from_state, float(np.nanmax(np.abs(fa - fb))))
        a.close()
        b.close()


@pytest.mark.parametrize("band_from_state", [1, 0])
@pytest.mark.parametrize("strip", [20, 0])
def test_live_chroma_change(strip, band_from_state):
    """chroma 30 % -> 0 -> 30 % over 12 frames equals a constant 30 % in the last phase (frames, float taps) and in the
    temporal state throughout: skipping the a and b planes at chroma 0 leaves nothing stale behind."""
    w, h, levels, lanes = 200, 136, 5, 2
    a, b = processor(lanes, strip, 0, band_from_state), processor(lanes, strip, 0, band_from_state)
    c30, c0 = params(levels, 0.3), params(levels, 0.0)
    for t in range(12):
        f = clip(t, w, h, lanes)
        _, oa = a.process_image(f, c0 if 4 <= t < 8 else c30)
        _, ob = b.process_image(f, c30)
        if t >= 8:
            assert np.array_equal(oa, ob), (t, int(u8_diff(oa, ob).max()))
            assert np.array_equal(a.float_output(w, h, 3), b.float_output(w, h, 3)), t
        for lvl in range(1, levels):
            for name in ("lowpassHi", "lowpassLo"):
                assert np.array_equal(a.get_state(name, lvl), b.get_state(name, lvl)), (t, lvl, name)


@pytest.fixture(scope="module")
def nan_fill_library(tmp_path_factory):
    """On the emulation (MC_EMU=1): a private build of the emulated library whose allocator fills new memory with 0xff
    bytes — every f32 a NaN — instead of its usual 0xcd pattern (a finite float, which a multiply by 0 would hide).
    None on a GPU, where what cudaMalloc returns is not under the test's control."""
    if os.environ.get("MC_EMU") != "1":
        return None
    import build_emu   # tests/cuda_emu, put on sys.path by conftest.py under MC_EMU=1
    tmp = tmp_path_factory.mktemp("emu_nan_fill")
    src = open(os.path.join(build_emu.HERE, "emu_runtime.cpp")).read()
    fill = "std::memset(q, 0xcd, n);"
    assert src.count(fill) == 1, "emu_runtime.cpp: allocation fill not found"
    (tmp / "emu_runtime.cpp").write_text(src.replace(fill, "std::memset(q, 0xff, n);"))
    os.symlink(os.path.join(build_emu.HERE, "include"), tmp / "include")
    mp = pytest.MonkeyPatch()
    mp.setattr(build_emu, "HERE", str(tmp))
    mp.setattr(build_emu, "GEN", str(tmp / "_gen"))
    try:
        return build_emu.build(force=True)
    finally:
        mp.undo()


@pytest.mark.parametrize("chroma", [0, 30])
@pytest.mark.parametrize("strip", [20, 0])
def test_nan_filled_buffers_match_oracle(monkeypatch, nan_fill_library, strip, chroma):
    """Every plane of the handle starts as NaN on the emulation (on a GPU this is a plain oracle check).  At chroma 0
    the a and b planes of the collapsed levels are never written: a kernel that read them would carry NaN into the
    conversion (NaN * 0 is NaN), which clips it to 0, far from the oracle.  chroma 30 % checks the fill itself."""
    w, h, levels = 200, 136, 5
    if nan_fill_library:
        from lvm_b200 import capi
        monkeypatch.setattr(capi, "LIB_PATH", nan_fill_library)
        monkeypatch.setattr(capi, "_lib", None)
    cfg, ocfg = make_cfgs(O.MODE_LAPLACE, 20, 50.0, 0.4, 3.0, chroma, levels)
    proc, oproc = processor(1, strip, 0), O.MagnificationProcessor()
    for t in range(6):
        f = synth_frame(t, w, h, 3)
        dbg = {}
        produced, out = proc.process_image(f, cfg)
        oprod, oout = oproc.process(f, ocfg, dbg)
        assert produced and oprod
        got = proc.float_output(w, h, 3)[0]
        assert float(np.abs(got - dbg["output_bgr_f32"]).max()) < F32_TOL, t
        assert int(u8_diff(out, oout).max()) <= 1, t
    proc.close()
