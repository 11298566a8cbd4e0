"""Pins the oracle (oracle/livim_oracle.py) against the original project's OWN hot-path code.

The original's sources (src/processing/**), compiled unmodified against the cvshim facade whose pixel operations are
the real OpenCV kernels in cv2 (oracle/build_ref.py), were run on every scenario below; what they returned is stored
as digests (tests/refpin.py, tests/golden/reference_digests.json).  The oracle, fed the same frames, must agree
BIT-EXACTLY: every u8 output, every passthrough decision, and the float temporal state (EMA planes, rolling window,
Riesz pyramids and IIR outputs).  CPU only.
"""
import os

import numpy as np
import pytest

from lvm_b200.synth import synth_frame
from oracle import livim_oracle as O
from oracle import livim_ref
from refpin import ref_pin  # noqa: F401  (fixture)

MAG_KEYS = ("amplification", "coWavelength", "coLow", "coHigh", "chromAttenuation", "levels", "framerate")


def cfg_pair(pin, mode, amp, wl, lo, hi, chroma, levels, fps=30.0, **extra):
    """-> (reference ProcessorConfig built by the reference's own toParams (None unless recording), oracle ProcessorConfig)."""
    oc = O.ProcessorConfig(magnification=O.to_params(mode, amp, wl, lo, hi, chroma, levels, fps))
    for k, v in extra.items():
        if k == "grayscale":
            oc.grayscale = v
        else:
            setattr(oc.preprocess, k, float(np.float32(v)) if isinstance(v, float) else v)
    rc = None
    if pin.R is not None:
        R = pin.R
        ui = R.MagUiValues()
        ui.mode = livim_ref.mode_enum(R, mode)
        ui.amplification, ui.wavelength, ui.low, ui.high, ui.chroma, ui.levels, ui.captureFps = amp, wl, lo, hi, chroma, levels, fps
        rc = R.ProcessorConfig()
        rc.magnification = R.toParams(ui)
        for k, v in extra.items():
            if k == "grayscale":
                rc.grayscale = v
            else:
                pp = rc.preprocess
                setattr(pp, k, v)
                rc.preprocess = pp
    # toParams restated exactly
    pin.check(lambda: [getattr(rc.magnification, k) for k in MAG_KEYS], [getattr(oc.magnification, k) for k in MAG_KEYS],
              "toParams")
    return rc, oc


def run_pair(pin, rc, oc, frames, rp=None, op=None):
    rp, op = rp or pin.ref(lambda R: R.Processor()), op or O.MagnificationProcessor()
    for t, f in enumerate(frames):
        po, oo = op.process(f, oc)
        pin.check(lambda: rp.process(f, rc), (po, oo if po else f), f"frame {t}: produced, output")
    return rp, op


# --------------------------------------------------------------------------------------------------
# scalar / host functions
# --------------------------------------------------------------------------------------------------
def test_host_functions_are_bit_identical(ref_pin):
    R = ref_pin.R
    sizes = [(w, h) for w in range(1, 70) for h in (1, 5, 6, 7, 11, 12, 13, 33, 64, 135, 1080)] + \
        [(1920, 1080), (3840, 2160), (640, 480)]
    ref_pin.check(lambda: [R.calculateMaxLevels(w, h) for w, h in sizes], [O.calculate_max_levels(w, h) for w, h in sizes],
                  "calculateMaxLevels")
    fpss = list(range(0, 130)) + [240, 1000]
    ref_pin.check(lambda: [R.getOptimalBufferSize(fps) for fps in fpss], [O.get_optimal_buffer_size(fps) for fps in fpss],
                  "getOptimalBufferSize")
    hz_fps = [(hz, fps) for hz in (0.0, -1.0, 0.05, 0.4, 1.0, 3.0, 14.9, 15.0, 100.0) for fps in (30.0, 0.0, -5.0, 24.0, 59.94)]
    ref_pin.check(lambda: [R.motionHzToBlend(hz, fps) for hz, fps in hz_fps],
                  [O.motion_hz_to_blend(hz, fps) for hz, fps in hz_fps], "motionHzToBlend")
    for wn in (0.4 / 15, 3.0 / 15, 0.8 / 15, 0.5, 0.9, 1e-3, 0.0):
        oa, ob = O.butterworth(2, wn)
        ref_pin.check(lambda: [np.array(x) for x in R.butterworth(2, wn)], [np.array(oa), np.array(ob)], f"butterworth {wn}")


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_to_params_matches_reference(mode, ref_pin):
    for amp, wl, lo, hi, chroma, levels, fps in ((20, 50.0, 0.4, 3.0, 50, 6, 30.0), (100, 0.0, 0.8, 1.2, 0, 3, 24.0),
                                                 (7, 99.5, 0.0, 14.0, 100, 1, 60.0)):
        cfg_pair(ref_pin, mode, amp, wl, lo, hi, chroma, levels, fps)


# --------------------------------------------------------------------------------------------------
# Motion (Laplace)
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,c,levels,chroma", [(96, 64, 3, 4, 50), (97, 67, 3, 3, 0), (131, 75, 1, 4, 0), (64, 48, 3, 9, 100)])
def test_laplace_outputs_and_state_bit_exact(w, h, c, levels, chroma, ref_pin):
    rc, oc = cfg_pair(ref_pin, 0, 20, 50.0, 0.4, 3.0, chroma, levels)
    core, st = ref_pin.ref(lambda R: R.Core()), O.MotionState()
    lv = min(max(levels, 1), O.calculate_max_levels(w, h))
    for t in range(7):
        f = synth_frame(t, w, h, c)
        po, oo = O.magnify_motion(f, oc.magnification, lv, c, st)
        assert po, t
        ref_pin.check(lambda: core.run(0, f, rc.magnification, lv), (po, oo), f"frame {t}: produced, output")
        assert len(st.lowpassHi) == len(st.lowpassLo) == lv + 1
        ref_pin.check(lambda: core.motion_state(), (st.lowpassHi, st.lowpassLo), f"frame {t}: lowpassHi / lowpassLo, every level")
    # the same through MagnificationProcessor (levels clamp + tracker)
    run_pair(ref_pin, rc, oc, [synth_frame(t, w, h, c) for t in range(5)])


def test_laplace_live_parameter_changes_resets_and_passthrough(ref_pin):
    w, h = 80, 60
    frames = [synth_frame(t, w, h, 3) for t in range(12)]
    rc, oc = cfg_pair(ref_pin, 0, 20, 50.0, 0.4, 3.0, 30, 3)
    rp, op = run_pair(ref_pin, rc, oc, frames[:4])
    rc2, oc2 = cfg_pair(ref_pin, 0, 45, 20.0, 0.0, 5.0, 80, 3)          # non-structural: alpha, wavelength, cutoffs (coLow = 0), chroma
    run_pair(ref_pin, rc2, oc2, frames[4:7], rp, op)
    rc3, oc3 = cfg_pair(ref_pin, 0, 45, 20.0, 0.0, 5.0, 80, 2)          # structural: levels -> state reset
    run_pair(ref_pin, rc3, oc3, frames[7:9], rp, op)
    run_pair(ref_pin, rc3, oc3, [synth_frame(t, 70, 50, 3) for t in range(3)], rp, op)   # structural: size
    run_pair(ref_pin, rc3, oc3, [synth_frame(t, 70, 50, 1) for t in range(3)], rp, op)   # structural: channels
    rcn, ocn = cfg_pair(ref_pin, 3, 45, 20.0, 0.0, 5.0, 80, 2)          # mode None: identity, frees state
    run_pair(ref_pin, rcn, ocn, frames[9:10], rp, op)
    run_pair(ref_pin, rc3, oc3, frames[10:12], rp, op)
    rp.reset(); op.reset()
    run_pair(ref_pin, rc3, oc3, frames[:2], rp, op)
    run_pair(ref_pin, rc, oc, [synth_frame(0, 5, 40, 3), synth_frame(1, 40, 5, 3), synth_frame(2, 6, 6, 3)], rp, op)   # <= 5 px: identity


def test_laplace_1080p_config2_first_frames(ref_pin):
    """BASELINE.json configs[1] (1920x1080x3, 6 levels) — the bench workload — two frames, bit-exact."""
    rc, oc = cfg_pair(ref_pin, 0, 20, 50.0, 0.4, 3.0, 0, 6)
    run_pair(ref_pin, rc, oc, [synth_frame(t, 1920, 1080, 3) for t in range(2)])


# --------------------------------------------------------------------------------------------------
# Color (Gaussian + ideal FFT)
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,c,levels,fps", [(96, 64, 3, 3, 8.0), (90, 70, 1, 2, 8.0), (64, 48, 3, 2, 12.0)])
def test_color_warmup_wraparound_and_window_bit_exact(w, h, c, levels, fps, ref_pin):
    rc, oc = cfg_pair(ref_pin, 2, 100, 0.0, 0.8, 1.2, 0, levels, fps)
    core, st = ref_pin.ref(lambda R: R.Core()), O.ColorState()
    n = O.get_optimal_buffer_size(int(fps)) + 5      # every DFT length 2..cap (odd ones included), then the shift
    for t in range(n):
        f = synth_frame(t, w, h, c, fps=fps)
        po, oo = O.magnify_color(f, oc.magnification, levels, c, st)
        assert po == (t >= 1), t
        ref_pin.check(lambda: core.run(2, f, rc.magnification, levels), (po, oo), f"frame {t}: produced, output")
        ow = st.window if c > 1 else st.window[:, :, 0]
        ref_pin.check(lambda: core.color_window(), ow, f"frame {t}: window")


def test_color_framerate_change_and_zero_low_cutoff(ref_pin):
    w, h = 72, 56
    rc, oc = cfg_pair(ref_pin, 2, 60, 0.0, 0.0, 1.5, 0, 2, 12.0)        # coLow == 0 -> 0.01 Hz
    rp, op = run_pair(ref_pin, rc, oc, [synth_frame(t, w, h, 3) for t in range(20)])
    rc2, oc2 = cfg_pair(ref_pin, 2, 60, 0.0, 0.0, 1.5, 0, 2, 8.0)       # smaller cap mid-stream (window shrinks by one per frame)
    run_pair(ref_pin, rc2, oc2, [synth_frame(20 + t, w, h, 3) for t in range(12)], rp, op)


# --------------------------------------------------------------------------------------------------
# Phase (Riesz)
# --------------------------------------------------------------------------------------------------
RIESZ_PLANES = (("lowpass", lambda l: l.lowpass), ("rx", lambda l: l.rx), ("ry", lambda l: l.ry),
                ("amplitude", lambda l: l.amplitude), ("amplitude_blurred", lambda l: l.amplitude_blurred),
                ("phase_diff_cos", lambda l: l.phase_diff[0]), ("phase_diff_sin", lambda l: l.phase_diff[1]))
RIESZ_IIR = (("lowpass_iir_cos", lambda l: l.lowpass_iir[0]), ("lowpass_iir_sin", lambda l: l.lowpass_iir[1]),
             ("highpass_iir_cos", lambda l: l.highpass_iir[0]), ("highpass_iir_sin", lambda l: l.highpass_iir[1]))


@pytest.mark.parametrize("w,h,levels", [(96, 64, 3), (101, 77, 4)])
def test_riesz_outputs_and_every_state_plane_bit_exact(w, h, levels, ref_pin):
    rc, oc = cfg_pair(ref_pin, 1, 50, 50.0, 0.4, 3.0, 0, levels)
    core, st = ref_pin.ref(lambda R: R.Core()), O.RieszState()
    for t in range(6):
        f = synth_frame(t, w, h, 3)
        po, oo = O.magnify_riesz(f, oc.magnification, levels, 3, st)
        assert po == (t >= 1), t
        ref_pin.check(lambda: core.run(1, f, rc.magnification, levels), (po, oo), f"frame {t}: produced, output")
        if not po:
            continue
        for which, opyr in ((True, st.old), (False, st.cur)):
            names = RIESZ_PLANES + (() if which else RIESZ_IIR)
            ref_pin.check(lambda: [[rl[name] for name, _ in names] for rl in core.riesz_levels(which)],
                          [[get(ol) for _, get in names] for ol in opyr.levels],
                          f"frame {t}: every plane of the {'old' if which else 'cur'} pyramid")
    ref_pin.check(lambda: list(core.riesz_coefficients()), [st.lo.A, st.lo.B, st.hi.A, st.hi.B], "IIR coefficients")


def test_riesz_cutoff_change_gray_passthrough_and_processor(ref_pin):
    w, h = 88, 66
    frames = [synth_frame(t, w, h, 3) for t in range(10)]
    rc, oc = cfg_pair(ref_pin, 1, 50, 50.0, 0.4, 3.0, 0, 3)
    rp, op = run_pair(ref_pin, rc, oc, frames[:4])
    rc2, oc2 = cfg_pair(ref_pin, 1, 35, 70.0, 0.8, 3.0, 0, 3)           # low cutoff changes: redesign + register reset + old rebuilt
    run_pair(ref_pin, rc2, oc2, frames[4:6], rp, op)
    rc3, oc3 = cfg_pair(ref_pin, 1, 35, 70.0, 0.8, 2.0, 0, 3)           # high cutoff changes
    run_pair(ref_pin, rc3, oc3, frames[6:8], rp, op)
    rc4, oc4 = cfg_pair(ref_pin, 1, 35, 70.0, 0.8, 2.0, 0, 3, 25.0)     # framerate alone: coefficients are NOT recomputed
    run_pair(ref_pin, rc4, oc4, frames[8:10], rp, op)
    run_pair(ref_pin, rc, oc, [synth_frame(t, w, h, 1) for t in range(3)])   # gray input: silent passthrough


# --------------------------------------------------------------------------------------------------
# Front of the chain (SURVEY 8f-1): PreprocessProcessor -> GrayscaleProcessor -> MagnificationProcessor
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("extra", [
    dict(downscale=2), dict(downscale=4, grayscale=True), dict(downscale=8),
    dict(roiEnabled=True, roiX=0.1, roiY=0.2, roiW=0.55, roiH=0.6),
    dict(roiEnabled=True, roiX=0.13, roiY=0.07, roiW=0.61, roiH=0.77, downscale=2, grayscale=True),
    dict(roiEnabled=True, roiX=0.9, roiY=0.9, roiW=0.5, roiH=0.5, downscale=4),    # clamped to the frame
    dict(grayscale=True), dict(),
])
def test_chain_bit_exact(extra, ref_pin):
    w, h = 203, 151
    rc, oc = cfg_pair(ref_pin, 0, 20, 50.0, 0.4, 3.0, 40, 3, **extra)
    chain, omag = ref_pin.ref(lambda R: R.Chain()), O.MagnificationProcessor()
    for t in range(4):
        f = synth_frame(t, w, h, 3)
        ocur, oorig, o_cur_is_in, o_orig_is_in = O.run_chain_once(omag, f, oc)
        ref_pin.check(lambda: chain.process(f, rc)[:4], (ocur, oorig, o_cur_is_in, o_orig_is_in),
                      f"frame {t}: processed, original tap, processed is input, original is input")


# --------------------------------------------------------------------------------------------------
# The drop-in: reference chain + reference headers + the product's adapter (needs a B200 to run)
# --------------------------------------------------------------------------------------------------
@pytest.mark.skipif(livim_ref.load() is None and os.environ.get("MC_REQUIRE_REF") != "1",
                    reason="compiles the adapter against the original project's headers: needs oracle/_ref/_livim_ref")
def test_dropin_chain_builds_against_real_reference_headers_and_has_no_cpu_fallback(built):
    """oracle/_ref/_livim_ref also holds the reference's chain with the ONE substitution of INTEGRATION.md
    (MagnificationProcessorB200 at ChainBuilder.cpp:15), compiled against the reference's real IProcessor.hpp /
    Frame.hpp.  Without a GPU constructing it must fail loudly: mc_create reports no device, the adapter throws."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by tests/test_gpu_vs_reference.py::test_dropin_chain_on_gpu")
    R = livim_ref.load()
    assert R is not None, "MC_REQUIRE_REF=1 but oracle/_ref/_livim_ref is missing"
    R.set_magcore_library(built[0])
    with pytest.raises(RuntimeError, match="magcore_b200"):
        R.DropInChain(0)
