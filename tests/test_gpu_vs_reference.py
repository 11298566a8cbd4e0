"""CUDA path (through the C ABI) checked DIRECTLY against the original project's own code on a B200.

The checker here is what the original's sources returned (src/processing/** compiled unmodified against OpenCV's
kernels, oracle/build_ref.py) on the same frames: the oracle reproduces each of those outputs and ``ref_pin`` holds
the reproduction bit-exact to the original's through stored digests (tests/refpin.py).  Same tolerances as the
oracle-based tests: Laplace / Color <= 1 LSB free-running, Phase <= 3 LSB and >= 99.5 % identical free-running;
passthrough decisions identical."""
import os

import numpy as np
import pytest

import lvm_b200 as L
from lvm_b200.synth import synth_frame
from oracle import livim_oracle as O
from oracle import livim_ref
from common import make_cfgs, u8_diff
from refpin import ref_pin  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def pair(pin, mode, amp, wl, lo, hi, chroma, levels, fps=30.0):
    """-> (product config, oracle config, the original's config (None unless recording))."""
    cfg, ocfg = make_cfgs(mode, amp, wl, lo, hi, chroma, levels, fps)
    return cfg, ocfg, (livim_ref.to_ref_config(pin.R, ocfg) if pin.R is not None else None)


@pytest.mark.parametrize("w,h,c,levels,chroma", [(320, 240, 3, 4, 50), (640, 480, 3, 4, 0), (241, 135, 1, 5, 0), (1920, 1080, 3, 6, 0)])
def test_laplace_vs_compiled_reference(w, h, c, levels, chroma, ref_pin):
    cfg, ocfg, rcfg = pair(ref_pin, O.MODE_LAPLACE, 20, 50.0, 0.4, 3.0, chroma, levels)
    proc, ref, oproc = L.MagnificationProcessor(0), ref_pin.ref(lambda R: R.Processor()), O.MagnificationProcessor()
    for t in range(6 if w > 1000 else 16):
        f = synth_frame(t, w, h, c)
        rprod, rout = ref_pin.process(ref, oproc, f, ocfg, rcfg, t)
        produced, out = proc.process_image(f, cfg)
        assert produced == rprod, t
        assert int(u8_diff(out, rout).max()) <= 1, t


def test_color_vs_compiled_reference(ref_pin):
    cfg, ocfg, rcfg = pair(ref_pin, O.MODE_COLOR, 100, 0.0, 0.8, 1.2, 0, 3, 8.0)
    proc, ref, oproc = L.MagnificationProcessor(0), ref_pin.ref(lambda R: R.Processor()), O.MagnificationProcessor()
    for t in range(24):   # every warm-up DFT length up to the 16-column cap, then the rolling window
        f = synth_frame(t, 320, 240, 3, fps=8.0)
        rprod, rout = ref_pin.process(ref, oproc, f, ocfg, rcfg, t)
        produced, out = proc.process_image(f, cfg)
        assert produced == rprod, t
        if produced:
            assert int(u8_diff(out, rout).max()) <= 1, t


def test_phase_vs_compiled_reference(ref_pin):
    cfg, ocfg, rcfg = pair(ref_pin, O.MODE_PHASE, 50, 50.0, 0.4, 3.0, 0, 4)
    proc, ref, oproc = L.MagnificationProcessor(0), ref_pin.ref(lambda R: R.Processor()), O.MagnificationProcessor()
    for t in range(12):
        f = synth_frame(t, 480, 270, 3)
        rprod, rout = ref_pin.process(ref, oproc, f, ocfg, rcfg, t)
        produced, out = proc.process_image(f, cfg)
        assert produced == rprod, t
        if produced:
            d = u8_diff(out, rout)
            assert int(d.max()) <= 3 and float((d == 0).mean()) >= 0.995, (t, int(d.max()), float((d == 0).mean()))


def test_chain_vs_compiled_reference(ref_pin):
    cfg, ocfg = make_cfgs(O.MODE_LAPLACE, 20, 50.0, 0.4, 3.0, 20, 4)
    cfg.grayscale = ocfg.grayscale = True
    cfg.preprocess = L.PreprocessParams(2, True, 0.1, 0.2, 0.77, 0.61)
    ocfg.preprocess = O.PreprocessParams(2, True, 0.1, 0.2, 0.77, 0.61)
    rcfg = livim_ref.to_ref_config(ref_pin.R, ocfg) if ref_pin.R is not None else None
    chain, rchain, omag = L.ProcessingChainB200(0), ref_pin.ref(lambda R: R.Chain()), O.MagnificationProcessor()
    for t in range(5):
        f = synth_frame(t, 641, 479, 3)
        rcur, rorig, _cur_same, _orig_same = O.run_chain_once(omag, f, ocfg)
        ref_pin.check(lambda: rchain.process(f, rcfg)[:2], (rcur, rorig), f"frame {t}: processed, original tap")
        cur, orig = chain.run_chain_once(L.Frame(image=f, seq=t), cfg)
        assert np.array_equal(orig.image, rorig), t                 # integer front stages: bit-exact
        assert cur.image.shape == rcur.shape and int(u8_diff(cur.image, rcur).max()) <= 1, t


@pytest.mark.skipif(livim_ref.load() is None and os.environ.get("MC_REQUIRE_REF") != "1",
                    reason="runs the original project's compiled front stages: needs oracle/_ref/_livim_ref")
def test_dropin_chain_on_gpu():
    """The drop-in as a maintainer would build it: the reference's PreprocessProcessor and GrayscaleProcessor
    (compiled reference code), MagnificationProcessorB200 (the product's adapter, compiled against the real
    reference headers) as the third stage, driven by the reference's runChainOnce — against the all-reference chain."""
    from lvm_b200 import capi
    R = livim_ref.load()
    assert R is not None, "MC_REQUIRE_REF=1 but oracle/_ref/_livim_ref is missing"
    R.set_magcore_library(capi.LIB_PATH)   # libmagcore_b200.so (tests/cuda_emu's build when MC_EMU=1)
    for mode, ui, gray, pre in ((O.MODE_LAPLACE, (20, 50.0, 0.4, 3.0, 30, 4), False, (2, True, 0.1, 0.1, 0.8, 0.8)),
                                (O.MODE_LAPLACE, (20, 50.0, 0.4, 3.0, 0, 3), True, (1, False, 0.0, 0.0, 1.0, 1.0)),
                                (O.MODE_COLOR, (100, 0.0, 0.8, 1.2, 0, 2), False, (4, False, 0.0, 0.0, 1.0, 1.0)),
                                (O.MODE_PHASE, (50, 50.0, 0.4, 3.0, 0, 3), False, (2, False, 0.0, 0.0, 1.0, 1.0))):
        _, ocfg = make_cfgs(mode, *ui)
        ocfg.grayscale = gray
        ocfg.preprocess = O.PreprocessParams(*pre)
        rcfg = livim_ref.to_ref_config(R, ocfg)
        dropin, ref = R.DropInChain(0), R.Chain()
        for t in range(8):
            f = synth_frame(t, 640, 480, 3)
            cur, orig, cur_is_in, orig_is_in, is_gray = dropin.process(f, rcfg)
            rcur, rorig, rcur_is_in, rorig_is_in, ris_gray = ref.process(f, rcfg)
            assert (cur_is_in, orig_is_in, is_gray) == (rcur_is_in, rorig_is_in, ris_gray), (mode, t)
            assert np.array_equal(orig, rorig), (mode, t)
            d = u8_diff(cur, rcur)
            if mode == O.MODE_PHASE:
                assert int(d.max()) <= 3 and float((d == 0).mean()) >= 0.995, (t, int(d.max()))
            else:
                assert int(d.max()) <= 1, (mode, t, int(d.max()))
        dropin.reset()
