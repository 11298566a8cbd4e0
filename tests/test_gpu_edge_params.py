"""Parameter and size corner cases through all three modes, checked against what the original project's own code
returned (reproduced by the oracle, held bit-exact to the original through stored digests, tests/refpin.py):
single-level pyramids, clamped level counts, zero amplification, thresholds at 0 and pi, cutoffs at 0 Hz / Nyquist /
beyond (degenerate Butterworth design), inverted cutoffs, a 1 fps window, black frames (Color: 0/0 in the min-max
stretch), 7x9 frames.  Passthrough decisions must be identical; outputs <= 1 LSB (Phase: <= 3 LSB, >= 99.5 % identical)."""
import numpy as np
import pytest

import lvm_b200 as L
from lvm_b200.synth import synth_frame
from oracle import livim_oracle as O
from oracle import livim_ref
from common import make_cfgs, u8_diff
from refpin import ref_pin  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def clip(w, h, n, fps=30.0):
    return [synth_frame(t, w, h, 3, fps=fps) for t in range(n)]


CASES = [
    ("riesz L=1", O.MODE_PHASE, (50, 50.0, 0.4, 3.0, 0, 1), 30.0, None),
    ("riesz L=2", O.MODE_PHASE, (50, 50.0, 0.4, 3.0, 0, 2), 30.0, None),
    ("riesz L=9 clamped", O.MODE_PHASE, (50, 50.0, 0.4, 3.0, 0, 9), 30.0, None),
    ("riesz threshold pi", O.MODE_PHASE, (50, 0.0, 0.4, 3.0, 0, 3), 30.0, None),
    ("riesz threshold 0", O.MODE_PHASE, (50, 100.0, 0.4, 3.0, 0, 3), 30.0, None),
    ("riesz alpha 0", O.MODE_PHASE, (0, 50.0, 0.4, 3.0, 0, 3), 30.0, None),
    ("riesz low 0 Hz", O.MODE_PHASE, (50, 50.0, 0.0, 3.0, 0, 3), 30.0, None),
    ("riesz high = Nyquist", O.MODE_PHASE, (50, 50.0, 0.4, 15.0, 0, 3), 30.0, None),
    ("riesz high > Nyquist", O.MODE_PHASE, (50, 50.0, 0.4, 20.0, 0, 3), 30.0, None),
    ("color L=1", O.MODE_COLOR, (100, 0.0, 0.8, 1.2, 0, 1), 8.0, None),
    ("color 0..0 Hz", O.MODE_COLOR, (100, 0.0, 0.0, 0.0, 0, 2), 8.0, None),
    ("color black", O.MODE_COLOR, (100, 0.0, 0.8, 1.2, 0, 2), 8.0, "black"),
    ("color alpha 0", O.MODE_COLOR, (0, 0.0, 0.8, 1.2, 0, 2), 8.0, None),
    ("color 1 fps", O.MODE_COLOR, (100, 0.0, 0.8, 1.2, 0, 2), 1.0, None),
    ("laplace alpha 0", O.MODE_LAPLACE, (0, 50.0, 0.4, 3.0, 0, 3), 30.0, None),
    ("laplace wavelength 0", O.MODE_LAPLACE, (20, 0.0, 0.4, 3.0, 0, 3), 30.0, None),
    ("laplace low > high, chroma 100", O.MODE_LAPLACE, (20, 50.0, 3.0, 0.4, 100, 3), 30.0, None),
    ("laplace alpha 200, 0 Hz .. Nyquist", O.MODE_LAPLACE, (200, 100.0, 0.0, 15.0, 0, 3), 30.0, None),
    ("laplace L=1", O.MODE_LAPLACE, (20, 50.0, 0.4, 3.0, 30, 1), 30.0, None),
    ("laplace 7x9", O.MODE_LAPLACE, (20, 50.0, 0.4, 3.0, 30, 3), 30.0, "7x9"),
    ("riesz 7x9", O.MODE_PHASE, (50, 50.0, 0.4, 3.0, 0, 3), 30.0, "7x9"),
    ("color 7x9", O.MODE_COLOR, (100, 0.0, 0.8, 1.2, 0, 3), 8.0, "7x9"),
]


@pytest.mark.parametrize("name,mode,ui,fps,special", CASES, ids=[c[0] for c in CASES])
def test_corner_case_matches_reference(name, mode, ui, fps, special, ref_pin):
    cfg, ocfg = make_cfgs(mode, *ui, fps)
    if special == "black":
        frames = [np.zeros((64, 96, 3), np.uint8) for _ in range(4)]
    elif special == "7x9":
        frames = clip(7, 9, 3, fps)
    else:
        frames = clip(96, 64, 6 if mode == O.MODE_COLOR else 4, fps)
    proc, ref, oproc = L.MagnificationProcessor(0), ref_pin.ref(lambda R: R.Processor()), O.MagnificationProcessor()
    rcfg = livim_ref.to_ref_config(ref_pin.R, ocfg) if ref_pin.R is not None else None
    for t, f in enumerate(frames):
        rprod, rout = ref_pin.process(ref, oproc, f, ocfg, rcfg, t)
        produced, out = proc.process_image(f, cfg)
        assert produced == bool(rprod), (name, t)
        if produced:
            d = u8_diff(out, rout)
            if mode == O.MODE_PHASE:
                assert int(d.max()) <= 3 and float((d == 0).mean()) >= 0.995, (name, t, int(d.max()))
            else:
                assert int(d.max()) <= 1, (name, t, int(d.max()))
