"""Results of the original project (tschnz/Live-Video-Magnification), stored as digests for tests that compare with it.

The original's own hot-path sources, compiled against oracle/cvshim (oracle/build_ref.py -> oracle/_ref/_livim_ref),
were run once on every scenario of the tests that use the ``ref_pin`` fixture, and a SHA-256 digest of each value
they returned is stored in tests/golden/reference_digests.json.  A test computes the same value with the oracle
(oracle/livim_oracle.py) and ``ref_pin.check`` requires it to equal the original's, bit for bit, through the digest.
The GPU tests then hold the CUDA path to that verified output, so they compare with the original without needing
its sources.

Digests treat +0.0 and -0.0 as equal and every NaN as equal, as ``np.array_equal(a, b, equal_nan=True)`` does;
shapes, dtypes, booleans and integers must match exactly.

Regenerating the digests needs the original's sources (oracle/build_ref.py, LIVIM_REFERENCE_SRC).  With
MC_REF_RECORD=1 the tests run the compiled original beside the oracle, assert that the two agree, and rewrite the
entries of the tests that ran:
    MC_REF_RECORD=1 python -m pytest tests/test_ref_pin.py
    MC_EMU=1 MC_REF_RECORD=1 python -m pytest -m gpu tests/test_gpu_vs_reference.py tests/test_gpu_edge_params.py
"""
import hashlib
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
RECORD = os.environ.get("MC_REF_RECORD") == "1"


def _feed(h, v):
    if v is None:
        h.update(b"N;")
    elif isinstance(v, (bool, np.bool_)):
        h.update(b"b%d;" % bool(v))
    elif isinstance(v, (int, np.integer)):
        h.update(b"i%d;" % int(v))
    elif isinstance(v, (float, np.floating)):
        h.update(b"f%s;" % repr(float(v) + 0.0).encode())
    elif isinstance(v, (list, tuple)):
        h.update(b"[%d;" % len(v))
        for x in v:
            _feed(h, x)
    elif isinstance(v, np.ndarray):
        a = np.ascontiguousarray(v)
        if a.dtype.kind == "f":
            a = a + a.dtype.type(0)          # -0.0 -> +0.0
            a[np.isnan(a)] = np.nan          # one NaN bit pattern
        h.update(f"a{a.dtype.str}{a.shape};".encode())
        h.update(a.tobytes())
    else:
        raise TypeError(f"no digest for {type(v).__name__}")


def digest(v) -> str:
    """SHA-256 (first 128 bits, hex) of a value: None, bool, int, float, ndarray, or lists / tuples of these."""
    h = hashlib.sha256()
    _feed(h, v)
    return h.hexdigest()[:32]


class _Absent:
    """Stands in for an object of the compiled original when it is not loaded: every method is a no-op."""

    def __getattr__(self, name):
        return lambda *a, **k: None


class RefPin:
    def __init__(self, key, stored, reference):
        self.key, self.i = key, 0
        self.R = reference                   # the compiled original (recording) or None (checking digests)
        self.seq = [] if reference is not None else stored.get(key)
        if self.seq is None:
            pytest.fail(f"{key}: no digests in {os.path.relpath(GOLDEN)}; record them (see tests/refpin.py)")

    def ref(self, make):
        """make(R) -> an object of the compiled original when recording, else a stand-in whose methods do nothing."""
        return make(self.R) if self.R is not None else _Absent()

    def check(self, ref_call, value, what=""):
        """value (computed by the oracle) must equal ref_call() of the original: live when recording, else by digest."""
        d = digest(value)
        if self.R is not None:
            rd = digest(ref_call())
            assert rd == d, f"{self.key} check {self.i} ({what}): the oracle differs from the original"
            self.seq.append(rd)
        else:
            assert self.i < len(self.seq), f"{self.key}: more checks than recorded digests"
            assert d == self.seq[self.i], f"{self.key} check {self.i} ({what}): differs from the original's result"
        self.i += 1

    def process(self, ref, oracle, frame, ocfg, rcfg, what=""):
        """(produced, output) of the original's MagnificationProcessor ``ref`` for the next frame, as the oracle's
        processor reproduces it; the frame itself when it passes through."""
        produced, out = oracle.process(frame, ocfg)
        self.check(lambda: ref.process(frame, rcfg), (produced, out), f"frame {what}: produced, output")
        return produced, out


def _load():
    if os.path.exists(GOLDEN):
        with open(GOLDEN) as f:
            return json.load(f)
    return {}


@pytest.fixture
def ref_pin(request):
    """RefPin for this test (key: module::test[params])."""
    R = None
    if RECORD:
        from oracle import livim_ref
        R = livim_ref.load()
        assert R is not None, "MC_REF_RECORD=1 needs the compiled original (oracle/_ref/_livim_ref)"
    stored = _load()
    pin = RefPin(f"{request.node.path.stem}::{request.node.name}", stored, R)
    yield pin
    if R is not None:
        stored = _load()
        stored[pin.key] = pin.seq
        with open(GOLDEN, "w") as f:
            json.dump(dict(sorted(stored.items())), f, indent=0)
            f.write("\n")
    else:
        assert pin.i == len(pin.seq), f"{pin.key}: {pin.i} checks ran, {len(pin.seq)} recorded"
