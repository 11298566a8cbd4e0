"""bench.py contract checks that need no GPU: the reference arm runs on the host and prints exactly one JSON
line with the keys the driver reads; the product arm refuses to run without a B200 (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"] == "1080p frames/sec (Laplace, 6-level)" and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    from oracle import livim_ref
    assert cb["kind"] == ("reference" if livim_ref.load() is not None else "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert "workload" in d["config"]


def test_product_arm_needs_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_kernel_table_accounting():
    """bench.kernel_table: interface / algorithmic byte models per kernel (no GPU needed), for the default data flow
    (level kernels store their band, option band_from_state = 0) and for the shipped default band_from_state = 1; ncu
    captures are only quoted for kernels whose interface still matches the capture."""
    sys.path.insert(0, ROOT)
    import bench
    px = bench.level_pixels(1920, 1080, 6)
    prof = {("ingest_lab", 0): (20, 10.3), ("egress", 0): (20, 8.0), ("level", 1): (20, 4.0), ("level", 2): (20, 1.3),
            ("collapse", 2): (20, 0.6), ("collapse", 4): (20, 0.2)}
    table, traffic = bench.kernel_table(prof, 32)
    by = {t["kernel"]: t for t in table}
    assert [t["kernel"] for t in table][0] == "ingest_lab[0]"                       # sorted by time share
    assert by["level[1]"]["interface_bytes"] == 32 * 3 * (16 * px[1] + 8 * px[1] + 4 * px[2])
    assert by["collapse[2]"]["interface_bytes"] == 32 * 3 * (8 * px[2] + 4 * px[3])
    assert by["egress[0]"]["interface_bytes"] == 32 * 3 * (3 * px[0] + 4 * px[1] + 4 * px[2])
    assert abs(by["level[1]"]["algorithmic_GBps"] - 16 * 3 * px[1] * 32 / 200e-6 / 1e9) < 1e-6
    assert abs(sum(t["share"] for t in table) - 1.0) < 1e-9
    assert "ingest_lab[0]" in traffic and "level[1]" not in traffic and "egress[0]" not in traffic   # captures are of the shipped flow
    table2, traffic2 = bench.kernel_table(prof, 32, band_from_state=True)
    by2 = {t["kernel"]: t for t in table2}
    assert by2["level[1]"]["interface_bytes"] == 32 * 3 * (16 * px[1] + 4 * px[1] + 4 * px[2])
    assert by2["collapse[2]"]["interface_bytes"] == 32 * 3 * (12 * px[2] + 4 * px[3])
    assert by2["collapse[4]"]["interface_bytes"] == 32 * 3 * (12 * px[4] + 8 * px[5])  # top band comes from state planes
    assert by2["egress[0]"]["interface_bytes"] == 32 * 3 * (3 * px[0] + 8 * px[1] + 4 * px[2])
    assert {"ingest_lab[0]", "egress[0]", "level[1]", "level[2]"} <= set(traffic2)  # round-2 captures: band rebuilt from state


@pytest.mark.emu
def test_product_arm_dry_run_on_emulation(monkeypatch, tmp_path):
    """bench.run_ours end to end (device-resident loop, output dump, pipelined e2e loop, per-kernel table, CPU baseline,
    JSON line) with the kernels on the CUDA-on-CPU emulation and a stand-in for the handful of torch.cuda calls it
    makes, at a tiny frame size.  Guards the bench's own logic in the GPU-less container; the numbers mean nothing."""
    import time
    import types
    if torch.cuda.is_available():
        pytest.skip("GPU present: the real bench runs")
    sys.path.insert(0, ROOT)
    import bench
    import conftest
    from lvm_b200 import capi
    saved = (capi.LIB_PATH, capi._lib)
    conftest.use_emulated_library()

    class FakeEvent:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, stream=None):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    real_empty = torch.empty
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "ExternalStream", lambda ptr, device=None: types.SimpleNamespace(ptr=ptr))
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    monkeypatch.setattr(torch, "empty", lambda *a, **k: real_empty(*a, **{kk: v for kk, v in k.items() if kk != "device"}))
    monkeypatch.setattr(bench, "W", 192)
    monkeypatch.setattr(bench, "H", 108)
    monkeypatch.setattr(bench, "LEVELS", 4)
    monkeypatch.setitem(bench.UI, "levels", 4)
    try:
        args = types.SimpleNamespace(gpus=1, steps=3, warmup=3, lanes=2, clip_frames=2, cpu_frames=2, no_cpu_baseline=False,
                                     ref_frames_per_step=1, opt=[], workload="1080p6", dump_outputs=str(tmp_path / "out"))
        d = json.loads(bench.run_ours(args, 0, 1, 0))
    finally:
        capi.LIB_PATH, capi._lib = saved
    assert d["metric"] == "1080p frames/sec (Laplace, 6-level)" and d["unit"] == "frames/s" and d["n_gpus"] == 1
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["steps"] == 3 and d["warmup"] == 3
    assert d["e2e"]["h2d_bytes_per_step"] == d["e2e"]["d2h_bytes_per_step"] == 2 * 192 * 108 * 3
    assert d["gpu_launches"] == 3 * 6                      # 4 levels: ingest, level 1-3, collapse 2, egress per step
    r = d["roofline"]
    assert r["bound"] == "hbm" and 0 < r["frac"] and r["fused_level_kernel"]["kernel"] == "level[1]"
    assert {k["kernel"] for k in r["kernels"]} >= {"ingest_lab[0]", "egress[0]", "level[1]", "level[2]", "level[3]", "collapse[2]"}
    assert d["cpu_baseline"]["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port")
    # 2 lanes of 192x108x3 fit the sample: the whole last output, in order
    import numpy as np
    vals, idx = np.load(tmp_path / "out" / "output.npy"), np.load(tmp_path / "out" / "output_index.npy")
    assert vals.dtype == np.float32 and idx.dtype == np.float64
    assert np.load(tmp_path / "out" / "output_shape.npy").tolist() == [2, 108, 192, 3]
    assert np.array_equal(idx, np.arange(2 * 108 * 192 * 3)) and 0 <= vals.min() and vals.max() <= 255 and vals.std() > 0


def test_dump_outputs_sample_is_fixed():
    """bench.dump_outputs: above its sample size the same seeded positions are written every time, within 64 MB."""
    import tempfile
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    out = torch.from_numpy(np.random.default_rng(1).integers(0, 256, (3, 1080, 1920, 3), dtype=np.uint8))
    with tempfile.TemporaryDirectory() as a, tempfile.TemporaryDirectory() as b:
        bench.dump_outputs(out, a)
        bench.dump_outputs(out, b)
        idx = np.load(os.path.join(a, "output_index.npy"))
        assert np.array_equal(idx, np.load(os.path.join(b, "output_index.npy")))
        assert len(idx) == bench.DUMP_SAMPLES and np.all(np.diff(idx) > 0)
        assert np.array_equal(np.load(os.path.join(a, "output.npy")), out.numpy().reshape(-1)[idx.astype(np.int64)])
        assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= 64 << 20
