"""bench.py contract: the reference arm prints the agreed JSON line; the product arm refuses to run without a GPU (no
CPU fallback); the clock sampler degrades to an explicit "unavailable" record; on the GPU (-m gpu), --steps is the
number of timed steps and --dump-outputs writes what the last of them computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, timeout=600)


def test_reference_arm_prints_the_contract_line():
    out = run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "encode+decode Mpixel/s" and d["unit"] == "Mpixel/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "u8" and d["data"] == "synthetic"
    assert "workload" in d["config"] and d["config"]["levels"] == 4
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    out = run("--steps", "1", "--warmup", "3", "--no-e2e", "--no-cpu")
    assert out.returncode != 0
    assert not any(l.startswith("{") and '"value"' in l for l in out.stdout.splitlines())


def test_clock_sampler_reports_unavailability():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.start()
    r = s.stop()
    assert r["sm_mhz"] is None and r["reasons"]


def test_arguments_it_cannot_honour_are_refused():
    for args in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", "out")):
        out = run(*args)
        assert out.returncode == 2 and "error:" in out.stderr, args


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_steps_outputs(tmp_path):
    """8 frames are one launch per encode and per decode, so the launch count gives the number of timed steps; the
    dumped sample equals the oracle's outputs for the bench's frames at the seeded positions."""
    from oracle import c as oc
    sys.path.insert(0, ROOT)
    import bench
    out = run("--frames", "8", "--steps", "5", "--warmup", "0", "--no-e2e", "--no-cpu", "--no-extra",
              "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 5 and d["gpu_launches"] == 5 * 4
    names = [f"{kind}_{q}" for q in ("lossless", "medium") for kind in ("grid", "decoded")]
    assert sorted(os.listdir(tmp_path)) == sorted(f"{n}_{part}.npy" for n in names for part in ("frame", "sample"))
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20
    yy, xx = np.mgrid[0:bench.H, 0:bench.W]
    frames = np.stack([((xx * yy + 31 * k) & 255).astype(np.uint8) for k in range(8)])
    frame, pix = bench.dump_positions(8)
    for q, qname in zip(bench.QLEVELS, ("lossless", "medium")):
        grids = oc.encode_batch(frames, bench.LEVELS, qlevel=q)
        for kind, want in (("grid", grids), ("decoded", oc.decode_batch(grids, bench.LEVELS))):
            got_frame = np.load(tmp_path / f"{kind}_{qname}_frame.npy")
            got_sample = np.load(tmp_path / f"{kind}_{qname}_sample.npy")
            assert got_frame.dtype == got_sample.dtype == np.float32
            assert (got_frame == want[frame]).all(), (kind, qname)
            assert (got_sample == want.reshape(-1)[pix]).all(), (kind, qname)
