"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`, the oracle port on the host
cores) prints one JSON line with the agreed keys, and the product arm fails loudly when there is no CUDA device
(no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--preset", "BGV_N15QP880"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "ct/s" and line["higher_is_better"] is True
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "ct/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["workload"] == "ckks_mulrelin_rescale" and line["config"]["preset"] == "BGV_N15QP880"


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-e2e", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0                      # loud failure, never a silent CPU path
    assert not any(l.startswith("{") for l in r.stdout.splitlines())


def test_bootstrap_workload_reference_arm_is_declared_unavailable():
    """BASELINE config 5 is an op-trace replay of the device path; there is no CPU restatement of circuits/ckks/bootstrapping, and the
    reference arm says so in the contract's `unavailable` form instead of timing something else."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "bootstrap", "--preset", "BOOT_N16QP1767"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and "unavailable" in line


def test_dump_outputs_sample_is_fixed_exact_and_bounded(tmp_path):
    """--dump-outputs at the headline shape (64 x 2 x 43 x 2^16 residues): the sampled positions are the same on every run,
    distinct and in range, residues up to 2^56 - 1 come back exactly from the float64 files, and the files stay under 64 MB."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    shape = (64, 2, 43, 1 << 16)
    n = int(np.prod(shape))
    idx = bench.dump_sample_index(n)
    assert np.array_equal(idx, bench.dump_sample_index(n))
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < n
    assert np.array_equal(bench.dump_sample_index(100), np.arange(100))
    vals = np.random.default_rng(5).integers(0, 1 << 56, len(idx), dtype=np.uint64)
    vals[:2] = [0, (1 << 56) - 1]
    bench.write_dump(str(tmp_path), shape, idx, vals)
    files = {f.name[:-4]: np.load(f) for f in tmp_path.iterdir()}
    assert sorted(files) == ["ct_out_hi32", "ct_out_index", "ct_out_lo32", "ct_out_shape"]
    assert all(a.dtype == np.float64 for a in files.values())
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20
    got = (files["ct_out_hi32"].astype(np.uint64) << np.uint64(32)) | files["ct_out_lo32"].astype(np.uint64)
    assert np.array_equal(got, vals) and np.array_equal(files["ct_out_index"].astype(np.int64), idx)
    assert tuple(files["ct_out_shape"].astype(np.int64)) == shape


def test_dump_outputs_is_refused_where_nothing_is_dumped(tmp_path):
    for extra in (["--impl", "reference"], ["--workload", "bootstrap"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "d")] + extra,
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr
        assert not (tmp_path / "d").exists()


def test_clock_sampler_keeps_the_samples_of_the_timed_region():
    """ClockSampler.stop(t0, t1): only lines that arrived during the timed region count (the poller runs from before the warm-up);
    throttle reasons outside it are not reported, reasons inside it are; a region shorter than the polling period keeps the nearest lines."""
    sys.path.insert(0, ROOT)
    import bench

    class FakeProc:
        def terminate(self): pass
        def wait(self, timeout=None): return 0
        def kill(self): pass

    def line(sm, hw="Not Active", pw="Not Active"):
        return "0, %d, 1965, 700.0, 0x0, %s, Not Active, Not Active, %s" % (sm, hw, pw)

    s = bench.ClockSampler(0)
    s.proc = FakeProc()
    s.lines = [(9.0, line(1200, hw="Active")), (10.05, line(1965)), (10.15, line(1950, pw="Active")), (10.25, line(1965)), (11.0, line(900, hw="Active"))]
    r = s.stop(10.0, 10.3)
    assert r["samples"] == 3 and r["sm_mhz"] == 1965.0 and r["sm_max_mhz"] == 1965.0 and r["reasons"] == ["sw_power_cap"]
    s = bench.ClockSampler(0)
    s.proc = FakeProc()
    s.lines = [(9.0, line(1200)), (10.02, line(1965)), (11.0, line(900))]
    r = s.stop(10.0, 10.01)                       # shorter than the polling period: nearest samples
    assert r["samples"] == 3 and r["sm_mhz"] == 1200.0
    assert bench.ClockSampler(0).stop()["reasons"] == ["nvidia-smi unavailable"]
