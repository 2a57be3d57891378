"""bench.py --dump-outputs on the device path: the files hold exactly the ciphertexts that the timed MulRelinNew + Rescale
steps return for bench.py's seeded inputs (checked against the CPU oracle), a second run with the same arguments writes the
same files, and --steps sets how many steps are timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRESET, BATCH = "CKKS_N15QP881", 2
NAMES = ("ct_out_hi32", "ct_out_lo32", "ct_out_index", "ct_out_shape")


def _bench(d, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--preset", PRESET, "--batch", str(BATCH), "--steps", str(steps),
                        "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(d)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1]), {n: np.load(os.path.join(d, n + ".npy")) for n in NAMES}


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    d = tmp_path_factory.mktemp("dump")
    return _bench(d / "one_step", 1), _bench(d / "three_steps", 3)


def _bench_inputs():
    """The evaluation key and ciphertexts of bench.py's rank 0: same generator seed, same draw order."""
    import torch
    from lattigo_b200 import params as presets
    s = presets.PRESETS[PRESET]
    Q, P, N = s["Q"], s["P"], 1 << s["logN"]
    nd = (len(Q) + len(P) - 1) // len(P)
    g = torch.Generator(device="cuda"); g.manual_seed(1000)

    def rand_rows(mods, lead):
        out = torch.empty(tuple(lead) + (len(mods), N), dtype=torch.int64, device="cuda")
        for i, m in enumerate(mods):
            out[..., i, :] = torch.randint(0, m, tuple(lead) + (N,), generator=g, device="cuda", dtype=torch.int64)
        return out.cpu().numpy().view(np.uint64)

    evk = rand_rows(Q + P, (nd, 1, 2))
    return s, evk, rand_rows(Q, (BATCH, 2)), rand_rows(Q, (BATCH, 2))


def _residues(files):
    return (files["ct_out_hi32"].astype(np.uint64) << np.uint64(32)) | files["ct_out_lo32"].astype(np.uint64)


def test_dump_is_the_timed_output(runs):
    (_, files), _ = runs
    s, evk, a, b = _bench_inputs()
    Q, P = s["Q"], s["P"]
    params = O.Parameters(s["logN"], Q, P)
    ev = O.CKKSEvaluator(params, O.GadgetCiphertext(evk, len(Q), len(P)))
    want = np.stack([np.stack(ev.Rescale(ev.MulRelinNew([a[i, 0], a[i, 1]], [b[i, 0], b[i, 1]]))) for i in range(BATCH)])
    assert tuple(files["ct_out_shape"].astype(np.int64)) == want.shape
    idx = files["ct_out_index"].astype(np.int64)
    assert len(idx) > 0 and (np.diff(idx) > 0).all()
    assert np.array_equal(_residues(files), want.reshape(-1)[idx])


def test_dump_repeats_and_steps_are_timed(runs):
    (one, f1), (three, f3) = runs
    for n in NAMES:
        assert np.array_equal(f1[n], f3[n]), n
    assert one["steps"] == 1 and three["steps"] == 3
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
