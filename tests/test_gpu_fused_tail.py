"""MulRelin + Rescale through the merged ModDown + Rescale tail (the default) against the two-pass tail (LGPU_FZ_RESCALE=0) and the
oracle, bit for bit: presets CKKS_L44 (FP64-pipe rows, 56-bit q0) and BOOT_N16QP1767 (integer rows, 60 / 61-bit moduli, 6 P limbs),
N = 2^13 and 2^16, levels L, L - 1 and 1, batches 1, 3 and 64 (the batch-1 and batch-3 results must equal the first rows of the
batch-64 one). The switch is read once per process, so the two-pass results come from a subprocess."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
U64 = np.uint64
HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [(preset, logN, lv) for preset in ("CKKS_L44", "BOOT_N16QP1767") for logN in (13, 16) for lv in ("L", "L-1", "1")]


def _case(preset, logN, lv, batches=(64, 3, 1)):
    """(level, {batch: [sha256 of each output ciphertext]}, host copies of inputs / key / output 0 for the oracle)"""
    import torch
    import lattigo_b200 as lb
    from lattigo_b200 import params as presets
    s = presets.PRESETS[preset]
    q, p = s["Q"], s["P"]
    ctx = lb.Context(logN, q, p)
    N = 1 << logN
    L, levelP = len(q) - 1, len(p) - 1
    level = {"L": L, "L-1": L - 1, "1": 1}[lv]
    nd = (L + levelP + 1) // (levelP + 1)
    g = torch.Generator(device="cuda")
    g.manual_seed(1000 * logN + len(q) + level)

    def rows(mods, lead):
        out = torch.empty(tuple(lead) + (len(mods), N), dtype=torch.int64, device="cuda")
        for i, m in enumerate(mods):
            out[..., i, :] = torch.randint(0, m, tuple(lead) + (N,), generator=g, device="cuda", dtype=torch.int64)
        return out

    evk_t = rows(q + p, (nd, 1, 2))
    rlk = lb.GadgetCiphertext(ctx, evk_t, L, levelP)
    ev = lb.CKKSEvaluator(ctx, rlk)
    a = rows(q[: level + 1], (max(batches), 2))
    b = rows(q[: level + 1], (max(batches), 2))
    digests = {}
    host = None
    for nb in batches:
        out = ev.MulRelinRescaleNew(a[:nb].contiguous(), b[:nb].contiguous())
        torch.cuda.synchronize()
        assert tuple(out.shape) == (nb, 2, level, N)
        oh = ctx.to_host(out)
        digests[nb] = [hashlib.sha256(np.ascontiguousarray(oh[i]).tobytes()).hexdigest() for i in range(nb)]
        if nb == 1:
            host = dict(a=ctx.to_host(a[:1]), b=ctx.to_host(b[:1]), evk=ctx.to_host(evk_t), out=oh[0], q=q, p=p, level=level, L=L)
    ctx.close()
    return level, digests, host


@pytest.fixture(scope="module")
def two_pass_digests(tmp_path_factory):
    path = tmp_path_factory.mktemp("fz") / "two_pass.json"
    code = ("import json, sys; sys.path.insert(0, %r); from tests.test_gpu_fused_tail import CASES, _case\n"
            "json.dump({'|'.join(map(str, c)): _case(*c)[1] for c in CASES}, open(%r, 'w'))") % (os.path.dirname(HERE), str(path))
    r = subprocess.run([sys.executable, "-c", code], cwd=os.path.dirname(HERE), env=dict(os.environ, LGPU_FZ_RESCALE="0"),
                       capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return {k: {int(nb): d for nb, d in v.items()} for k, v in json.load(open(path)).items()}


@pytest.mark.parametrize("preset,logN,lv", CASES)
def test_merged_tail_matches_two_pass_tail_and_oracle(preset, logN, lv, two_pass_digests):
    from oracle import oracle as O
    level, digests, host = _case(preset, logN, lv)
    assert digests == two_pass_digests["|".join(map(str, (preset, logN, lv)))]
    for nb in (3, 1):
        assert digests[nb] == digests[64][:nb]
    q, p, L = host["q"], host["p"], host["L"]
    params = O.Parameters(logN, q, p)
    ev_o = O.CKKSEvaluator(params, O.GadgetCiphertext(host["evk"], L + 1, len(p)))
    a, b = host["a"][0], host["b"][0]
    want = np.stack(ev_o.Rescale(ev_o.MulRelinNew([a[0], a[1]], [b[0], b[1]])))
    assert want.shape == (2, level, 1 << logN)
    assert np.array_equal(host["out"], want)
