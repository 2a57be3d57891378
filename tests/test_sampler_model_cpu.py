"""CPU side of the device samplers (csrc/encrypt.cu): the Philox4x32-10 restatement of tests/sampler_model.py against
Random123's known-answer vectors, the separation of the random streams (no two sampler calls, kinds or rings ever read the
same Philox block), the stream ids the Python wrapper hands out, and the power of the statistical checks that
tests/test_gpu_samplers.py applies to the device output: at the GPU sample sizes they accept the model and reject
deliberately wrong samplers."""
import itertools

import numpy as np
import pytest

from tests import helpers as H
from tests import sampler_model as M

Q40, Q60, Q30 = 0x10000140001, 0x1000000000980001, 0x30340001     # first NTT-friendly (1 mod 2^18) primes above 2^40, 2^60, 1.5 * 2^29
SEED = 0x8000000000001234


def test_philox_known_answers():
    """Random123's kat_vectors for philox4x32_10: zero counter / key and all-ones counter / key."""
    got = [int(v) for v in M.philox4x32_10(0, 0, 0, 0, 0, 0)]
    assert got == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    f = 0xFFFFFFFF
    got = [int(v) for v in M.philox4x32_10(f, f, f, f, f, f)]
    assert got == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


def _calls(stream, N=64, batch=3):
    """The block sets of one stream id: uniform over 5 Q rows and 2 P rows, ternary P, ternary H, Gaussian."""
    q, p = [Q40, Q60, Q30] + H.Qi60[:2], H.Pi60[:2]
    out = {}
    for name, fn in (("uniform Q", lambda b: M.uniform(SEED, stream, q, range(5), N, batch, b)),
                     ("uniform P", lambda b: M.uniform(SEED, stream, p, range(5, 7), N, batch, b)),
                     ("ternary P", lambda b: M.ternary_p(SEED, stream, 0.5, N, batch, b)),
                     ("ternary H", lambda b: M.ternary_h(SEED, stream, N // 2, N, batch, b)),
                     ("gaussian", lambda b: M.gaussian(SEED, stream, 3.2, 19.2, N, batch, b))):
        blocks = []
        fn(blocks)
        out[(stream, name)] = M.block_set(blocks)
    return out


def test_sampler_kinds_and_rings_read_disjoint_blocks():
    """For one (seed, stream id), every sampler kind and the Q and P rows of a uniform draw read their own Philox blocks;
    so do two stream ids that agree in their low 32 bits."""
    sets = {}
    for stream in (7, (1 << 32) + 7, (1 << 63) | 7):
        sets.update(_calls(stream))
    assert all(len(s) > 0 for s in sets.values())
    for (a, sa), (b, sb) in itertools.combinations(sets.items(), 2):
        assert len(sa & sb) == 0, "%r and %r share Philox blocks" % (a, b)


class _Recorder:
    """Stands in for the CUDA library: records the sampler calls of lattigo_b200.encryptor.Samplers."""

    def __init__(self):
        self.calls = []

    def lgpu_sample_uniform(self, h, ring, level, seed, sid, out, batch, bs, stream):
        self.calls.append(("uniform", ring, level, seed, sid, batch))
        return 0

    def lgpu_sample_ternary(self, h, p, hw, seed, sid, out, batch, stream):
        self.calls.append(("ternary", p, hw, seed, sid, batch))
        return 0

    def lgpu_sample_gaussian(self, h, sigma, bound, seed, sid, out, batch, stream):
        self.calls.append(("gaussian", sigma, bound, seed, sid, batch))
        return 0


class _HostContext:
    def __init__(self, N, Q, P):
        self.h, self.N, self.Q, self.P, self.device = None, N, Q, P, -1

    def new_poly(self, limbs, batch=None):
        import torch
        return torch.zeros((limbs, self.N) if batch is None else (batch, limbs, self.N), dtype=torch.int64)


def test_wrapper_default_stream_ids_never_share_blocks(monkeypatch):
    """Samplers hands out one stream id per call from a single counter -- UniformQP included, for both of its rings -- so
    `a = UniformQP(...); e = Gaussian(...)` cannot draw the error from the blocks of the public `a`."""
    import ctypes
    import lattigo_b200 as lb
    from lattigo_b200 import _lib, encryptor
    rec = _Recorder()
    monkeypatch.setattr(_lib, "lib", lambda: rec)
    monkeypatch.setattr(encryptor, "_dptr", lambda t: ctypes.c_void_p(t.data_ptr()))
    monkeypatch.setattr(encryptor, "_stream", lambda: None)
    N, Q, P = 64, [Q40, Q60, Q30], H.Pi60[:2]
    S = lb.encryptor.Samplers(_HostContext(N, Q, P), seed=SEED)
    a = S.UniformQP(2, 1, batch=2)
    S.Gaussian(batch=2)
    S.Ternary(P=2.0 / 3.0)
    S.Ternary(H=N // 4, batch=2)
    S.Uniform(encryptor.RING_Q, 1, batch=3)
    S.Uniform(encryptor.RING_P, 0)
    assert tuple(a.shape) == (2, 5, N)
    assert [c[4] for c in rec.calls] == [1, 1, 2, 3, 4, 5, 6]          # UniformQP: one id for both rings
    assert [c[1] for c in rec.calls[:2]] == [encryptor.RING_Q, encryptor.RING_P]
    sets = []
    for c in rec.calls:
        blocks = []
        if c[0] == "uniform":
            _, ring, level, seed, sid, batch = c
            mods, off = (Q, 0) if ring == encryptor.RING_Q else (P, len(Q))
            M.uniform(seed, sid, mods[: level + 1], range(off, off + level + 1), N, batch, blocks)
        elif c[0] == "ternary":
            _, p, hw, seed, sid, batch = c
            (M.ternary_h(seed, sid, hw, N, batch, blocks) if hw else M.ternary_p(seed, sid, p, N, batch, blocks))
        else:
            _, sigma, bound, seed, sid, batch = c
            M.gaussian(seed, sid, sigma, bound, N, batch, blocks)
        sets.append(M.block_set(blocks))
    for (i, si), (j, sj) in itertools.combinations(enumerate(sets), 2):
        assert len(si & sj) == 0, "calls %r and %r share Philox blocks" % (rec.calls[i], rec.calls[j])


# ---- the statistical checks of tests/test_gpu_samplers.py have power at its sample sizes ---------------------------------
N, B = M.STAT_N, M.STAT_BATCH


@pytest.mark.parametrize("sigma,bound,variant", [(3.2, 19.2, "floor"), (3.2, 6.0, "round_then_bound")])
def test_gaussian_check_rejects_wrong_samplers(sigma, bound, variant):
    good, _ = M.gaussian(SEED, 11, sigma, bound, N, B)
    bad, _ = M.gaussian(SEED, 11, sigma, bound, N, B, variant=variant)
    assert M.gaussian_pvalue(good, sigma, bound) >= M.P_MIN
    assert M.gaussian_pvalue(bad, sigma, bound) < M.P_MIN


def test_uniform_check_rejects_reduction_mod_q():
    """v mod q in place of rejection. Just above a power of two (Q40, Q60) it differs from rejection only on a 2 (q - 2^k) / q
    sliver, which no sample size can see; a prime in the middle of its binade (Q30 = 1.51 * 2^29) makes a third of [0, q)
    twice as likely."""
    assert M.uniform_pvalue(M.uniform(SEED, 12, [Q30], [0], N, B), Q30) >= M.P_MIN
    assert M.uniform_pvalue(M.uniform(SEED, 12, [Q30], [0], N, B, variant="mod"), Q30) < M.P_MIN


def test_ternary_p_check_rejects_p_read_per_sign():
    good = M.ternary_p(SEED, 13, 2.0 / 3.0, N, B)
    bad = M.ternary_p(SEED, 13, 2.0 / 3.0, N, B, variant="half")
    assert M.ternary_p_pvalue(good, 2.0 / 3.0) >= M.P_MIN
    assert M.ternary_p_pvalue(bad, 2.0 / 3.0) < M.P_MIN


def test_ternary_h_check_rejects_positions_from_half_the_ring():
    good = M.ternary_h(SEED, 14, M.STAT_H, M.STAT_H_N, M.STAT_H_BATCH)
    bad = M.ternary_h(SEED, 14, M.STAT_H, M.STAT_H_N, M.STAT_H_BATCH, variant="half")
    assert min(M.ternary_h_pvalues(good, M.STAT_H)) >= M.P_MIN
    assert M.ternary_h_pvalues(bad, M.STAT_H)[0] < M.P_MIN
