"""The device samplers (csrc/encrypt.cu) bit for bit against the CPU model of tests/sampler_model.py, their distributions
against the reference's (ring/sampler_*.go) by chi-square at about 4M samples, the independence of default-id draws, and
lgpu_small_poly_to_rns at the edges of its range."""
import numpy as np
import pytest
from scipy import stats

from tests import helpers as H
from tests import sampler_model as M

pytestmark = pytest.mark.gpu
Q40, Q60, Q30 = 0x10000140001, 0x1000000000980001, 0x30340001     # first NTT-friendly (1 mod 2^18) primes above 2^40, 2^60, 1.5 * 2^29
SEED_HI = 0x8000000000001234                                       # high bit set
SEED = 20240917


def _samplers(ctx, seed):
    import lattigo_b200 as lb
    return lb.encryptor.Samplers(ctx, seed)


@pytest.mark.parametrize("logN", [4, 8, 12, 16, 17])
def test_uniform_matches_model(logN):
    """Q rows: a prime just above 2^40 (about half the masked words rejected, so three and more attempts occur), one just
    above 2^60, two Qi60 primes and a 30-bit prime; P rows: two more Qi60 primes. Both rings at the maximum and at a lower
    level, batch 1 and 5, a seed with its high bit set and a stream id above 2^32."""
    import lattigo_b200 as lb
    from lattigo_b200.ring import RING_Q, RING_P
    q, p = [Q40, Q60, H.Qi60[0], Q30, H.Qi60[1]], H.Qi60[2:4]
    N = 1 << logN
    ctx = lb.Context(logN, q, p)
    try:
        for ring, level in ((RING_Q, 4), (RING_Q, 1), (RING_P, 1), (RING_P, 0)):
            mods, off = (q, 0) if ring == RING_Q else (p, len(q))
            for seed, sid, batch in ((SEED_HI, (1 << 32) + 3, 5), (SEED, 7, 1)):
                got = ctx.to_host(_samplers(ctx, seed).Uniform(ring, level, batch=batch, stream_id=sid))
                want = M.uniform(seed, sid, mods[: level + 1], range(off, off + level + 1), N, batch)
                assert np.array_equal(got, want), (ring, level, seed, sid, batch)
    finally:
        ctx.close()


def test_uniform_qp_ckks_l44_matches_model():
    """One full UniformQP draw on the benchmarked parameters: 44 Q + 4 P rows, batch 4, N = 2^16, default stream id."""
    import lattigo_b200 as lb
    from lattigo_b200 import params as presets
    s = presets.PRESETS["CKKS_L44"]
    q, p, N = s["Q"], s["P"], 1 << s["logN"]
    ctx = lb.Context(s["logN"], q, p)
    try:
        S = _samplers(ctx, SEED_HI)
        got = ctx.to_host(S.UniformQP(len(q) - 1, len(p) - 1, batch=4))
        want = np.concatenate([M.uniform(SEED_HI, 1, q, range(len(q)), N, 4), M.uniform(SEED_HI, 1, p, range(len(q), len(q) + len(p)), N, 4)], axis=1)
        assert np.array_equal(got, want)
    finally:
        ctx.close()


@pytest.fixture(scope="module")
def ctx16():
    import lattigo_b200 as lb
    ctx = lb.Context(16, [Q40, Q60, H.Qi60[0]], [H.Qi60[1]])
    yield ctx
    ctx.close()


@pytest.mark.parametrize("p", [0.5, 2.0 / 3.0, 2.0 ** -20, 1.0])
def test_ternary_p_matches_model(ctx16, p):
    got = _samplers(ctx16, SEED_HI).Ternary(P=p, batch=4, stream_id=(1 << 32) + 5).cpu().numpy()
    assert np.array_equal(got, M.ternary_p(SEED_HI, (1 << 32) + 5, p, 1 << 16, 4))


@pytest.mark.parametrize("logN", [10, 16])
def test_ternary_h_matches_model(logN):
    """h = N is the longest run of the rejection loop (every position must be hit)."""
    import lattigo_b200 as lb
    N = 1 << logN
    ctx = lb.Context(logN, [Q40])
    try:
        for h in (1, 64, N // 2, N):
            got = _samplers(ctx, SEED).Ternary(H=h, batch=2, stream_id=9).cpu().numpy()
            assert np.array_equal(got, M.ternary_h(SEED, 9, h, N, 2)), h
    finally:
        ctx.close()


def test_gaussian_matches_model_except_flagged(ctx16):
    """Bit-exact except where an attempt's |z| sigma lies within M.gaussian_window of the bound or of a rounding boundary:
    CUDA's log / cospi and the model's need not round those alike. Batch 16 at N = 2^16 per case."""
    flagged = 0
    for sigma, bound in ((3.2, 19.2), (3.2, 6.0), (1.0, 1.0), (2.0 ** 20, 6 * 2.0 ** 20)):
        got = _samplers(ctx16, SEED_HI).Gaussian(sigma, bound, batch=16, stream_id=(1 << 40) + 1).cpu().numpy()
        want, flag = M.gaussian(SEED_HI, (1 << 40) + 1, sigma, bound, 1 << 16, 16)
        assert np.array_equal(got[~flag], want[~flag]), (sigma, bound, int((got != want).sum()))
        flagged += int(flag.sum())
        print("gaussian sigma=%g bound=%g: %d flagged, %d of them differ" % (sigma, bound, flag.sum(), (got != want).sum()))
    assert flagged < 10, flagged


# ---- distributions: against the reference's, not the model's, so that a mistake shared by both is caught ------------------
@pytest.mark.parametrize("sigma,bound", [(3.2, 19.2), (3.2, 6.0)])
def test_gaussian_distribution(ctx16, sigma, bound):
    g = _samplers(ctx16, 101).Gaussian(sigma, bound, batch=M.STAT_BATCH, stream_id=1).cpu().numpy()
    pv = M.gaussian_pvalue(g, sigma, bound)
    print("gaussian sigma=%g bound=%g: p = %.3g" % (sigma, bound, pv))
    assert pv >= M.P_MIN


@pytest.mark.parametrize("row,q", [(0, Q40), (1, Q60)])
def test_uniform_distribution(ctx16, row, q):
    from lattigo_b200.ring import RING_Q
    u = ctx16.to_host(_samplers(ctx16, 102).Uniform(RING_Q, row, batch=M.STAT_BATCH, stream_id=1))[:, row]
    pv = M.uniform_pvalue(u, q)
    print("uniform q=%#x: p = %.3g" % (q, pv))
    assert pv >= M.P_MIN


def test_uniform_distribution_mid_binade():
    """A prime at 1.5 * 2^29, where reducing the masked word mod q instead of rejecting it would show."""
    import lattigo_b200 as lb
    from lattigo_b200.ring import RING_Q
    ctx = lb.Context(16, [Q30])
    try:
        u = ctx.to_host(_samplers(ctx, 103).Uniform(RING_Q, 0, batch=M.STAT_BATCH, stream_id=1))
        pv = M.uniform_pvalue(u, Q30)
        print("uniform q=%#x: p = %.3g" % (Q30, pv))
        assert pv >= M.P_MIN
    finally:
        ctx.close()


def test_ternary_p_distribution(ctx16):
    t = _samplers(ctx16, 104).Ternary(P=2.0 / 3.0, batch=M.STAT_BATCH, stream_id=1).cpu().numpy()
    pv = M.ternary_p_pvalue(t, 2.0 / 3.0)
    print("ternary P=2/3: p = %.3g" % pv)
    assert pv >= M.P_MIN


def test_ternary_h_distribution():
    import lattigo_b200 as lb
    ctx = lb.Context(M.STAT_H_N.bit_length() - 1, [Q40])
    try:
        t = _samplers(ctx, 105).Ternary(H=M.STAT_H, batch=M.STAT_H_BATCH, stream_id=1).cpu().numpy()
        pos, sgn = M.ternary_h_pvalues(t, M.STAT_H)
        print("ternary H=%d: positions p = %.3g, signs p = %.3g" % (M.STAT_H, pos, sgn))
        assert pos >= M.P_MIN and sgn >= M.P_MIN
    finally:
        ctx.close()


# ---- stream properties ---------------------------------------------------------------------------------------------------
def test_default_ids_give_independent_draws():
    """a = UniformQP(L, 0); e = Gaussian() with default stream ids: |e| must not depend on a. Spearman correlation between |e|
    and the top 32 bits of a's row 0 (a Qi60 prime, so the masked word keeps all of x); null sd about 1 / sqrt(N) = 0.004."""
    import lattigo_b200 as lb
    ctx = lb.Context(16, H.Qi60[:3], H.Qi60[3:4])
    try:
        S = _samplers(ctx, 77)
        a = ctx.to_host(S.UniformQP(2, 0, batch=1))
        e = S.Gaussian(batch=1).cpu().numpy()
        rho = stats.spearmanr(np.abs(e[0]), (a[0, 0] >> np.uint64(29)).astype(np.int64)).statistic
        print("spearman(|e|, a[0] >> 29) = %.4f" % rho)
        assert abs(rho) < 0.02, rho
    finally:
        ctx.close()


def test_uniform_rows_do_not_depend_on_level(ctx16):
    """A row is keyed by its limb: the rows of a lower-level draw are the leading rows of a maximum-level draw; the P row is
    not a copy of any Q row's stream."""
    from lattigo_b200.ring import RING_Q, RING_P
    S = _samplers(ctx16, 106)
    full = ctx16.to_host(S.Uniform(RING_Q, 2, batch=3, stream_id=4))
    for level in (0, 1):
        assert np.array_equal(ctx16.to_host(S.Uniform(RING_Q, level, batch=3, stream_id=4)), full[:, : level + 1])
    pr = ctx16.to_host(S.Uniform(RING_P, 0, batch=3, stream_id=4))
    assert np.array_equal(pr, M.uniform(106, 4, [H.Qi60[1]], [3], 1 << 16, 3))


def test_small_poly_to_rns_edges():
    """0, +-1 and +-(floor(q0/2) - 1) on every Q and P row against Python integers; q0 is the smallest modulus, as the
    kernel (like ExtendBasisSmallNormAndCenter) needs |v| < q_i on every row."""
    import torch
    import lattigo_b200 as lb
    q, p = [Q30, Q40, Q60, H.Qi60[0]], H.Qi60[1:3]
    logN = 6
    N = 1 << logN
    ctx = lb.Context(logN, q, p)
    try:
        big = q[0] // 2 - 1
        vals = np.array([0, 1, -1, big, -big], dtype=np.int64)
        small = np.tile(vals, (2, N // len(vals) + 1))[:, :N].copy()
        small[1] = small[1, ::-1]
        rq, rp = lb.encryptor.small_poly_to_rns(ctx, torch.from_numpy(small).cuda(), len(q) - 1, len(p) - 1)
        for rows, mods in ((ctx.to_host(rq), q), (ctx.to_host(rp), p)):
            for b in range(2):
                for i, m in enumerate(mods):
                    assert [int(x) for x in rows[b, i]] == [int(v) % m for v in small[b]], (b, m)
    finally:
        ctx.close()
