"""Bit-exact CPU model of the device samplers in lattigo_b200/csrc/encrypt.cu (lgpu_sample_uniform / _ternary / _gaussian),
and the statistical checks the GPU tests apply to their output.

This restates the KERNELS, not the reference: the reference draws from a blake2b byte stream (sampling/prng.go) that the
device does not reproduce. Every sampler reads Philox4x32-10 blocks keyed by make_key(seed, stream id) at the counter

    {x, y, z, w} = {coefficient or draw index, kind << 30 | polynomial, low 32 bits of the stream id, attempt}

with kind 0 = uniform (polynomial = batch * 128 + global limb index), 1 = ternary P, 2 = ternary H, 3 = Gaussian (polynomial =
batch index). Every sampler takes `blocks`: when it is a list, the (k0, k1, x, y, z, w) blocks the call consumes are appended
to it, one uint32 array of shape (n, 6) per pass, so tests can assert that two calls never share a block.

Each sampler also takes `variant`: None is the kernel; the named variants are deliberately wrong restatements, used only to
show that the statistical checks at the end of this file reject a subtly wrong sampler."""
import numpy as np
from scipy import special, stats

U64 = np.uint64
M32 = U64(0xFFFFFFFF)
KIND_UNIFORM, KIND_TERNARY_P, KIND_TERNARY_H, KIND_GAUSSIAN = 0, 1, 2, 3
MAX_ROWS = 128                      # kMaxRows (csrc/engine.h): uniform polynomial index = batch * 128 + limb


# ---- Philox4x32-10 (Salmon et al., SC'11), as philox4x32_10 in encrypt.cu ---------------------------------------------------
def philox4x32_10(x, y, z, w, k0, k1):
    """Vectorized over the counter words (uint64 arrays holding 32-bit values); returns the four output words."""
    c = np.broadcast_arrays(*(np.asarray(v, dtype=U64) for v in (x, y, z, w)))
    shape = c[0].shape
    c = [v.ravel() for v in c]
    out = [np.empty(c[0].size, dtype=U64) for _ in range(4)]
    step = 1 << 15                  # cache-sized chunks: about 3x faster than whole arrays
    for s in range(0, c[0].size, step):
        x, y, z, w = (v[s:s + step] for v in c)
        k0_, k1_ = U64(k0), U64(k1)
        for _ in range(10):
            p0 = U64(0xD2511F53) * x
            p1 = U64(0xCD9E8D57) * z
            x, y, z, w = (p1 >> U64(32)) ^ y ^ k0_, p1 & M32, (p0 >> U64(32)) ^ w ^ k1_, p0 & M32
            k0_ = (k0_ + U64(0x9E3779B9)) & M32
            k1_ = (k1_ + U64(0xBB67AE85)) & M32
        for o, v in zip(out, (x, y, z, w)):
            o[s:s + step] = v
    return tuple(o.reshape(shape) for o in out)


def make_key(seed: int, stream: int):
    """(k0, k1, counter word z) of make_key in encrypt.cu: the high half of the stream id is folded into k1 by an odd
    multiplier, so for one seed every 64-bit stream id has its own (k1, z)."""
    seed &= (1 << 64) - 1
    stream &= (1 << 64) - 1
    k0 = seed & 0xFFFFFFFF
    k1 = (seed >> 32) ^ (((stream >> 32) * 0x85EBCA6B) & 0xFFFFFFFF)
    return k0, k1, stream & 0xFFFFFFFF


def _draw(key, kind, poly, coeff, attempt, blocks):
    k0, k1, s = key
    coeff = np.asarray(coeff, dtype=U64)
    y = (U64(kind << 30) | np.asarray(poly, dtype=U64)) + np.zeros_like(coeff)
    z = np.full_like(coeff, s)
    w = np.asarray(attempt, dtype=U64) + np.zeros_like(coeff)
    if blocks is not None:
        blocks.append(np.stack([np.full_like(coeff, k0), np.full_like(coeff, k1), coeff, y, z, w], axis=-1).reshape(-1, 6).astype(np.uint32))
    return philox4x32_10(coeff, y, z, w, k0, k1)


def block_set(blocks):
    """The consumed blocks of one or more calls as a set of 24-byte keys."""
    a = np.concatenate(blocks) if blocks else np.zeros((0, 6), np.uint32)
    return set(np.ascontiguousarray(a).view("V24").ravel().tolist())


# ---- samplers ----------------------------------------------------------------------------------------------------------
def uniform(seed, stream, moduli, limbs, N, batch, blocks=None, variant=None):
    """lgpu_sample_uniform: out[b, r, i] uniform in [0, moduli[r]); row r is keyed by its global limb index limbs[r] (Q limbs
    first, then P limbs), so a row's values do not depend on the level it is drawn at. Each attempt masks x||y, then z||w, to
    the bit length of q - 1 and rejects values >= q. variant "mod": the first masked word reduced mod q (biased)."""
    key = make_key(seed, stream)
    q = np.array([int(m) for m in moduli], dtype=U64)[:, None]
    mask = np.array([(1 << (int(m) - 1).bit_length()) - 1 for m in moduli], dtype=U64)[:, None]
    coeff = np.broadcast_to(np.arange(N, dtype=U64), (len(moduli), N)).ravel()
    out = np.empty((batch, len(moduli), N), dtype=U64)
    for b in range(batch):
        poly = (U64(b * MAX_ROWS) + np.array(limbs, dtype=U64)[:, None] + np.zeros((1, N), U64)).ravel()
        qq = np.broadcast_to(q, (len(moduli), N)).ravel()
        mm = np.broadcast_to(mask, (len(moduli), N)).ravel()
        v = np.zeros(len(coeff), dtype=U64)
        todo = np.arange(len(coeff))
        a = 0
        while len(todo):
            x, y, z, w = _draw(key, KIND_UNIFORM, poly[todo], coeff[todo], a, blocks)
            v1 = ((x << U64(32)) | y) & mm[todo]
            if variant == "mod":
                v[todo] = v1 % qq[todo]
                break
            v2 = ((z << U64(32)) | w) & mm[todo]
            ok1, ok2 = v1 < qq[todo], v2 < qq[todo]
            v[todo] = np.where(ok1, v1, v2)
            todo = todo[~(ok1 | ok2)]
            a += 1
        out[b] = v.reshape(len(moduli), N)
    return out


def ternary_p(seed, stream, p, N, batch, blocks=None, variant=None):
    """lgpu_sample_ternary with hamming_weight = 0: non-zero when u = (x 2^32 + y) 2^-64 < p (the float64 arithmetic of the
    kernel, so the comparison is bit-identical), sign +1 when z is odd. variant "half": non-zero only when u < p / 2."""
    key = make_key(seed, stream)
    coeff = np.broadcast_to(np.arange(N, dtype=U64), (batch, N))
    poly = np.arange(batch, dtype=U64)[:, None]
    x, y, z, _ = _draw(key, KIND_TERNARY_P, poly, coeff, 0, blocks)
    u = (x.astype(np.float64) * 4294967296.0 + y.astype(np.float64)) * (1.0 / 18446744073709551616.0)
    thr = p / 2 if variant == "half" else p
    return np.where(u < thr, np.where(z & U64(1), 1, -1), 0).astype(np.int64)


def ternary_h(seed, stream, h, N, batch, blocks=None, variant=None):
    """lgpu_sample_ternary with hamming_weight = h: thread 0 of the polynomial's CTA takes draws a = 0, 1, ...; candidates
    x & (N-1) then z & (N-1) with signs y & 1, w & 1 (1 -> +1); a position already taken is skipped; it stops at h placed.
    Vectorized: the first occurrences of positions in draw order, first h of them. variant "half": positions x & (N/2-1)."""
    key = make_key(seed, stream)
    pos_mask = U64(N // 2 - 1 if variant == "half" else N - 1)
    out = np.zeros((batch, N), dtype=np.int64)
    A = max(16, int(h * 1.3) // 2 + 8)
    while True:
        a = np.broadcast_to(np.arange(A, dtype=U64), (batch, A))
        x, y, z, w = _draw(key, KIND_TERNARY_H, np.arange(batch, dtype=U64)[:, None], a, 0, None)
        cand = np.stack([x & pos_mask, z & pos_mask], axis=-1).reshape(batch, 2 * A).astype(np.int64)
        sign = np.stack([y & U64(1), w & U64(1)], axis=-1).reshape(batch, 2 * A)
        flat = cand + (np.arange(batch, dtype=np.int64) * N)[:, None]
        _, first = np.unique(flat.ravel().astype(np.int32 if batch * N < 1 << 31 else np.int64), return_index=True)
        is_first = np.zeros(batch * 2 * A, dtype=bool)
        is_first[first] = True
        is_first = is_first.reshape(batch, 2 * A)
        rank = np.cumsum(is_first, axis=1)
        if (rank[:, -1] >= h).all():
            break
        A *= 2
    take = is_first & (rank <= h)
    rows, cols = np.nonzero(take)
    out[rows, cand[rows, cols]] = np.where(sign[rows, cols] == 1, 1, -1)
    if blocks is not None:          # draws 0 .. last used, per polynomial
        last = np.argmax(rank >= h, axis=1) // 2
        for b in range(batch):
            _draw(key, KIND_TERNARY_H, b, np.arange(last[b] + 1, dtype=U64), 0, blocks)
    return out


def _abs_cospi(t):
    """|cos(pi t)| for t in [0, 2) to a few ulp: exact reductions to [0, 1/2], then cos or sin of an argument <= pi / 4."""
    t = np.where(t > 1.0, 2.0 - t, t)
    t = np.where(t > 0.5, 1.0 - t, t)
    return np.where(t <= 0.25, np.cos(np.pi * t), np.sin(np.pi * (0.5 - t)))


def gaussian_window(m):
    """Half-width of the band around a rounding or acceptance boundary inside which the device's m = |z| sigma may fall on
    the other side from the model's: neither CUDA's log and cospi nor numpy's are correctly rounded (a few ulp of m each). 1e-9 absolute, widened
    in proportion to m where 1e-9 is below the float64 resolution of m (ulp(2^22) ~ 1e-9)."""
    return 1e-9 + m * 2.0 ** -44


def gaussian(seed, stream, sigma, bound, N, batch, blocks=None, variant=None):
    """lgpu_sample_gaussian: Box-Muller on u1 = ((x<<21 | y>>11) + 1) 2^-53 in (0, 1], u2 = (z<<21 | w>>11) 2^-53 in [0, 1),
    m = |sqrt(-2 log u1) cospi(2 u2)| sigma, redrawn (attempt + 1) while m > bound, output (long long)(m + 0.5) with sign
    bit w & 1 (1 -> negative). Returns (values, flagged): flagged marks coefficients where some
    attempt's m lies within gaussian_window(m) of the bound or of a rounding boundary k + 1/2; only those may differ from the
    device. variant "floor": output floor(m); "round_then_bound": accept when the rounded value is <= bound."""
    key = make_key(seed, stream)
    coeff = np.broadcast_to(np.arange(N, dtype=U64), (batch, N)).ravel()
    poly = np.broadcast_to(np.arange(batch, dtype=U64)[:, None], (batch, N)).ravel()
    out = np.zeros(batch * N, dtype=np.int64)
    flagged = np.zeros(batch * N, dtype=bool)
    todo = np.arange(batch * N)
    a = 0
    while len(todo):
        x, y, z, w = _draw(key, KIND_GAUSSIAN, poly[todo], coeff[todo], a, blocks)
        u1 = (((x << U64(21)) | (y >> U64(11))) + U64(1)).astype(np.float64) * 2.0 ** -53
        u2 = ((z << U64(21)) | (w >> U64(11))).astype(np.float64) * 2.0 ** -53
        m = np.sqrt(-2.0 * np.log(u1)) * _abs_cospi(2.0 * u2) * sigma
        tol = gaussian_window(m)
        near_half = np.abs(m - (np.floor(m) + 0.5)) <= tol
        near_bound = np.abs(m - bound) <= tol
        r = np.floor(m) if variant == "floor" else np.floor(m + 0.5)
        ok = (r <= bound) if variant == "round_then_bound" else (m <= bound)
        flagged[todo] |= near_bound | (ok & near_half)
        v = np.where(w & U64(1), -r, r).astype(np.int64)
        out[todo[ok]] = v[ok]
        todo = todo[~ok]
        a += 1
    return out.reshape(batch, N), flagged.reshape(batch, N)


# ---- statistical checks against the reference's distributions ------------------------------------------------------------
# The GPU tests draw these many samples per case, and the CPU tests show at the same sizes that each check rejects a
# deliberately wrong sampler. All draws use fixed seeds, so every p-value is deterministic.
STAT_N = 1 << 16
STAT_BATCH = 64                     # 4M samples: Gaussian, uniform, ternary P
STAT_H_N, STAT_H, STAT_H_BATCH = 1 << 12, 1024, 4096     # 4M non-zero positions of ternary H
P_MIN = 1e-6


def chisquare_merged(observed, expected, min_expected=20.0):
    """p-value of scipy.stats.chisquare after merging adjacent cells until each expects >= min_expected samples."""
    observed = np.asarray(observed, dtype=np.float64)
    expected = np.asarray(expected, dtype=np.float64)
    obs, exp, o, e = [], [], 0.0, 0.0
    for oi, ei in zip(observed, expected):
        o += oi; e += ei
        if e >= min_expected:
            obs.append(o); exp.append(e); o = e = 0.0
    if e > 0 or o > 0:
        if exp:
            obs[-1] += o; exp[-1] += e
        else:
            obs.append(o); exp.append(e)
    exp = np.array(exp); obs = np.array(obs)
    exp *= obs.sum() / exp.sum()        # chisquare wants equal totals; the pmf sums to 1 only up to rounding
    return float(stats.chisquare(obs, exp).pvalue)


def gaussian_pmf(sigma, bound):
    """ring/sampler_gaussian.go:160-182 (bound < 2^53 branch): m = |N(0,1)| sigma, kept when m <= bound, magnitude
    floor(m + 1/2) with a fair sign. Values -K..K with K = floor(bound + 1/2)."""
    K = int(np.floor(bound + 0.5))
    k = np.arange(K + 1, dtype=np.float64)
    lo = np.maximum(k - 0.5, 0.0)
    hi = np.minimum(k + 0.5, bound)
    w = np.where(lo <= bound, special.ndtr(hi / sigma) - special.ndtr(lo / sigma), 0.0)
    w /= special.ndtr(bound / sigma) - 0.5
    pmf = np.concatenate([w[:0:-1] / 2, w[:1], w[1:] / 2])
    return np.arange(-K, K + 1), pmf


def gaussian_pvalue(values, sigma, bound):
    support, pmf = gaussian_pmf(sigma, bound)
    v = np.asarray(values).ravel()
    if np.abs(v).max() > support[-1]:
        return 0.0
    counts = np.bincount(v - support[0], minlength=len(support))
    return chisquare_merged(counts, pmf * len(v))


def uniform_pvalue(values, q, bins=256):
    """256 equal bins over [0, q): bin j = [floor(j q / 256), floor((j+1) q / 256))."""
    v = np.asarray(values, dtype=U64).ravel()
    if int(v.max()) >= q:
        return 0.0
    edges = np.array([j * q // bins for j in range(bins + 1)], dtype=U64)
    counts = np.bincount(np.searchsorted(edges, v, side="right") - 1, minlength=bins)
    widths = np.diff(np.array([j * q // bins for j in range(bins + 1)], dtype=object)).astype(np.float64)
    return chisquare_merged(counts, widths / q * len(v))


def ternary_p_pvalue(values, p):
    v = np.asarray(values).ravel()
    if not np.isin(v, (-1, 0, 1)).all():
        return 0.0
    counts = [(v == -1).sum(), (v == 0).sum(), (v == 1).sum()]
    return chisquare_merged(counts, np.array([p / 2, 1 - p, p / 2]) * len(v))


def ternary_h_pvalues(values, h, bins=64):
    """(positions, signs): how often each of 64 equal position bins is non-zero (uniform positions; sampling without
    replacement within a polynomial only makes the statistic smaller), and the balance of +1 against -1."""
    v = np.asarray(values)
    nz = v != 0
    if np.abs(v).max() > 1 or (nz.sum(axis=1) != h).any():
        return 0.0, 0.0
    per_bin = nz.sum(axis=0).reshape(bins, -1).sum(axis=1)
    pos = chisquare_merged(per_bin, np.full(bins, per_bin.sum() / bins))
    plus = int((v == 1).sum())
    sgn = chisquare_merged([plus, nz.sum() - plus], [nz.sum() / 2] * 2)
    return pos, sgn
