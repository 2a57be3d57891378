"""FP64 sequences of the merged ModDown + Rescale tail (keyswitch_fused.cu: ks_ext_split<NSMAX, true>, bcast_lt2q, the RS epilogue) on
worst-case operands, modelled as in test_fp64_arith_model_cpu.py: the broadcast term below 2q enters the last reduction of the 23-bit-halves
extension, whose sum must stay an exact integer below 2^52 and whose result must keep the (-0.66q, 0.66q) range the FP64 butterflies assume."""
import random

import pytest

from tests.test_fp64_arith_model_cpu import TWO52, fma, fp_canon, fp_mulmod, fp_reduce, primes_near_limit


def ks_ext_split_bc(ys, cs, vt, half, bc, q):
    fq, fqinv = float(q), 1.0 / float(q)
    w = float(fp_canon(8388608.0, fq, fqinv))
    A = B = 0
    for y, c in zip(ys, cs):
        d = fp_canon(fp_mulmod(float(c), w, fq, fqinv), fq, fqinv)
        y0, y1, c0, c1, d0, d1 = y & 0x7FFFFF, y >> 23, c & 0x7FFFFF, c >> 23, d & 0x7FFFFF, d >> 23
        A += y0 * c0 + y1 * d0
        B += y0 * c1 + y1 * d1
    assert A < (1 << 51) and B < (1 << 52)
    ab, bb = TWO52 + float(A), TWO52 + float(B)
    vtb = (float(vt) - float(half)) - TWO52
    t = fp_reduce(fma(bb, 8388608.0, -37778931862957161709568.0), fq, fqinv)
    s = ((ab + vtb) + t) + float(bc)
    assert s == int(s) and abs(s) < TWO52                                  # exact: the broadcast term costs no precision
    return fp_reduce(s, fq, fqinv)


def bcast_lt2q(c, qL, s0, q):
    e = (c + ((qL - 1) >> 1)) % qL + s0
    return e % q if qL > q else e


@pytest.mark.parametrize("logN", [13, 16])
def test_merged_prologue_split_extension(logN):
    rng = random.Random(5)
    for q in primes_near_limit(logN):
        srcq = primes_near_limit(logN)[:3] * 2
        for qL in (q, q - 2, (1 << 45) + 59, (1 << 61) - 1):               # last modulus equal, below, far below and far above the row
            s0 = q - (((qL - 1) >> 1) % q)
            for c in (qL - 1, 0, (qL - 1) >> 1, rng.randrange(qL)):
                bc = bcast_lt2q(c, qL, s0, q)
                assert 0 <= bc < 2 * q
                cases = [([s - 1 for s in srcq], [q - 1] * 6)] + [([rng.randrange(s) for s in srcq], [rng.randrange(q) for _ in srcq]) for _ in range(20)]
                for ys, cs in cases:
                    for vt, half in ((q - 1, 0), (0, (q - 1) // 2)):
                        r = ks_ext_split_bc(ys, cs, vt, half, bc, q)
                        assert r == int(r) and abs(r) <= 0.66 * q, (q, r)
                        want = sum(y * cc for y, cc in zip(ys, cs)) + vt - half + (c + ((qL - 1) >> 1)) % qL - ((qL - 1) >> 1)
                        assert (int(r) - want) % q == 0


@pytest.mark.parametrize("logN", [13, 16])
def test_merged_epilogue_operand_ranges(logN):
    """RS epilogue: x is the biased integer of a lazy transform output (< 2^52 on the FP64 rows, < kq <= 2^63 on the integer rows); x + 2q - d
    stays below 2^64 and both Montgomery products have a factor below q, so each MRed is canonical and their sum is below 2q."""
    for q in primes_near_limit(logN) + [(1 << 61) - 1]:
        for x in (0, (1 << 52) - 1, (1 << 63) - 1):
            for d in (0, q - 1):
                assert x + 2 * q - d < 1 << 64
                assert (x + 2 * q - d) * (q - 1) < q << 64                # MRed input range: hi < q
        assert 2 * (q - 1) < 1 << 64
