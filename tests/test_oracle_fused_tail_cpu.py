"""The merged ModDown + Rescale tail of the fused MulRelinRescale (keyswitch_fused.cu: moddown_ntt_fused with rescale = 1), restated on the
oracle: for every output row j < L
    out_j = (acc_j P^-1 + d_j - NTT(P^-1 E_j + ext_L,j)) q_L^-1   (mod q_j),
E_j = ModUpPtoQ(INTT(acc_P)) row j, ext_L,j = (c_L + floor(q_L/2)) mod q_L - floor(q_L/2) mod q_j, c_L = INTT(ModDown output row L),
must equal the oracle's ModDownQPtoQNTT -> add d -> DivRoundByLastModulusNTT word for word. Also checked: the extension evaluated with the
constants pre-multiplied by P^-1 (Ctx::muc_PtoQ_pinv) is P^-1 E_j, and the epilogue's Montgomery constants (RescaleConstants and
MForm(P^-1 q_L^-1) derived from the ModDown and Rescale constants) give the formula above. Small rings, 1..6 P limbs, and a 60-bit last
modulus above 40-bit rows."""
import numpy as np
import pytest

from oracle import oracle as O
from tests import helpers as H

U64 = np.uint64
R64 = 1 << 64


def _mred(x, y, q):
    return x * y * pow(R64, -1, q) % q


def _intt_row(ring, level, row):
    out = np.empty_like(row)
    ring.SubRings[level].INTT(np.ascontiguousarray(row), out)
    return out


def _ntt_row(ring, j, row):
    out = np.empty_like(row)
    ring.SubRings[j].NTT(np.ascontiguousarray(row), out)
    return out


def _ext_scaled(x_p, P, q):
    """basis extension P -> q of the centred P-residues x_p (as ModUpPtoQ: + floor(P/2), extend, - floor(P/2)) with every target constant
    multiplied by P^-1 mod q: sum_i y_i (S/s_i mod q) P^-1 - v S P^-1 - floor(S/2) P^-1, y_i = (x_i + floor(S/2)) (S/s_i)^-1 mod s_i"""
    S = 1
    for s in P:
        S *= s
    pinv = pow(S % q, -1, q)
    c = [(S // s) % q * pinv % q for s in P]
    vt = (q - S % q) * pinv % q
    half_t = (S >> 1) % q * pinv % q
    out = []
    for k in range(len(x_p[0])):
        ys = [(int(x_p[i][k]) + (S >> 1)) * pow((S // s) % s, -1, s) % s for i, s in enumerate(P)]
        v = sum(y * (S // s) for y, s in zip(ys, P)) // S      # floor(sum y_i / s_i): the overflow count
        out.append((sum(y * ci for y, ci in zip(ys, c)) + v * vt - half_t) % q)
    return out


@pytest.mark.parametrize("logN,logQ,logP", [
    (4, [45, 40, 40, 40], [50]),
    (6, [55, 40, 40, 40, 40], [61, 61]),
    (7, [45, 35, 35, 35, 35, 35], [50, 50, 50]),
    (8, [50, 40, 40, 40, 60], [61, 61, 61, 61]),          # 60-bit last modulus above 40-bit rows
    (9, [60, 40, 40, 60], [61, 61, 61, 61, 61]),
    (10, [55, 40, 40, 40, 40], [50, 50, 50, 50, 50, 50]),
])
def test_merged_tail_equals_moddown_then_rescale(logN, logQ, logP):
    q, p = O.gen_moduli(logN + 1, logQ, logP)
    N = 1 << logN
    ringQ, ringP = O.Ring(N, q), O.Ring(N, p)
    be = O.BasisExtender(ringQ, ringP)
    rng = np.random.default_rng(logN)
    L, levelP = len(q) - 1, len(p) - 1
    accQ, accP, d = H.rand_poly(q, N, rng), H.rand_poly(p, N, rng), H.rand_poly(q, N, rng)
    # oracle: ModDown, + d, Rescale
    md = np.empty_like(accQ)
    be.ModDownQPtoQNTT(L, levelP, accQ.copy(), accP.copy(), md)
    for j, qj in enumerate(q):
        md[j] = ((md[j].astype(object) + d[j].astype(object)) % qj).astype(U64)
    want = np.empty((L, N), dtype=U64)
    ringQ.DivRoundByLastModulusNTT(md, want)
    # merged tail
    P = 1
    for s in p:
        P *= s
    qL = q[L]
    pHalf = (qL - 1) >> 1
    cL = [int(x) for x in _intt_row(ringQ, L, md[L])]
    xP = np.stack([_intt_row(ringP, i, accP[i]) for i in range(len(p))])
    E = np.empty((L + 1, N), dtype=U64)
    be.ModUpPtoQ(levelP, L, xP.copy(), E)
    mdc, resc = be.modDownConstantsPtoQ[levelP], ringQ.RescaleConstants[L - 1]
    for j in range(L):
        qj = q[j]
        pinv, qLinv = pow(P % qj, -1, qj), pow(qL % qj, -1, qj)
        ext = [((c + pHalf) % qL + qj - pHalf % qj) % qj for c in cL]
        scaled = _ext_scaled(xP, p, qj)
        assert scaled == [int(e) * pinv % qj for e in E[j]]
        x = [int(v) for v in _ntt_row(ringQ, j, np.array([(a + b) % qj for a, b in zip(scaled, ext)], dtype=U64))]
        out = [(int(a) * pinv + int(dd) - xx) * qLinv % qj for a, dd, xx in zip(accQ[j], d[j], x)]
        assert out == [int(w) for w in want[j]], j
        # the epilogue's constants: CRed(MRed(x + 2q - d, s) + MRed(a, s2)), s = RescaleConstant, s2 from the ModDown one
        s, s2 = int(resc[j]), _mred(int(mdc[j]), (qj - int(resc[j])) % qj, qj)
        assert s2 == pinv * qLinv * R64 % qj
        dev = [(_mred(xx + 2 * qj - int(dd), s, qj) + _mred(int(a), s2, qj)) % qj for a, dd, xx in zip(accQ[j], d[j], x)]
        assert dev == out
