"""GPU side of SURVEY 8(f) rank 3 (csrc/encrypt.cu): the encryptor / key-generator inner loops bit for bit against
oracle/encryptor.py on the same sampled polynomials, the samplers' stream handling, and an end-to-end check (device-sampled
secret / error / uniform polynomials -> device evaluation key -> key switch -> oracle-side noise measurement)."""
import numpy as np
import pytest

from oracle import encryptor as E
from oracle import oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu
U64 = np.uint64


def _sk_rows(params, s, q, p):
    sk = E.small_rows(s, q + p)
    params.ringQ.NTT(sk[: len(q)], sk[: len(q)]); params.ringQ.MForm(sk[: len(q)], sk[: len(q)])
    if p:
        params.ringP.NTT(sk[len(q):], sk[len(q):]); params.ringP.MForm(sk[len(q):], sk[len(q):])
    return sk


@pytest.mark.parametrize("logN,with_p", [(9, True), (9, False), (13, True)])
def test_encrypt_zero_paths_match_the_oracle(logN, with_p):
    import torch
    import lattigo_b200 as lb
    q, p = O.gen_moduli(logN + 1, [55, 45, 45, 45], [55, 55] if with_p else [])
    params = O.Parameters(logN, q, p)
    N = params.N()
    rng = np.random.default_rng(logN + with_p)
    ctx = lb.Context(logN, q, p)
    try:
        enc_o = E.Encryptor(params); enc = lb.encryptor.Encryptor(ctx)
        s = rng.integers(-1, 2, N)
        sk = _sk_rows(params, s, q, p)
        d_sk = ctx.to_device(sk)
        batch = 3
        gauss = lambda: np.rint(rng.normal(0, 3.2, (batch, N))).astype(np.int64)
        # secret-key encryption of zero: plain (levelP = -1) and over QP, all flag combinations
        for levelQ, levelP in ((3, -1), (1, -1)) + (((3, 1), (2, 0)) if with_p else ()):
            for ntt, mont in ((True, False), (False, False), (True, True)):
                mods = q[: levelQ + 1] + p[: levelP + 1]
                c1 = np.stack([H.rand_poly(mods, N, rng) for _ in range(batch)])
                e = gauss()
                d_c1 = ctx.to_device(c1)
                c0 = enc.EncryptZeroSk(levelQ, levelP, d_sk, d_c1, torch.from_numpy(e).cuda(), ntt, mont)
                for b in range(batch):
                    w1 = c1[b].copy()
                    w0 = enc_o.encryptZeroSkFromC1QP(levelQ, levelP, sk, w1, e[b], ntt, mont)
                    assert np.array_equal(ctx.to_host(c0)[b], w0), (levelQ, levelP, ntt, mont)
                    assert np.array_equal(ctx.to_host(d_c1)[b], w1)
        # public key = encryptZeroSk over QP (NTT + Montgomery), then public-key encryptions of zero
        a = H.rand_poly(q + p, N, rng)
        epk = np.rint(rng.normal(0, 3.2, N)).astype(np.int64)
        pk1 = a.copy()
        pk0 = enc_o.encryptZeroSkFromC1QP(len(q) - 1, len(p) - 1, sk, pk1, epk, True, True)
        pk = np.stack([pk0, pk1])
        d_pk = ctx.to_device(pk)
        for levelQ in (3, 2):
            for ntt, mont in ((True, False), (False, False)) + (((True, True),) if with_p else ()):
                u = rng.integers(-1, 2, (batch, N)); e0 = gauss(); e1 = gauss()
                ct = enc.EncryptZeroPk(levelQ, d_pk, torch.from_numpy(u).cuda(), torch.from_numpy(e0).cuda(), torch.from_numpy(e1).cuda(), ntt, mont)
                for b in range(batch):
                    w = enc_o.encryptZeroPk(levelQ, pk, u[b], e0[b], e1[b], ntt, mont) if with_p else enc_o.encryptZeroPkNoP(levelQ, pk, u[b], e0[b], e1[b], ntt)
                    assert np.array_equal(ctx.to_host(ct)[b, 0], w[0]) and np.array_equal(ctx.to_host(ct)[b, 1], w[1]), (levelQ, ntt, mont)
    finally:
        ctx.close()


@pytest.mark.parametrize("pw2,lp", [(0, [55, 55]), (0, [55, 55, 55]), (13, [55]), (11, [])])
def test_gen_evaluation_key_matches_the_oracle(pw2, lp):
    import torch
    import lattigo_b200 as lb
    logN = 9
    q, p = O.gen_moduli(logN + 1, [55, 45, 45, 45, 45], lp)
    params = O.Parameters(logN, q, p)
    N = params.N()
    rng = np.random.default_rng(pw2 + len(lp))
    levelQ, levelP = len(q) - 1, len(p) - 1
    n = params.BaseRNSDecompositionVectorSize(levelQ, levelP)
    sizes = params.BaseTwoDecompositionVectorSize(levelQ, levelP, pw2)[:n]
    s_in = rng.integers(-1, 2, N); s_out = rng.integers(-1, 2, N)
    sk_out = _sk_rows(params, s_out, q, p); sk_in = _sk_rows(params, s_in, q, [])
    a = np.stack([np.stack([H.rand_poly(q + p, N, rng) for _ in range(max(sizes))]) for _ in range(n)])
    e = np.rint(rng.normal(0, 3.2, (n, max(sizes), N))).astype(np.int64)
    want = E.gen_evaluation_key(params, sk_in, sk_out, [[a[i, j] for j in range(sizes[i])] for i in range(n)], [[e[i, j] for j in range(sizes[i])] for i in range(n)], pw2)
    ctx = lb.Context(logN, q, p)
    try:
        evk = lb.encryptor.KeyGenerator(ctx).GenEvaluationKey(ctx.to_device(sk_in), ctx.to_device(sk_out), ctx.to_device(a), torch.from_numpy(e).cuda(), pw2, sizes)
        got = ctx.to_host(evk.data)
        for i in range(n):
            for j in range(sizes[i]):
                assert np.array_equal(got[i, j], want.data[i, j]), (i, j)
    finally:
        ctx.close()


def test_samplers_distributions_and_streams():
    """Wrapper-level stream handling (the kernels themselves are pinned in tests/test_gpu_samplers.py): an explicit stream id
    reproduces its draw, another id gives another draw, and a polynomial does not depend on the batch it was drawn in."""
    import lattigo_b200 as lb
    logN = 12
    q, p = O.gen_moduli(logN + 1, [55, 45, 30], [61])
    ctx = lb.Context(logN, q, p)
    try:
        S = lb.encryptor.Samplers(ctx, seed=0x1234567890ABCDEF)
        u = ctx.to_host(S.UniformQP(2, 0, batch=4, stream_id=7))
        assert np.array_equal(u, ctx.to_host(S.UniformQP(2, 0, batch=4, stream_id=7)))      # reproducible
        assert not np.array_equal(u, ctx.to_host(S.UniformQP(2, 0, batch=4, stream_id=8)))
        # the counter-based streams do not depend on the batch they were drawn in
        assert np.array_equal(u[:2], ctx.to_host(S.UniformQP(2, 0, batch=2, stream_id=7)))
        g = S.Gaussian(3.2, 19.2, batch=3, stream_id=5).cpu().numpy()
        assert np.array_equal(g[:1], S.Gaussian(3.2, 19.2, batch=1, stream_id=5).cpu().numpy())
        assert np.array_equal(S.Ternary(H=32, batch=3, stream_id=6).cpu().numpy()[:2], S.Ternary(H=32, batch=2, stream_id=6).cpu().numpy())
    finally:
        ctx.close()


def test_device_keygen_end_to_end_keyswitch_noise():
    """Everything sampled on the device: s_in, s_out (ternary), a (uniform), e (Gaussian) -> evaluation key -> GadgetProduct;
    the oracle-side noise of the switched ciphertext must be key-switch sized."""
    import torch
    import lattigo_b200 as lb
    logN = 10
    q, p = O.gen_moduli(logN + 1, [55, 45, 45, 45], [55, 55])
    params = O.Parameters(logN, q, p)
    N = params.N()
    ctx = lb.Context(logN, q, p)
    try:
        S = lb.encryptor.Samplers(ctx, seed=99)
        levelQ, levelP = len(q) - 1, len(p) - 1
        n = params.BaseRNSDecompositionVectorSize(levelQ, levelP)
        s_in = S.Ternary(H=N // 4); s_out = S.Ternary(P=2.0 / 3.0)
        skq, skp = lb.encryptor.small_poly_to_rns(ctx, torch.cat([s_in, s_out]), levelQ, levelP)
        ringQ, ringP = ctx.ringQ, ctx.ringP
        ringQ.NTT(skq, skq); ringQ.MForm(skq, skq); ringP.NTT(skp, skp); ringP.MForm(skp, skp)
        sk_in = skq[0].contiguous(); sk_out = torch.cat([skq[1], skp[1]]).contiguous()
        a = S.UniformQP(levelQ, levelP, batch=n).view(n, 1, levelQ + 1 + levelP + 1, N)
        e = S.Gaussian(3.2, 19.2, batch=n).view(n, 1, N)
        evk = lb.encryptor.KeyGenerator(ctx).GenEvaluationKey(sk_in, sk_out, a, e)
        rng = np.random.default_rng(5)
        cx = H.rand_poly(q, N, rng)
        c0 = ctx.new_poly(levelQ + 1); c1 = ctx.new_poly(levelQ + 1)
        lb.Evaluator(ctx).GadgetProduct(levelQ, ctx.to_device(cx), evk, c0, c1)
        noise = H.keyswitch_noise_log2(params, levelQ, cx, [ctx.to_host(c0), ctx.to_host(c1)], s_in.cpu().numpy()[0], s_out.cpu().numpy()[0])
        assert noise < 16, noise
    finally:
        ctx.close()
