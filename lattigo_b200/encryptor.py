"""Host-side mirror of the encryptor / key-generator inner loops and the samplers (include/lattigo_b200.h, csrc/encrypt.cu):
rlwe.Encryptor.EncryptZero (core/rlwe/encryptor.go:170-430), rlwe.KeyGenerator.GenEvaluationKey
(core/rlwe/keygenerator.go:261-330), ring.{Uniform,Ternary,Gaussian}Sampler."""
from __future__ import annotations

import ctypes

from . import _lib
from .ring import Context, RING_Q, RING_P, _dptr, _stream
from .rlwe import GadgetCiphertext


class Samplers:
    """Device samplers: the reference's distributions on counter-based streams keyed by (seed, stream id)."""

    def __init__(self, ctx: Context, seed: int):
        self.ctx, self.seed = ctx, seed & 0xFFFFFFFFFFFFFFFF
        self._next = 0

    def _sid(self, stream_id):
        if stream_id is None:
            self._next += 1
            return self._next
        return stream_id

    def Uniform(self, ring: int, level: int, batch: int = 1, stream_id=None):
        out = self.ctx.new_poly(level + 1, batch)
        _lib.check(_lib.lib().lgpu_sample_uniform(self.ctx.h, ring, level, self.seed, self._sid(stream_id), _dptr(out), batch, (level + 1) * self.ctx.N, _stream()))
        return out

    def UniformQP(self, levelQ: int, levelP: int, batch: int = 1, stream_id=None):
        """A uniform ringqp.Poly block (batch, levelQ+1 + levelP+1, N). Both rings draw from one stream id: the device keys
        every row by its limb, so the Q and P rows never share random blocks."""
        sid = self._sid(stream_id)
        rows = levelQ + 1 + levelP + 1
        out = self.ctx.new_poly(rows, batch)
        L = _lib.lib()
        _lib.check(L.lgpu_sample_uniform(self.ctx.h, RING_Q, levelQ, self.seed, sid, _dptr(out), batch, rows * self.ctx.N, _stream()))
        if levelP >= 0:
            _lib.check(L.lgpu_sample_uniform(self.ctx.h, RING_P, levelP, self.seed, sid,
                                             ctypes.c_void_p(out.data_ptr() + 8 * (levelQ + 1) * self.ctx.N), batch, rows * self.ctx.N, _stream()))
        return out

    def _small(self, batch):
        return self.ctx.new_poly(1, batch).view(batch, self.ctx.N)

    def Ternary(self, P: float = 0.0, H: int = 0, batch: int = 1, stream_id=None):
        out = self._small(batch)
        _lib.check(_lib.lib().lgpu_sample_ternary(self.ctx.h, float(P), int(H), self.seed, self._sid(stream_id), _dptr(out), batch, _stream()))
        return out

    def Gaussian(self, sigma: float = 3.2, bound: float = 19.2, batch: int = 1, stream_id=None):
        out = self._small(batch)
        _lib.check(_lib.lib().lgpu_sample_gaussian(self.ctx.h, float(sigma), float(bound), self.seed, self._sid(stream_id), _dptr(out), batch, _stream()))
        return out


def small_poly_to_rns(ctx: Context, small, levelQ: int, levelP: int = -1):
    """(batch, N) signed coefficients -> (batch, levelQ+1, N) [and (batch, levelP+1, N)] residues."""
    batch = small.shape[0]
    outq = ctx.new_poly(levelQ + 1, batch)
    outp = ctx.new_poly(levelP + 1, batch) if levelP >= 0 else None
    _lib.check(_lib.lib().lgpu_small_poly_to_rns(ctx.h, levelQ, levelP, _dptr(small), _dptr(outq), _dptr(outp), batch, (levelQ + 1) * ctx.N,
                                                 (levelP + 1) * ctx.N, _stream()))
    return (outq, outp) if levelP >= 0 else outq


class Encryptor:
    """rlwe.Encryptor's zero-encryption paths with the sampled polynomials as arguments."""

    def __init__(self, ctx: Context):
        self.ctx = ctx

    def EncryptZeroPk(self, levelQ: int, pk, u, e0, e1, is_ntt=True, is_montgomery=False):
        """pk: (2, nQ + nP, N) device tensor; u, e0, e1: (batch, N) int64 -> (batch, 2, levelQ+1, N)."""
        import torch
        batch = u.shape[0]
        out = torch.empty((batch, 2, levelQ + 1, self.ctx.N), dtype=torch.int64, device=u.device)
        _lib.check(_lib.lib().lgpu_encrypt_zero_pk(self.ctx.h, levelQ, _dptr(pk), _dptr(u), _dptr(e0), _dptr(e1), _dptr(out), int(is_ntt), int(is_montgomery),
                                                   batch, _stream()))
        return out

    def EncryptZeroSk(self, levelQ: int, levelP: int, sk, c1, e, is_ntt=True, is_montgomery=False):
        """sk: (nQ + nP, N); c1: (batch, levelQ+1 + levelP+1, N) uniform (NTT domain); e: (batch, N) -> c0, same shape as c1."""
        import torch
        c0 = torch.empty_like(c1)
        _lib.check(_lib.lib().lgpu_encrypt_zero_sk(self.ctx.h, levelQ, levelP, _dptr(sk), _dptr(c1), _dptr(e), _dptr(c0), int(is_ntt), int(is_montgomery),
                                                   c1.shape[0], _stream()))
        return c0


class KeyGenerator:
    """rlwe.KeyGenerator.GenEvaluationKey at the maximum levels (core/rlwe/keygenerator.go:261-330)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx

    def GenEvaluationKey(self, skIn, skOut, a, e, pw2: int = 0, pw2_sizes=None) -> GadgetCiphertext:
        """a: (digits, pw2, nQ + nP, N) uniform; e: (digits, pw2, N) int64. Returns the device-resident key."""
        import torch
        ctx = self.ctx
        nd, npw2 = a.shape[0], a.shape[1]
        rows = len(ctx.Q) + len(ctx.P)
        data = torch.zeros((nd, npw2, 2, rows, ctx.N), dtype=torch.int64, device=a.device)
        data[:, :, 1] = a
        evk = GadgetCiphertext(ctx, data, len(ctx.Q) - 1, len(ctx.P) - 1, pw2, pw2_sizes)
        _lib.check(_lib.lib().lgpu_gen_evaluation_key(ctx.h, _dptr(skIn), _dptr(skOut), evk.ref(), _dptr(e.contiguous()), _stream()))
        return evk
