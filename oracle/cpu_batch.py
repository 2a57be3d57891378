"""oracle/cpu_batch.py -- TEST / BASELINE INFRASTRUCTURE ONLY.

Python side of oracle/lattigo_cpu_batch.c: builds the library on the box it runs on (gcc -O3 -march=native, as
BASELINE.md section 3 asks; the binary is therefore NOT portable and is rebuilt whenever the host CPU changes), flattens
the oracle's constants (oracle.Parameters / Decomposer / BasisExtender: the big-integer restatements of
ring/basis_extension.go:25-172,318-377 and ring/ring.go:329-346) into the C plan, and runs batches of ciphertext pairs on
a chosen number of threads. Used by bench.py's cpu_baseline / --impl reference legs and by tests/test_cpu_batch.py."""
import ctypes
import hashlib
import os
import platform
import shutil
import subprocess
import tempfile
from typing import Optional, Sequence

import numpy as np

from . import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
U64 = np.uint64


def _cpu_tag() -> str:
    flags = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("flags") or ln.startswith("model name"):
                flags += ln
                if ln.startswith("flags"):
                    break
    except OSError:
        flags = platform.processor()
    return hashlib.sha1(flags.encode()).hexdigest()[:10]


_SRCS = [os.path.join(_HERE, "lattigo_cpu_batch.c"), os.path.join(_HERE, "lattigo_oracle.c")]
_BUILD = os.path.join(_HERE, "_build")


def _target(out_dir: str) -> str:
    return os.path.join(out_dir, "liblattigo_cpubatch_%s.so" % _cpu_tag())


def _stale(out: str) -> bool:
    return not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in _SRCS)


def build(force: bool = False, out_dir: Optional[str] = None) -> str:
    """gcc -O3 -march=native of lattigo_cpu_batch.c (+ the #included lattigo_oracle.c) into `out_dir` (default oracle/_build/)."""
    out = _target(out_dir or _BUILD)
    if force or _stale(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        cmd = ["gcc", "-O3", "-march=native", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math",
               "-Wall", "-Wextra", "-Wno-unused-function", "-o", out, _SRCS[0]]
        subprocess.check_call(cmd)
    return out


class _Plan(ctypes.Structure):
    _fields_ = [("N", ctypes.c_int), ("nQ", ctypes.c_int), ("nP", ctypes.c_int), ("nd", ctypes.c_int),
                ("qi_overf", ctypes.c_int), ("pi_overf", ctypes.c_int),
                ("mod", ctypes.c_void_p), ("qinv", ctypes.c_void_p), ("bred", ctypes.c_void_p), ("ninv", ctypes.c_void_p),
                ("roots_fwd", ctypes.c_void_p), ("roots_bwd", ctypes.c_void_p), ("evk", ctypes.c_void_p),
                ("dig_start", ctypes.c_void_p), ("dig_n", ctypes.c_void_p), ("dmax", ctypes.c_int),
                ("dec_qhalf", ctypes.c_void_p), ("dec_inv", ctypes.c_void_p), ("dec_c", ctypes.c_void_p),
                ("dec_v", ctypes.c_void_p), ("dec_half_t", ctypes.c_void_p),
                ("md_phalf_p", ctypes.c_void_p), ("md_inv", ctypes.c_void_p), ("md_c", ctypes.c_void_p), ("md_v", ctypes.c_void_p),
                ("md_phalf_q", ctypes.c_void_p), ("md_scal", ctypes.c_void_p), ("rescale", ctypes.c_void_p)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = None
        if _stale(_target(_BUILD)):
            # build() ran on another host CPU, or not at all: compile for this host outside the source tree
            tmp = tempfile.mkdtemp(prefix="lattigo_cpubatch_")
        L = ctypes.CDLL(build(out_dir=tmp))
        if tmp:
            shutil.rmtree(tmp)
        p, i, u, z = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_size_t
        L.lo_ckks_mulrelin_rescale_batch.argtypes = [ctypes.POINTER(_Plan), p, p, z, p, p, i, i, p, p]
        L.lo_ckks_mulrelin_rescale_batch.restype = ctypes.c_double
        L.lb_ntt.argtypes = [p, p, i, u, u, p, p]
        L.lb_ntt_lazy.argtypes = [p, p, i, u, u, p]
        L.lb_intt.argtypes = [p, p, i, u, u, u, p]
        L.lo_batch_release.argtypes = []
        _lib = L
    return _lib


class CKKSBatchPlan:
    """Constants of MulRelinNew + Rescale at level `level` (default: max) for `params` and the relinearisation key."""

    def __init__(self, params: O.Parameters, rlk: O.GadgetCiphertext, level: Optional[int] = None):
        ringQ, ringP = params.ringQ, params.ringP
        nQfull = ringQ.ModuliChainLength()
        level = params.MaxLevelQ() if level is None else level
        levelP = rlk.LevelP()
        assert levelP >= 1, "multiple-P key-switch only (core/rlwe/evaluator_gadget_product.go:129-201)"
        nQ, nP = level + 1, levelP + 1
        N = params.N()
        Qc, Pc = ringQ.ModuliChain(), ringP.ModuliChain()
        mods = Qc[:nQ] + Pc[:nP]
        subs = ringQ.SubRings[:nQ] + ringP.SubRings[:nP]
        nT = nQ + nP
        nd = params.BaseRNSDecompositionVectorSize(level, levelP)
        k = self._keep = {}
        k["mod"] = np.array(mods, dtype=U64)
        k["qinv"] = np.array([s.MRedConstant for s in subs], dtype=U64)
        k["bred"] = np.array([c for s in subs for c in s.BRedConstant], dtype=U64)
        k["ninv"] = np.array([s.NInv for s in subs], dtype=U64)
        k["rf"] = (ctypes.c_void_p * nT)(*[s.RootsForward.ctypes.data for s in subs])
        k["rb"] = (ctypes.c_void_p * nT)(*[s.RootsBackward.ctypes.data for s in subs])
        k["subs"] = subs
        # evaluation key restricted to the limbs in use: [nd][2][nQ+nP][N]
        data = rlk.data
        assert data.shape[1] == 1 and rlk.BaseTwoDecomposition == 0
        sel = list(range(nQ)) + list(range(rlk.nQ, rlk.nQ + nP))
        if nQ == rlk.nQ and nP == rlk.nP and data.flags["C_CONTIGUOUS"]:
            k["evk"] = data.reshape(data.shape[0], 2, nT, N)[:nd]
        else:
            k["evk"] = np.ascontiguousarray(data[:nd, 0][:, :, sel, :])
        assert k["evk"].flags["C_CONTIGUOUS"]
        # Decomposer tables (ring/basis_extension.go:381-502)
        dec = O.Decomposer(ringQ, ringP)
        nbPi = nP
        dmax = nbPi
        dig_start = np.zeros(nd, dtype=np.int32); dig_n = np.zeros(nd, dtype=np.int32)
        qhalf = np.zeros((nd, dmax), dtype=U64); inv = np.zeros((nd, dmax), dtype=U64)
        C = np.zeros((nd, nT, dmax), dtype=U64); V = np.zeros((nd, nT, dmax + 1), dtype=U64)
        half_t = np.zeros((nd, nT), dtype=U64)
        for d in range(nd):
            st = d * nbPi
            decompLvl = nbPi - 2 if level > nbPi * (d + 1) - 1 else (level % nbPi) - 1
            dig_start[d] = st
            if decompLvl < 0:
                dig_n[d] = 1
                continue
            ed = min(st + nbPi, level + 1)
            nD = ed - st
            assert nD == decompLvl + 2
            dig_n[d] = nD
            muc = dec._muc(nbPi, d, decompLvl)
            QBig = 1
            for x in Qc[st:ed]:
                QBig *= x
            QHalf = QBig >> 1
            qhalf[d, :nD] = [QHalf % Qc[i] for i in range(st, ed)]
            inv[d, :nD] = muc.qoverqiinvqi
            for g in range(nT):
                src = g if g < nQ else nQfull + (g - nQ)
                C[d, g, :nD] = muc.qoverqimodp[src]
                V[d, g, :nD + 1] = muc.vtimesqmodp[src]
                half_t[d, g] = QHalf % mods[g]
        k.update(dig_start=dig_start, dig_n=dig_n, qhalf=qhalf, inv=inv, C=C, V=V, half_t=half_t)
        # ModDown P -> Q (ring/basis_extension.go:235-256)
        be = O.BasisExtender(ringQ, ringP)
        muc = be.constantsPtoQ[levelP]
        PBig = 1
        for x in Pc[:nP]:
            PBig *= x
        PHalf = PBig >> 1
        k["md_phalf_p"] = np.array([PHalf % x for x in Pc[:nP]], dtype=U64)
        k["md_inv"] = np.ascontiguousarray(muc.qoverqiinvqi)
        k["md_c"] = np.ascontiguousarray(muc.qoverqimodp[:nQ])
        k["md_v"] = np.ascontiguousarray(muc.vtimesqmodp[:nQ])
        k["md_phalf_q"] = np.array([PHalf % x for x in Qc[:nQ]], dtype=U64)
        k["md_scal"] = np.array([Qc[i] - be.modDownConstantsPtoQ[levelP][i] for i in range(nQ)], dtype=U64)
        k["rescale"] = np.array(ringQ.RescaleConstants[level - 1][:level], dtype=U64)
        pl = _Plan()
        pl.N, pl.nQ, pl.nP, pl.nd = N, nQ, nP, nd
        pl.qi_overf = params.QiOverflowMargin(level) >> 1
        pl.pi_overf = params.PiOverflowMargin(levelP) >> 1
        pl.dmax = dmax
        for name, key in (("mod", "mod"), ("qinv", "qinv"), ("bred", "bred"), ("ninv", "ninv"), ("evk", "evk"),
                          ("dig_start", "dig_start"), ("dig_n", "dig_n"), ("dec_qhalf", "qhalf"), ("dec_inv", "inv"),
                          ("dec_c", "C"), ("dec_v", "V"), ("dec_half_t", "half_t"), ("md_phalf_p", "md_phalf_p"),
                          ("md_inv", "md_inv"), ("md_c", "md_c"), ("md_v", "md_v"), ("md_phalf_q", "md_phalf_q"),
                          ("md_scal", "md_scal"), ("rescale", "rescale")):
            setattr(pl, name, k[key].ctypes.data)
        pl.roots_fwd = ctypes.cast(k["rf"], ctypes.c_void_p).value
        pl.roots_bwd = ctypes.cast(k["rb"], ctypes.c_void_p).value
        self.plan = pl
        self.N, self.nQ, self.nP = N, nQ, nP

    def run(self, a: np.ndarray, b: np.ndarray, npairs: int, nthreads: int, store: bool = False, store_mid: bool = False,
            cpus: Optional[Sequence[int]] = None):
        """a, b: (npairs, 2, nQ, N) or (1, 2, nQ, N) (every pair reads the same inputs, like the reference's RunParallel
        benchmark). Returns (wall_seconds, per_pair_seconds, out or None, mid or None)."""
        assert a.dtype == U64 and b.dtype == U64 and a.flags["C_CONTIGUOUS"] and b.flags["C_CONTIGUOUS"]
        assert a.shape[1:] == (2, self.nQ, self.N) and b.shape == a.shape
        stride = 0 if a.shape[0] == 1 and npairs > 1 else 2 * self.nQ * self.N
        assert a.shape[0] in (1, npairs)
        out = np.zeros((npairs, 2, self.nQ - 1, self.N), dtype=U64) if store else None
        mid = np.zeros((npairs, 2, self.nQ, self.N), dtype=U64) if store_mid else None
        per = np.zeros(npairs, dtype=np.float64)
        cp = None
        if cpus is not None:
            assert len(cpus) >= nthreads
            cp = (ctypes.c_int * nthreads)(*[int(c) for c in cpus[:nthreads]])
        t = lib().lo_ckks_mulrelin_rescale_batch(ctypes.byref(self.plan), a.ctypes.data, b.ctypes.data, stride,
                                                 out.ctypes.data if store else None, mid.ctypes.data if store_mid else None,
                                                 npairs, nthreads, cp, per.ctypes.data)
        assert t >= 0, "lo_ckks_mulrelin_rescale_batch failed (%r)" % t
        return t, per, out, mid


def usable_cpus():
    """CPUs this process may actually use: affinity mask, capped by the cgroup CPU quota (cpu.max) if any."""
    aff = sorted(os.sched_getaffinity(0))
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except (OSError, ValueError, IndexError):
            continue
    n = len(aff)
    if quota is not None:
        n = max(1, min(n, int(quota)))
    return {"affinity": len(aff), "cgroup_quota": quota, "os_cpu_count": os.cpu_count(), "usable": n, "cpu_ids": aff}
