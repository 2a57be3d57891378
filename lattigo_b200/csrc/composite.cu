// composite.cu -- the multi-kernel operations of the hot path, written as the reference composes them:
//   BasisExtender.ModDownQPtoQ / ModDownQPtoQNTT / ModDownQPtoP      ring/basis_extension.go:215-278
//   Ring.DivRound/DivFloorByLastModulus[NTT][Many]                   ring/scaling.go:6-212
//   Ring.AutomorphismNTTIndex / AutomorphismNTTWithIndex[ThenAddLazy] / Automorphism   ring/automorphism.go
//   rlwe.Evaluator.DecomposeSingleNTT / DecomposeNTT / GadgetProduct[Lazy|Hoisted[Lazy]] / ModDown
//                                                                    core/rlwe/evaluator_gadget_product.go
//   rlwe.Evaluator.Automorphism / AutomorphismHoisted / Relinearize  core/rlwe/evaluator_automorphism.go,
//                                                                    core/rlwe/evaluator_evaluationkey.go:121-148
//   ckks.Evaluator.mulRelin (ct x ct) + Rescale                      schemes/ckks/evaluator.go:477-515,764-872
// All take a batch of independent polynomials / ciphertexts. Scratch comes from the stream-ordered allocator
// (cudaMallocAsync), so concurrent callers on different streams never share buffers (the reference's ops are
// safe for concurrent use, ring/ring.go:184-186).
#include <cstdlib>
#include <cstring>
#include "../../include/lattigo_b200.h"
#include "composite.h"
#include "modarith.cuh"

namespace lgpu {

// ---------------------------------------------------------------------------------------------------------
// ModDown
// ---------------------------------------------------------------------------------------------------------
static int moddown_finish(const Ctx* c, bool toQ, int levelQ, int levelP, CSpan ext, CSpan p1, Span p2, int batch, cudaStream_t st) {
    // (p1 - ext) * (-S^-1): SubThenMulScalarMontgomeryTwoModulus(ext, p1, q_i - modDownConstants[i], p2)
    const int n = toQ ? levelQ + 1 : levelP + 1;
    std::vector<u64> s(n);
    for (int i = 0; i < n; i++) {
        const u64 q = toQ ? c->Q[i] : c->P[i];
        const u64 k = toQ ? c->mdc_PtoQ[(size_t)levelP * c->nQ + i] : c->mdc_QtoP[(size_t)levelQ * c->nP + i];
        s[i] = q - k;
    }
    RowMap rm = rows_range(toQ ? 0 : c->nQ, 0, n);
    return launch_vecop(c, rm, LGPU_OP_SUBTHENMULSCALARMONTGOMERYTWOMODULUS, ext, p1, p2, batch, s.data(), nullptr, 0, 0, c->N, st);
}

int moddown_qp_to_q(const Ctx* c, int levelQ, int levelP, CSpan p1Q, CSpan p1P, Span p2Q, int batch, cudaStream_t st) {
    const size_t N = c->N, nq = levelQ + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * nq * N, st)) return -1;
    Span bq{buf.p, N, nq * N};
    if (launch_modup_qp(c, false, levelQ, levelP, p1P, bq, batch, st)) return -1;
    return moddown_finish(c, true, levelQ, levelP, CSpan{bq.p, N, nq * N}, p1Q, p2Q, batch, st);
}

int moddown_qp_to_q_ntt(const Ctx* c, int levelQ, int levelP, CSpan p1Q, CSpan p1P, Span p2Q, int batch, cudaStream_t st) {
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * (nq + np) * N, st)) return -1;
    Span bp{buf.p, N, np * N};
    Span bq{buf.p + (size_t)batch * np * N, N, nq * N};
    if (launch_intt(c, rows_range(c->nQ, 0, (int)np), p1P, bp, batch, NTT_EXACT_LAZY, st)) return -1;
    if (launch_modup_qp(c, false, levelQ, levelP, CSpan{bp.p, N, np * N}, bq, batch, st)) return -1;
    if (launch_ntt(c, rows_range(0, 0, (int)nq), CSpan{bq.p, N, nq * N}, bq, batch, NTT_EXACT_LAZY, st)) return -1;
    return moddown_finish(c, true, levelQ, levelP, CSpan{bq.p, N, nq * N}, p1Q, p2Q, batch, st);
}

int moddown_qp_to_p(const Ctx* c, int levelQ, int levelP, CSpan p1Q, CSpan p1P, Span p2P, int batch, cudaStream_t st) {
    const size_t N = c->N, np = levelP + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * np * N, st)) return -1;
    Span bp{buf.p, N, np * N};
    if (launch_modup_qp(c, true, levelQ, levelP, p1Q, bp, batch, st)) return -1;
    return moddown_finish(c, false, levelQ, levelP, CSpan{bp.p, N, np * N}, p1P, p2P, batch, st);
}

// ---------------------------------------------------------------------------------------------------------
// DivRound / DivFloor by last modulus (ring/scaling.go). `ring` selects Q or P; level = input level.
// ---------------------------------------------------------------------------------------------------------
static const std::vector<u64>& ring_mods(const Ctx* c, int ring) { return ring == LGPU_RING_Q ? c->Q : c->P; }
static int ring_off(const Ctx* c, int ring) { return ring == LGPU_RING_Q ? 0 : c->nQ; }
static u64 rescale_const(const Ctx* c, int ring, int level, int i) {
    const std::vector<u64>& rc = ring == LGPU_RING_Q ? c->rescaleQ : c->rescaleP;
    const int n = ring == LGPU_RING_Q ? c->nQ : c->nP;
    return rc[(size_t)(level - 1) * n + i];
}

// DivRoundByLastModulusNTT (:101-122) / DivFloorByLastModulusNTT (:6-22)
int div_by_last_modulus_ntt(const Ctx* c, int ring, int level, bool round, CSpan p0, Span p1, int batch, cudaStream_t st) {
    if (level < 1) { set_error("cannot divide by last modulus at level 0"); return -1; }
    const std::vector<u64>& M = ring_mods(c, ring);
    const int off = ring_off(c, ring);
    const size_t N = c->N;
    Scratch buf;
    if (buf.alloc((size_t)batch * (1 + level) * N, st)) return -1;
    Span b0{buf.p, N, N};                                   // [batch][1][N]
    Span b1{buf.p + (size_t)batch * N, N, (size_t)level * N};  // [batch][level][N]
    // INTTLazy of the last row
    RowMap rl = rows_range(off + level, level, 1);
    RowMap rl0 = rl; rl0.drow[0] = 0;
    {
        // in: row `level` of p0 ; out: row 0 of b0
        NttMode mode = NTT_EXACT_LAZY;
        CSpan in{p0.p + (size_t)level * p0.row_stride, p0.row_stride, p0.batch_stride};
        if (launch_intt(c, rl0, in, b0, batch, mode, st)) return -1;
    }
    const u64 qL = M[level];
    const u64 pHalf = (qL - 1) >> 1;
    std::vector<u64> s0(level), sc(level);
    if (round) {
        if (launch_vecop(c, rl0, LGPU_OP_ADDSCALAR, CSpan{b0.p, N, N}, CSpan{nullptr, 0, 0}, b0, batch, nullptr, nullptr, pHalf, 0, c->N, st)) return -1;
        for (int i = 0; i < level; i++) s0[i] = M[i] - (pHalf % M[i]);
    } else {
        for (int i = 0; i < level; i++) s0[i] = 0;
    }
    for (int i = 0; i < level; i++) sc[i] = rescale_const(c, ring, level, i);
    RowMap rm = rows_range(off, 0, level);
    // broadcast the single row to all lower limbs (AddScalarLazy with row stride 0), NTTLazy, then (b1 - p0) * const
    if (launch_vecop(c, rm, LGPU_OP_ADDSCALARLAZY, CSpan{b0.p, 0, N}, CSpan{nullptr, 0, 0}, b1, batch, s0.data(), nullptr, 0, 0, c->N, st)) return -1;
    if (launch_ntt(c, rm, CSpan{b1.p, N, (size_t)level * N}, b1, batch, NTT_EXACT_LAZY, st)) return -1;
    return launch_vecop(c, rm, LGPU_OP_SUBTHENMULSCALARMONTGOMERYTWOMODULUS, CSpan{b1.p, N, (size_t)level * N}, p0, p1, batch,
                        sc.data(), nullptr, 0, 0, c->N, st);
}

// DivRoundByLastModulus (:126-144) / DivFloorByLastModulus (:26-33), coefficient domain.
int div_by_last_modulus(const Ctx* c, int ring, int level, bool round, CSpan p0, Span p1, int batch, cudaStream_t st) {
    if (level < 1) { set_error("cannot divide by last modulus at level 0"); return -1; }
    const std::vector<u64>& M = ring_mods(c, ring);
    const int off = ring_off(c, ring);
    const size_t N = c->N;
    std::vector<u64> sc(level);
    for (int i = 0; i < level; i++) sc[i] = rescale_const(c, ring, level, i);
    RowMap rm = rows_range(off, 0, level);
    CSpan last{p0.p + (size_t)level * p0.row_stride, 0, p0.batch_stride};   // broadcast row `level`
    if (!round)
        return launch_vecop(c, rm, LGPU_OP_SUBTHENMULSCALARMONTGOMERYTWOMODULUS, last, p0, p1, batch, sc.data(), nullptr, 0, 0, c->N, st);
    Scratch buf;
    if (buf.alloc((size_t)batch * (1 + level) * N, st)) return -1;
    Span b0{buf.p, N, N};
    Span b1{buf.p + (size_t)batch * N, N, (size_t)level * N};
    const u64 pHalf = (M[level] - 1) >> 1;
    RowMap rl0 = rows_range(off + level, 0, 1);
    if (launch_vecop(c, rl0, LGPU_OP_ADDSCALAR, CSpan{last.p, 0, p0.batch_stride}, CSpan{nullptr, 0, 0}, b0, batch, nullptr, nullptr, pHalf, 0, c->N, st)) return -1;
    std::vector<u64> s0(level);
    for (int i = 0; i < level; i++) s0[i] = M[i] - (pHalf % M[i]);
    if (launch_vecop(c, rm, LGPU_OP_ADDSCALARLAZYTHENNEGTWOMODULUSLAZY, p0, CSpan{nullptr, 0, 0}, b1, batch, s0.data(), nullptr, 0, 0, c->N, st)) return -1;
    return launch_vecop(c, rm, LGPU_OP_ADDLAZYTHENMULSCALARMONTGOMERY, CSpan{b0.p, 0, N}, CSpan{b1.p, N, (size_t)level * N}, p1, batch,
                        sc.data(), nullptr, 0, 0, c->N, st);
}

// Div{Round,Floor}ByLastModulusMany[NTT] (:37-97, :148-212)
int div_by_last_modulus_many(const Ctx* c, int ring, int level, bool round, bool ntt, int nb, CSpan p0, Span p1, int batch, cudaStream_t st) {
    const size_t N = c->N;
    if (nb < 0 || nb > level) { set_error("invalid number of rescales"); return -1; }
    if (nb == 0) {
        if (p0.p != p1.p)
            LGPU_CUDA_OK(cudaMemcpy2DAsync(p1.p, p1.batch_stride * 8, p0.p, p0.batch_stride * 8, (size_t)(level + 1) * N * 8, batch,
                                           cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    if (ntt && nb == 1 && round) return div_by_last_modulus_ntt(c, ring, level, true, p0, p1, batch, st);
    const int off = ring_off(c, ring);
    Scratch buf;
    if (buf.alloc((size_t)batch * (level + 1) * N, st)) return -1;
    Span b{buf.p, N, (size_t)(level + 1) * N};
    CSpan cur = p0;
    if (ntt) {
        // INTT -> nb coefficient-domain divisions -> NTT (:37-61 floor; :158-171 round with nb > 1)
        if (launch_intt(c, rows_range(off, 0, level + 1), p0, b, batch, NTT_CANONICAL, st)) return -1;
        cur = CSpan{b.p, b.row_stride, b.batch_stride};
        int lv = level;
        for (int i = 0; i < nb; i++, lv--)
            if (div_by_last_modulus(c, ring, lv, round, cur, b, batch, st)) return -1;
        return launch_ntt(c, rows_range(off, 0, lv + 1), cur, p1, batch, NTT_CANONICAL, st);
    }
    int lv = level;
    for (int i = 0; i < nb; i++, lv--) {
        Span dst = (i == nb - 1) ? p1 : b;
        if (div_by_last_modulus(c, ring, lv, round, cur, dst, batch, st)) return -1;
        cur = CSpan{dst.p, dst.row_stride, dst.batch_stride};
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Automorphisms
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 brev_bits(u64 x, int bits) { return __brevll(x) >> (64 - bits); }

// AutomorphismNTTIndex, ring/automorphism.go:12-34
__global__ void auto_index_kernel(u64* index, int N, u64 nthroot, u64 galEl, int logNthRootHalf) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const u64 mask = nthroot - 1;
    const u64 tmp1 = 2 * brev_bits((u64)i, logNthRootHalf) + 1;
    const u64 tmp2 = ((galEl * tmp1 & mask) - 1) >> 1;
    index[i] = brev_bits(tmp2, logNthRootHalf);
}
int automorphism_ntt_index(const Ctx* c, u64 galEl, u64* d_index, cudaStream_t st) {
    int lg = 0;
    while ((1ull << (lg + 1)) < c->nthroot) lg++;   // bits.Len64(NthRoot-1) - 1
    count_launch(1);
    auto_index_kernel<<<(c->N + 255) / 256, 256, 0, st>>>(d_index, c->N, c->nthroot, galEl, lg);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

struct AutoParams {
    const u64* in; size_t in_rs, in_bs;
    u64* out; size_t out_rs, out_bs;
    const u64* index;
    int n, accumulate;
};
// AutomorphismNTTWithIndex[ThenAddLazy], ring/automorphism.go:50-109: out[j] (+)= in[index[j]]
__global__ void __launch_bounds__(256) auto_ntt_kernel(AutoParams p) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p.n) return;
    const u64 src = __ldg(p.index + j);
    const u64* in = p.in + (size_t)blockIdx.z * p.in_bs + (size_t)blockIdx.y * p.in_rs;
    u64* out = p.out + (size_t)blockIdx.z * p.out_bs + (size_t)blockIdx.y * p.out_rs;
    const u64 v = in[src];
    out[j] = p.accumulate ? out[j] + v : v;
}
int automorphism_ntt_with_index(const Ctx* c, int rows, CSpan in, const u64* d_index, Span out, bool accumulate, int batch, cudaStream_t st) {
    if (in.p == out.p) { set_error("AutomorphismNTT cannot be in-place"); return -1; }
    ProfScope ps(LGPU_KCLASS_AUTOMORPHISM, st, 8.0 * c->N * rows * batch * (accumulate ? 3 : 2), 1);
    AutoParams p{in.p, in.row_stride, in.batch_stride, out.p, out.row_stride, out.batch_stride, d_index, c->N, accumulate ? 1 : 0};
    dim3 grid((c->N + 255) / 256, rows, batch);
    auto_ntt_kernel<<<grid, 256, 0, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

struct AutoCoeffParams {
    const LimbConst* limbs; RowMap rm;
    const u64* in; size_t in_rs, in_bs;
    u64* out; size_t out_rs, out_bs;
    u64 gen; int n, logN;
};
// Ring.Automorphism (coefficient domain, Standard ring), ring/automorphism.go:158-175
__global__ void __launch_bounds__(256) auto_coeff_kernel(AutoCoeffParams p) {
    const u64 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (u64)p.n) return;
    const u64 q = p.limbs[p.rm.limb[blockIdx.y]].q;
    const u64 raw = i * p.gen;
    const u64 idx = raw & (u64)(p.n - 1);
    const u64 neg = (raw >> p.logN) & 1;
    const u64* in = p.in + (size_t)blockIdx.z * p.in_bs + (size_t)blockIdx.y * p.in_rs;
    u64* out = p.out + (size_t)blockIdx.z * p.out_bs + (size_t)blockIdx.y * p.out_rs;
    const u64 v = in[i];
    out[idx] = neg ? (q - v) : v;     // in[i]*(tmp^1) | (q - in[i])*tmp
}
// ConjugateInvariant ring, ring/automorphism.go:123-155: i runs over [0, 2N); only images below N are written, sources
// in [N, 2N) wrap to 2N - i with a sign flip. i -> i*gen mod 2N is a bijection, so every output is written exactly once.
__global__ void __launch_bounds__(256) auto_coeff_ci_kernel(AutoCoeffParams p) {
    const u64 i = blockIdx.x * blockDim.x + threadIdx.x;
    const u64 N = (u64)p.n;
    if (i >= 2 * N) return;
    const u64 raw = i * p.gen;
    const u64 idx = raw & (2 * N - 1);
    if (idx >= N) return;
    u64 neg = (raw >> (p.logN + 1)) & 1;
    u64 src = i;
    if (src >= N) { src = 2 * N - src; neg ^= 1; }
    const u64 q = p.limbs[p.rm.limb[blockIdx.y]].q;
    const u64* in = p.in + (size_t)blockIdx.z * p.in_bs + (size_t)blockIdx.y * p.in_rs;
    u64* out = p.out + (size_t)blockIdx.z * p.out_bs + (size_t)blockIdx.y * p.out_rs;
    const u64 v = in[src];
    out[idx] = neg ? (q - v) : v;
}
int automorphism_coeff(const Ctx* c, const RowMap& rm, CSpan in, u64 gen, Span out, int batch, cudaStream_t st) {
    if (in.p == out.p) { set_error("Automorphism cannot be in-place"); return -1; }
    if (c->ring_type != 0) {
        AutoCoeffParams p;
        p.limbs = c->d_limbs; p.rm = rm; p.in = in.p; p.in_rs = in.row_stride; p.in_bs = in.batch_stride;
        p.out = out.p; p.out_rs = out.row_stride; p.out_bs = out.batch_stride; p.gen = gen; p.n = c->N; p.logN = c->logN;
        ProfScope ps(LGPU_KCLASS_AUTOMORPHISM, st, 16.0 * c->N * rm.nrows * batch, 1);
        dim3 grid((2 * c->N + 255) / 256, rm.nrows, batch);
        auto_coeff_ci_kernel<<<grid, 256, 0, st>>>(p);
        LGPU_CUDA_OK(cudaGetLastError());
        return 0;
    }
    AutoCoeffParams p;
    p.limbs = c->d_limbs; p.rm = rm; p.in = in.p; p.in_rs = in.row_stride; p.in_bs = in.batch_stride;
    p.out = out.p; p.out_rs = out.row_stride; p.out_bs = out.batch_stride; p.gen = gen; p.n = c->N; p.logN = c->logN;
    ProfScope ps(LGPU_KCLASS_AUTOMORPHISM, st, 16.0 * c->N * rm.nrows * batch, 1);
    dim3 grid((c->N + 255) / 256, rm.nrows, batch);
    auto_coeff_kernel<<<grid, 256, 0, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Key-switch: decomposition, MAC, gadget products
// ---------------------------------------------------------------------------------------------------------
int base_rns_decomposition_vector_size(int levelQ, int levelP) {   // core/rlwe/params.go:543-550
    if (levelP == -1) return levelQ + 1;
    return (levelQ + levelP + 1) / (levelP + 1);
}

// MAC: acc[comp][row] (+)= MRedLazy(evk[comp][row], x[row]) over rows = Q limbs 0..levelQ then P limbs 0..levelP.
// x rows come from `xa` (QP-stacked decomposition buffer) except rows [dlo, dhi), which are read from `xb`
// (the NTT-domain input itself: DecomposeSingleNTT copies those rows, :498-500).
// Accumulators are kept in [0, 2q) between digits and canonicalised on the last digit, which is what the
// reference's periodic + final Reduce leaves (core/rlwe/evaluator_gadget_product.go:179-200).
struct MacParams {
    const LimbConst* limbs;
    const u64* evk0; const u64* evk1;      // row r of the key = evk + erow(r) * N
    int nQk;                               // Q rows in the key
    const u64* xa; size_t xa_rs, xa_bs;    // decomposition buffer, QP stacked with nq + xa_pshift Q rows
    int xa_pshift;                         // the buffer was laid out for a higher level: its P rows start xa_pshift rows later
    const u64* xb; size_t xb_rs, xb_bs;    // NTT input (digit rows)
    int dlo, dhi;
    u64* accQ[2]; size_t accQ_rs, accQ_bs;
    u64* accP[2]; size_t accP_rs, accP_bs;
    int nq, np, nQfull;
    int first, last, batch, n;
};
__global__ void __launch_bounds__(256) mac_kernel(MacParams p) {
    const int r = blockIdx.y;                       // launch row: [0,nq) Q, [nq,nq+np) P
    const bool isP = r >= p.nq;
    const int j = isP ? r - p.nq : r;
    const LimbConst L = p.limbs[isP ? p.nQfull + j : j];
    const u64 q = L.q, qinv = L.qinv, twoq = q << 1;
    const size_t erow = isP ? (size_t)p.nQk + j : (size_t)j;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;   // index of a 2-word vector
    if (i * 2 >= p.n) return;
    const ulonglong2 e0 = reinterpret_cast<const ulonglong2*>(p.evk0 + erow * p.n)[i];
    const ulonglong2 e1 = reinterpret_cast<const ulonglong2*>(p.evk1 + erow * p.n)[i];
    const bool fromB = (!isP) && r >= p.dlo && r < p.dhi;
    for (int b = blockIdx.z; b < p.batch; b += gridDim.z) {
        const u64* xrow = fromB ? p.xb + (size_t)b * p.xb_bs + (size_t)r * p.xb_rs
                                : p.xa + (size_t)b * p.xa_bs + (size_t)(isP ? r + p.xa_pshift : r) * p.xa_rs;
        const ulonglong2 x = reinterpret_cast<const ulonglong2*>(xrow)[i];
        u64* a0 = isP ? p.accP[0] + (size_t)b * p.accP_bs + (size_t)j * p.accP_rs : p.accQ[0] + (size_t)b * p.accQ_bs + (size_t)j * p.accQ_rs;
        u64* a1 = isP ? p.accP[1] + (size_t)b * p.accP_bs + (size_t)j * p.accP_rs : p.accQ[1] + (size_t)b * p.accQ_bs + (size_t)j * p.accQ_rs;
        ulonglong2 v0 = make_ulonglong2(0, 0), v1 = v0;
        if (!p.first) { v0 = reinterpret_cast<ulonglong2*>(a0)[i]; v1 = reinterpret_cast<ulonglong2*>(a1)[i]; }
        v0.x += mred_lazy(e0.x, x.x, q, qinv); v0.y += mred_lazy(e0.y, x.y, q, qinv);
        v1.x += mred_lazy(e1.x, x.x, q, qinv); v1.y += mred_lazy(e1.y, x.y, q, qinv);
        v0.x = v0.x >= twoq ? v0.x - twoq : v0.x; v0.y = v0.y >= twoq ? v0.y - twoq : v0.y;
        v1.x = v1.x >= twoq ? v1.x - twoq : v1.x; v1.y = v1.y >= twoq ? v1.y - twoq : v1.y;
        if (p.last) { v0.x = cred(v0.x, q); v0.y = cred(v0.y, q); v1.x = cred(v1.x, q); v1.y = cred(v1.y, q); }
        reinterpret_cast<ulonglong2*>(a0)[i] = v0;
        reinterpret_cast<ulonglong2*>(a1)[i] = v1;
    }
}
static int launch_mac(const MacParams& p, cudaStream_t st) {
    // algorithmic bytes: evk (2 rows) once + per ciphertext x (1 row) + accumulators (2 rows written, 2 read unless first)
    ProfScope ps(LGPU_KCLASS_MAC, st, 8.0 * p.n * (p.nq + p.np) * (2.0 + p.batch * (p.first ? 3.0 : 5.0)), 1);
    int zb = p.batch < 4 ? p.batch : 4;
    dim3 grid((p.n / 2 + 255) / 256, p.nq + p.np, zb);
    mac_kernel<<<grid, 256, 0, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

// DecomposeSingleNTT (core/rlwe/evaluator_gadget_product.go:487-510) into a QP-stacked buffer c2 ([batch][nq+np][N]).
// The digit's own rows are NOT materialised in c2 unless `copy_digit_rows` (the MAC reads them from c2NTT directly).
int decompose_single_ntt(const Ctx* c, int levelQ, int levelP, int nbPi, int digit, CSpan c2NTT, CSpan c2Inv,
                         Span c2Q, Span c2P, bool copy_digit_rows, int batch, cudaStream_t st) {
    const size_t N = c->N;
    if (launch_decompose_and_split(c, levelQ, levelP, nbPi, digit, c2Inv, c2Q, c2P, batch, st)) return -1;
    const int st0 = digit * nbPi;
    int ed0 = st0 + nbPi;
    if (ed0 > levelQ + 1) ed0 = levelQ + 1;
    // NTT of every Q row outside the digit, and of all P rows
    RowMap rq;
    rq.nrows = 0;
    for (int x = 0; x <= levelQ; x++) {
        if (x >= st0 && x < st0 + nbPi) continue;
        rq.limb[rq.nrows] = (unsigned char)x; rq.drow[rq.nrows] = (unsigned char)x; rq.nrows++;
    }
    if (rq.nrows > 0 && launch_ntt(c, rq, CSpan{c2Q.p, c2Q.row_stride, c2Q.batch_stride}, c2Q, batch, NTT_CANONICAL, st)) return -1;
    if (levelP >= 0 && launch_ntt(c, rows_range(c->nQ, 0, levelP + 1), CSpan{c2P.p, c2P.row_stride, c2P.batch_stride}, c2P, batch, NTT_CANONICAL, st)) return -1;
    if (copy_digit_rows && ed0 > st0) {
        LGPU_CUDA_OK(cudaMemcpy2DAsync(c2Q.p + (size_t)st0 * c2Q.row_stride, c2Q.batch_stride * 8,
                                       c2NTT.p + (size_t)st0 * c2NTT.row_stride, c2NTT.batch_stride * 8,
                                       (size_t)(ed0 - st0) * N * 8, batch, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

// gadgetProductMultiplePLazy, core/rlwe/evaluator_gadget_product.go:129-201 (cx in the NTT domain)
static int gadget_product_multiple_p_lazy(const Ctx* c, int levelQ, CSpan cx, const GadgetCt& evk, const AccSpans& acc, int batch, cudaStream_t st) {
    const int levelP = evk.levelP;
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    // fused pipeline (keyswitch_fused.cu) when the accumulators are QP-stacked blocks with uniform strides
    if (ks_fused_applicable(c, levelQ, evk) && cx.row_stride == N && acc.q[0].row_stride == N && acc.p[0].row_stride == N &&
        acc.p[0].p == acc.q[0].p + nq * N && acc.p[1].p == acc.q[1].p + nq * N && acc.q[1].p > acc.q[0].p &&
        acc.q[0].batch_stride == acc.q[1].batch_stride && acc.p[0].batch_stride == acc.q[0].batch_stride &&
        acc.p[1].batch_stride == acc.q[0].batch_stride) {
        Scratch inv;
        if (inv.alloc((size_t)batch * nq * N, st)) return -1;
        Span cxInv{inv.p, N, nq * N};
        if (launch_intt(c, rows_range(0, 0, (int)nq), cx, cxInv, batch, NTT_CANONICAL, st)) return -1;
        return gadget_product_multiple_p_fused(c, levelQ, cx, CSpan{inv.p, N, nq * N}, evk, acc.q[0].p, (size_t)(acc.q[1].p - acc.q[0].p),
                                               acc.q[0].batch_stride, batch, st);
    }
    Scratch buf;
    if (buf.alloc((size_t)batch * (nq + nq + np) * N, st)) return -1;
    Span cxInv{buf.p, N, nq * N};
    u64* c2 = buf.p + (size_t)batch * nq * N;
    Span c2Q{c2, N, (nq + np) * N};
    Span c2P{c2 + nq * N, N, (nq + np) * N};
    if (launch_intt(c, rows_range(0, 0, (int)nq), cx, cxInv, batch, NTT_CANONICAL, st)) return -1;
    const int nd = base_rns_decomposition_vector_size(levelQ, levelP);
    for (int i = 0; i < nd; i++) {
        if (decompose_single_ntt(c, levelQ, levelP, levelP + 1, i, cx, CSpan{cxInv.p, N, nq * N}, c2Q, c2P, false, batch, st)) return -1;
        MacParams m;
        memset(&m, 0, sizeof(m));
        m.limbs = c->d_limbs; m.evk0 = evk.at(i, 0, 0, N); m.evk1 = evk.at(i, 0, 1, N); m.nQk = evk.levelQ + 1;
        m.xa = c2; m.xa_rs = N; m.xa_bs = (nq + np) * N;
        m.xb = cx.p; m.xb_rs = cx.row_stride; m.xb_bs = cx.batch_stride;
        m.dlo = i * (levelP + 1); m.dhi = m.dlo + levelP + 1;
        for (int k = 0; k < 2; k++) { m.accQ[k] = acc.q[k].p; m.accP[k] = acc.p[k].p; }
        m.accQ_rs = acc.q[0].row_stride; m.accQ_bs = acc.q[0].batch_stride; m.accP_rs = acc.p[0].row_stride; m.accP_bs = acc.p[0].batch_stride;
        m.nq = (int)nq; m.np = (int)np; m.nQfull = c->nQ;
        m.first = (i == 0); m.last = (i == nd - 1); m.batch = batch; m.n = c->N;
        if (launch_mac(m, st)) return -1;
    }
    return 0;
}

// gadgetProductSinglePAndBitDecompLazy, core/rlwe/evaluator_gadget_product.go:203-338 (levelP <= 0)
// rgsw_mode (core/rgsw/evaluator.go:130-208): the digit is ALWAYS MaskVec(limb i, j*pw2, mask) with mask = 2^64-1 when pw2 == 0 (the raw,
// uncentred limb -- not the Decomposer's single-limb rule), and the accumulation runs over both components of the RGSW ciphertext
// (acc_first / acc_last tell which call opens and which one closes it).
static int gadget_product_single_p_lazy(const Ctx* c, int levelQ, CSpan cx, const GadgetCt& evk, const AccSpans& acc, int batch, cudaStream_t st,
                                        bool rgsw_mode = false, bool acc_first = true, bool acc_last = true) {
    const int levelP = evk.levelP;
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * (nq + nq + np) * N, st)) return -1;
    Span cxInv{buf.p, N, nq * N};
    u64* c2 = buf.p + (size_t)batch * nq * N;
    Span c2Q{c2, N, (nq + np) * N};
    Span c2P{c2 + nq * N, N, (nq + np) * N};
    if (launch_intt(c, rows_range(0, 0, (int)nq), cx, cxInv, batch, NTT_CANONICAL, st)) return -1;
    const int pw2 = evk.pw2;
    const u64 mask = pw2 ? ((1ull << pw2) - 1) : (rgsw_mode ? ~0ull : 0);
    const RowMap rqp = rows_qp(c, (int)nq, (int)np);
    int total = 0;
    for (int i = 0; i <= levelQ; i++) total += evk.pw2_sizes ? evk.pw2_sizes[i] : 1;
    int done = 0;
    for (int i = 0; i <= levelQ; i++) {
        if (mask == 0) {
            if (launch_decompose_and_split(c, levelQ, levelP, levelP + 1, i, CSpan{cxInv.p, N, nq * N}, c2Q, c2P, batch, st)) return -1;
        }
        const int nj = evk.pw2_sizes ? evk.pw2_sizes[i] : 1;
        for (int j = 0; j < nj; j++) {
            if (mask != 0) {
                // MaskVec of row i broadcast to every Q and P row, ring/vec_ops.go:870
                CSpan src{cxInv.p + (size_t)i * N, 0, nq * N};
                if (launch_vecop(c, rqp, LGPU_OP_MASK, src, CSpan{nullptr, 0, 0}, Span{c2, N, (nq + np) * N}, batch, nullptr, nullptr,
                                 (u64)(j * pw2), mask, c->N, st)) return -1;
            }
            if (mask == ~0ull) {
                // a raw limb of another prime (up to 61 bits) under every modulus: reduce first, the transforms assume lazily reduced input
                if (launch_vecop(c, rqp, LGPU_OP_REDUCE, CSpan{c2, N, (nq + np) * N}, CSpan{nullptr, 0, 0}, Span{c2, N, (nq + np) * N}, batch, nullptr, nullptr,
                                 0, 0, c->N, st)) return -1;
                if (launch_ntt(c, rqp, CSpan{c2, N, (nq + np) * N}, Span{c2, N, (nq + np) * N}, batch, NTT_CANONICAL, st)) return -1;
            } else if (launch_ntt(c, rqp, CSpan{c2, N, (nq + np) * N}, Span{c2, N, (nq + np) * N}, batch, NTT_EXACT_LAZY, st)) return -1;
            MacParams m;
            memset(&m, 0, sizeof(m));
            m.limbs = c->d_limbs; m.evk0 = evk.at(i, j, 0, N); m.evk1 = evk.at(i, j, 1, N); m.nQk = evk.levelQ + 1;
            m.xa = c2; m.xa_rs = N; m.xa_bs = (nq + np) * N;
            m.xb = nullptr; m.dlo = m.dhi = 0;
            for (int k = 0; k < 2; k++) { m.accQ[k] = acc.q[k].p; m.accP[k] = acc.p[k].p; }
            m.accQ_rs = acc.q[0].row_stride; m.accQ_bs = acc.q[0].batch_stride; m.accP_rs = acc.p[0].row_stride; m.accP_bs = acc.p[0].batch_stride;
            m.nq = (int)nq; m.np = (int)np; m.nQfull = c->nQ;
            m.first = acc_first && (done == 0); m.last = acc_last && (done == total - 1); m.batch = batch; m.n = c->N;
            if (launch_mac(m, st)) return -1;
            done++;
        }
    }
    return 0;
}

static int check_evk(const Ctx* c, int levelQ, const GadgetCt& evk) {
    if (!evk.data) { set_error("null evaluation key"); return -1; }
    if (evk.levelQ < 0 || evk.levelQ >= c->nQ || evk.levelP < -1 || evk.levelP >= c->nP) { set_error("evaluation key levels out of range"); return -1; }
    if (levelQ < 0 || levelQ > evk.levelQ) { set_error("levelQ out of range for this evaluation key"); return -1; }
    // shape of Value[digit][pw2] against what the products will index (core/rlwe/params.go:543-565)
    const int nd = evk.levelP > 0 ? base_rns_decomposition_vector_size(levelQ, evk.levelP) : levelQ + 1;
    if (evk.ndigits < nd) { set_error("evaluation key has fewer digits than BaseRNSDecompositionVectorSize(levelQ, levelP)"); return -1; }
    if (evk.npw2max < 1) { set_error("evaluation key: n_pw2_max must be >= 1"); return -1; }
    if (evk.pw2_sizes)
        for (int i = 0; i < nd; i++)
            if (evk.pw2_sizes[i] < 1 || evk.pw2_sizes[i] > evk.npw2max) { set_error("evaluation key: pw2_sizes[i] out of [1, n_pw2_max]"); return -1; }
    return 0;
}

// GadgetProductLazy (core/rlwe/evaluator_gadget_product.go:108-127), NTT-domain input and output.
int gadget_product_lazy(const Ctx* c, int levelQ, CSpan cx, const GadgetCt& evk, const AccSpans& acc, int batch, cudaStream_t st) {
    if (check_evk(c, levelQ, evk)) return -1;
    if (evk.levelP > 0) {
        if (evk.pw2 != 0) { set_error("BaseTwoDecomposition != 0 requires levelP <= 0"); return -1; }
        return gadget_product_multiple_p_lazy(c, levelQ, cx, evk, acc, batch, st);
    }
    return gadget_product_single_p_lazy(c, levelQ, cx, evk, acc, batch, st);
}

// Evaluator.ModDown (core/rlwe/evaluator_gadget_product.go:39-97), NTT -> NTT case.
int evaluator_moddown_ntt(const Ctx* c, int levelQ, int levelP, const AccSpans& acc, Span ct0, Span ct1, int batch, cudaStream_t st) {
    Span out[2] = {ct0, ct1};
    {
        const size_t N = c->N, nq = levelQ + 1;
        if (levelP >= 0 && fz_applicable(c, levelQ, levelP) && acc.q[0].row_stride == N && acc.p[0].row_stride == N &&
            acc.p[0].p == acc.q[0].p + nq * N && acc.p[1].p == acc.q[1].p + nq * N && acc.q[1].p > acc.q[0].p &&
            acc.q[0].batch_stride == acc.q[1].batch_stride && acc.p[0].batch_stride == acc.q[0].batch_stride &&
            acc.p[1].batch_stride == acc.q[0].batch_stride && ct0.row_stride == N && ct1.row_stride == N && ct1.p > ct0.p &&
            ct0.batch_stride == ct1.batch_stride && ct0.p != acc.q[0].p) {
            return moddown_ntt_fused(c, levelQ, levelP, acc.q[0].p, (size_t)(acc.q[1].p - acc.q[0].p), acc.q[0].batch_stride, nullptr, 0, 0,
                                     ct0.p, (size_t)(ct1.p - ct0.p), ct0.batch_stride, 2, batch, st);
        }
    }
    for (int k = 0; k < 2; k++) {
        CSpan aq{acc.q[k].p, acc.q[k].row_stride, acc.q[k].batch_stride};
        if (levelP != -1) {
            CSpan ap{acc.p[k].p, acc.p[k].row_stride, acc.p[k].batch_stride};
            if (moddown_qp_to_q_ntt(c, levelQ, levelP, aq, ap, out[k], batch, st)) return -1;
        } else if (aq.p != out[k].p) {
            LGPU_CUDA_OK(cudaMemcpy2DAsync(out[k].p, out[k].batch_stride * 8, aq.p, aq.batch_stride * 8, (size_t)(levelQ + 1) * c->N * 8, batch,
                                           cudaMemcpyDeviceToDevice, st));
        }
    }
    return 0;
}

// GadgetProduct (core/rlwe/evaluator_gadget_product.go:16-36): ct = ModDown(GadgetProductLazy(cx, evk)).
int gadget_product(const Ctx* c, int levelQ, CSpan cx, const GadgetCt& evk, Span ct0, Span ct1, int batch, cudaStream_t st) {
    if (check_evk(c, levelQ, evk)) return -1;
    const int levelP = evk.levelP;
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * 2 * (nq + np) * N, st)) return -1;
    AccSpans acc;
    for (int k = 0; k < 2; k++) {
        u64* base = buf.p + (size_t)k * batch * (nq + np) * N;
        acc.q[k] = Span{base, N, (nq + np) * N};
        acc.p[k] = Span{base + nq * N, N, (nq + np) * N};
    }
    if (gadget_product_lazy(c, levelQ, cx, evk, acc, batch, st)) return -1;
    return evaluator_moddown_ntt(c, levelQ, levelP, acc, ct0, ct1, batch, st);
}

// rgsw.Evaluator.ExternalProduct (core/rgsw/evaluator.go:39-88): out = ModDown( <decomp(ct[0]), rgsw[0]> + <decomp(ct[1]), rgsw[1]> ) at the
// RGSW ciphertext's levels; NTT-domain RLWE ciphertext; out may alias ct (the way both of the reference's callers use it,
// core/rgsw/rgsw_test.go:84, core/rgsw/blindrot/evaluator.go:212). The three reference code paths leave the same canonical residues:
//   levelP >= 1   externalProductInPlaceMultipleP (:210-283)            = two lazy gadget products (fused pipeline where it applies)
//   levelP <  1   externalProductInPlaceSinglePAndBitDecomp (:130-208)  = mask / raw-limb digits, Montgomery MAC
//   32-bit case   externalProduct32Bit (:90-128) + IMForm               = the same sum: IMForm(sum key * x) == sum MRed(key, x)
int rgsw_external_product(const Ctx* c, const GadgetCt& rg0, const GadgetCt& rg1, CSpan ct0, CSpan ct1, Span out0, Span out1, int batch, cudaStream_t st) {
    const int levelQ = rg0.levelQ, levelP = rg0.levelP;
    if (rg1.levelQ != levelQ || rg1.levelP != levelP || rg1.pw2 != rg0.pw2) { set_error("RGSW ciphertext: the two gadget ciphertexts differ in level or base"); return -1; }
    if (check_evk(c, levelQ, rg0) || check_evk(c, levelQ, rg1)) return -1;
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    Scratch buf;
    const size_t per = (size_t)2 * batch * (nq + np) * N;
    if (buf.alloc(2 * per, st)) return -1;
    auto stacked = [&](u64* base) {
        AccSpans a;
        for (int k = 0; k < 2; k++) {
            u64* b = base + (size_t)k * batch * (nq + np) * N;
            a.q[k] = Span{b, N, (nq + np) * N};
            a.p[k] = Span{b + nq * N, N, (nq + np) * N};
        }
        return a;
    };
    AccSpans A = stacked(buf.p), B = stacked(buf.p + per);
    if (levelP >= 1) {
        if (rg0.pw2 != 0) { set_error("RGSW external product: BaseTwoDecomposition != 0 requires levelP <= 0"); return -1; }
        if (gadget_product_multiple_p_lazy(c, levelQ, ct0, rg0, A, batch, st)) return -1;
        if (gadget_product_multiple_p_lazy(c, levelQ, ct1, rg1, B, batch, st)) return -1;
        if (launch_vecop(c, rows_qp(c, (int)nq, (int)np), LGPU_OP_ADD, CSpan{buf.p, N, (nq + np) * N}, CSpan{buf.p + per, N, (nq + np) * N},
                         Span{buf.p, N, (nq + np) * N}, 2 * batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    } else {
        if (gadget_product_single_p_lazy(c, levelQ, ct0, rg0, A, batch, st, true, true, false)) return -1;
        if (gadget_product_single_p_lazy(c, levelQ, ct1, rg1, A, batch, st, true, false, true)) return -1;
    }
    return evaluator_moddown_ntt(c, levelQ, levelP, A, out0, out1, batch, st);
}

// DecomposeNTT (:459-483): decomp = [digit][batch?]... layout: decomp[digit] is a QP-stacked poly
// ([batch][nq+np][N] per digit, digit stride = batch * (nq+np) * N), digit rows included.
int decompose_ntt(const Ctx* c, int levelQ, int levelP, int nbPi, CSpan c2, bool c2IsNTT, u64* decomp, int batch, cudaStream_t st) {
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * nq * N, st)) return -1;
    Span other{buf.p, N, nq * N};
    CSpan ntt = c2, inv = c2;
    if (c2IsNTT) {
        if (launch_intt(c, rows_range(0, 0, (int)nq), c2, other, batch, NTT_CANONICAL, st)) return -1;
        inv = CSpan{other.p, N, nq * N};
    } else {
        if (launch_ntt(c, rows_range(0, 0, (int)nq), c2, other, batch, NTT_CANONICAL, st)) return -1;
        ntt = CSpan{other.p, N, nq * N};
    }
    const int nd = base_rns_decomposition_vector_size(levelQ, levelP);
    for (int i = 0; i < nd; i++) {
        u64* d = decomp + (size_t)i * batch * (nq + np) * N;
        Span dq{d, N, (nq + np) * N};
        Span dp{d + nq * N, N, (nq + np) * N};
        if (decompose_single_ntt(c, levelQ, levelP, nbPi, i, ntt, inv, dq, dp, true, batch, st)) return -1;
    }
    return 0;
}

// gadgetProductMultiplePLazyHoisted (:401-453): pure MAC over the pre-decomposed digits.
int gadget_product_hoisted_lazy(const Ctx* c, int levelQ, const u64* decomp, const GadgetCt& evk, const AccSpans& acc, int batch, cudaStream_t st,
                                int decomp_levelQ) {
    if (check_evk(c, levelQ, evk)) return -1;
    if (decomp_levelQ < 0) decomp_levelQ = levelQ;
    if (decomp_levelQ < levelQ) { set_error("the decomposition was computed at a lower level than levelQ"); return -1; }
    const size_t nqd = decomp_levelQ + 1;
    if (evk.pw2 != 0) { set_error("method is unsupported for BaseTwoDecomposition != 0"); return -1; }
    if (evk.levelP < 0) { set_error("hoisted gadget product requires a P ring"); return -1; }
    const int levelP = evk.levelP;
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    const int nd = base_rns_decomposition_vector_size(levelQ, levelP);
    for (int i = 0; i < nd; i++) {
        MacParams m;
        memset(&m, 0, sizeof(m));
        m.limbs = c->d_limbs; m.evk0 = evk.at(i, 0, 0, N); m.evk1 = evk.at(i, 0, 1, N); m.nQk = evk.levelQ + 1;
        m.xa = decomp + (size_t)i * batch * (nqd + np) * N; m.xa_rs = N; m.xa_bs = (nqd + np) * N; m.xa_pshift = (int)(nqd - nq);
        m.xb = nullptr; m.dlo = m.dhi = 0;
        for (int k = 0; k < 2; k++) { m.accQ[k] = acc.q[k].p; m.accP[k] = acc.p[k].p; }
        m.accQ_rs = acc.q[0].row_stride; m.accQ_bs = acc.q[0].batch_stride; m.accP_rs = acc.p[0].row_stride; m.accP_bs = acc.p[0].batch_stride;
        m.nq = (int)nq; m.np = (int)np; m.nQfull = c->nQ;
        m.first = (i == 0); m.last = (i == nd - 1); m.batch = batch; m.n = c->N;
        if (launch_mac(m, st)) return -1;
    }
    return 0;
}

int gadget_product_hoisted(const Ctx* c, int levelQ, const u64* decomp, const GadgetCt& evk, Span ct0, Span ct1, int batch, cudaStream_t st) {
    if (check_evk(c, levelQ, evk)) return -1;
    const int levelP = evk.levelP;
    const size_t N = c->N, nq = levelQ + 1, np = levelP + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * 2 * (nq + np) * N, st)) return -1;
    AccSpans acc;
    for (int k = 0; k < 2; k++) {
        u64* base = buf.p + (size_t)k * batch * (nq + np) * N;
        acc.q[k] = Span{base, N, (nq + np) * N};
        acc.p[k] = Span{base + nq * N, N, (nq + np) * N};
    }
    if (gadget_product_hoisted_lazy(c, levelQ, decomp, evk, acc, batch, st)) return -1;
    return evaluator_moddown_ntt(c, levelQ, levelP, acc, ct0, ct1, batch, st);
}

// Evaluator.Automorphism (core/rlwe/evaluator_automorphism.go:13-57), NTT-domain degree-1 ciphertexts:
//   tmp = GadgetProduct(ct[1], gk); tmp[0] += ct[0]; out[k] = AutomorphismNTT(tmp[k], galEl)
int evaluator_automorphism(const Ctx* c, int level, CSpan in0, CSpan in1, u64 galEl, const GadgetCt& gk, Span out0, Span out1,
                           const u64* decomp_hoisted, int batch, cudaStream_t st) {
    const size_t N = c->N, nq = level + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * 2 * nq * N + N, st)) return -1;
    Span t0{buf.p, N, nq * N}, t1{buf.p + (size_t)batch * nq * N, N, nq * N};
    u64* index = buf.p + (size_t)batch * 2 * nq * N;
    if (decomp_hoisted) { if (gadget_product_hoisted(c, level, decomp_hoisted, gk, t0, t1, batch, st)) return -1; }
    else { if (gadget_product(c, level, in1, gk, t0, t1, batch, st)) return -1; }
    if (launch_vecop(c, rows_range(0, 0, (int)nq), LGPU_OP_ADD, CSpan{t0.p, N, nq * N}, in0, t0, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    if (automorphism_ntt_index(c, galEl, index, st)) return -1;
    if (automorphism_ntt_with_index(c, (int)nq, CSpan{t0.p, N, nq * N}, index, out0, false, batch, st)) return -1;
    return automorphism_ntt_with_index(c, (int)nq, CSpan{t1.p, N, nq * N}, index, out1, false, batch, st);
}

// Evaluator.Relinearize (core/rlwe/evaluator_evaluationkey.go:121-148): out = (c0, c1) + GadgetProduct(c2, rlk)
int evaluator_relinearize(const Ctx* c, int level, CSpan c0, CSpan c1, CSpan c2, const GadgetCt& rlk, Span out0, Span out1, int batch, cudaStream_t st) {
    const size_t N = c->N, nq = level + 1;
    Scratch buf;
    if (buf.alloc((size_t)batch * 2 * nq * N, st)) return -1;
    Span t0{buf.p, N, nq * N}, t1{buf.p + (size_t)batch * nq * N, N, nq * N};
    if (gadget_product(c, level, c2, rlk, t0, t1, batch, st)) return -1;
    RowMap rm = rows_range(0, 0, (int)nq);
    if (launch_vecop(c, rm, LGPU_OP_ADD, c0, CSpan{t0.p, N, nq * N}, out0, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    return launch_vecop(c, rm, LGPU_OP_ADD, c1, CSpan{t1.p, N, nq * N}, out1, batch, nullptr, nullptr, 0, 0, c->N, st);
}

// ---------------------------------------------------------------------------------------------------------
// CKKS ct x ct multiply + relinearize (+ rescale)
// ---------------------------------------------------------------------------------------------------------
struct TensorParams {
    const LimbConst* limbs;
    const u64* a0; const u64* a1; const u64* b0; const u64* b1; size_t in_rs, in_bs;
    u64* d0; u64* d1; u64* d2; size_t out_rs, out_bs;
    int n;
};
// schemes/ckks/evaluator.go:807-820: c00 = MForm(a0), c01 = MForm(a1);
//   d0 = MRed(c00, b0); d2 = MRed(c01, b1); d1 = MRed(c00, b1) (+) MRed(c01, b0)  -- all canonical.
__global__ void __launch_bounds__(256) ckks_tensor_kernel(TensorParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i * 2 >= p.n) return;
    const LimbConst L = p.limbs[blockIdx.y];
    const u64 q = L.q, qinv = L.qinv;
    const size_t off = (size_t)blockIdx.z * p.in_bs + (size_t)blockIdx.y * p.in_rs;
    const size_t ooff = (size_t)blockIdx.z * p.out_bs + (size_t)blockIdx.y * p.out_rs;
    const ulonglong2 a0 = reinterpret_cast<const ulonglong2*>(p.a0 + off)[i];
    const ulonglong2 a1 = reinterpret_cast<const ulonglong2*>(p.a1 + off)[i];
    const ulonglong2 b0 = reinterpret_cast<const ulonglong2*>(p.b0 + off)[i];
    const ulonglong2 b1 = reinterpret_cast<const ulonglong2*>(p.b1 + off)[i];
    ulonglong2 d0, d1, d2;
    {
        const u64 m0 = mform(a0.x, q, L.bred_hi, L.bred_lo), m1 = mform(a1.x, q, L.bred_hi, L.bred_lo);
        d0.x = mred(m0, b0.x, q, qinv); d2.x = mred(m1, b1.x, q, qinv);
        d1.x = cred(mred(m0, b1.x, q, qinv) + mred(m1, b0.x, q, qinv), q);
    }
    {
        const u64 m0 = mform(a0.y, q, L.bred_hi, L.bred_lo), m1 = mform(a1.y, q, L.bred_hi, L.bred_lo);
        d0.y = mred(m0, b0.y, q, qinv); d2.y = mred(m1, b1.y, q, qinv);
        d1.y = cred(mred(m0, b1.y, q, qinv) + mred(m1, b0.y, q, qinv), q);
    }
    reinterpret_cast<ulonglong2*>(p.d0 + ooff)[i] = d0;
    reinterpret_cast<ulonglong2*>(p.d1 + ooff)[i] = d1;
    reinterpret_cast<ulonglong2*>(p.d2 + ooff)[i] = d2;
}

// ckks.Evaluator.MulRelinNew(ct0, ct1) [+ Rescale]: schemes/ckks/evaluator.go:719-872 and :477-515.
// ctA, ctB: [batch][2][level+1][N]; out: [batch][2][level+1-nbRescales][N].
static int ckks_mulrelin_rescale_chunk(const Ctx* c, int level, const u64* ctA, const u64* ctB, const GadgetCt& rlk, int nb_rescales,
                                       u64* out, int batch, cudaStream_t st);

// Sub-batches bound the key-switch scratch (P1 is 270 MB per ciphertext at L = 44: 17 GB for 64) while the evaluation key is streamed
// once per sub-batch. Measured at L = 44, batch 64 (profiles/README.md): 1 542 ct/s with sub-batches of 16, 1 573 with 32, 1 584 with 64.
// LGPU_BATCH_CHUNK overrides the default.
static int batch_chunk() {
    static int v = [] {
        const char* e = getenv("LGPU_BATCH_CHUNK");
        int x = e ? atoi(e) : 64;
        return x > 0 ? x : 64;
    }();
    return v;
}

int ckks_mulrelin_rescale(const Ctx* c, int level, const u64* ctA, const u64* ctB, const GadgetCt& rlk, int nb_rescales,
                          u64* out, int batch, cudaStream_t st) {
    if (level < 0 || level >= c->nQ) { set_error("level out of range"); return -1; }
    if (nb_rescales < 0 || nb_rescales > level) { set_error("cannot Rescale: input Ciphertext level is too low"); return -1; }
    const size_t N = c->N, nq = level + 1, nqo = nq - nb_rescales;
    const int ch = batch_chunk();
    for (int k = 0; k < batch; k += ch) {
        const int nb = batch - k < ch ? batch - k : ch;
        if (ckks_mulrelin_rescale_chunk(c, level, ctA + (size_t)k * 2 * nq * N, ctB + (size_t)k * 2 * nq * N, rlk, nb_rescales,
                                        out + (size_t)k * 2 * nqo * N, nb, st)) return -1;
    }
    return 0;
}

static int ckks_mulrelin_rescale_chunk(const Ctx* c, int level, const u64* ctA, const u64* ctB, const GadgetCt& rlk, int nb_rescales,
                                       u64* out, int batch, cudaStream_t st) {
    if (level < 0 || level >= c->nQ) { set_error("level out of range"); return -1; }
    if (nb_rescales < 0 || nb_rescales > level) { set_error("cannot Rescale: input Ciphertext level is too low"); return -1; }
    if (check_evk(c, level, rlk)) return -1;
    const size_t N = c->N, nq = level + 1;
    const size_t ct_stride = 2 * nq * N;
    Scratch buf;
    // d0,d1,d2 (3*nq) + t0,t1 (2*nq)
    if (buf.alloc((size_t)batch * 5 * nq * N, st)) return -1;
    u64* d0 = buf.p;
    u64* d1 = d0 + (size_t)batch * nq * N;
    u64* d2 = d1 + (size_t)batch * nq * N;
    u64* t0 = d2 + (size_t)batch * nq * N;
    u64* t1 = t0 + (size_t)batch * nq * N;
    {
        TensorParams p;
        p.limbs = c->d_limbs;
        p.a0 = ctA; p.a1 = ctA + nq * N; p.b0 = ctB; p.b1 = ctB + nq * N; p.in_rs = N; p.in_bs = ct_stride;
        p.d0 = d0; p.d1 = d1; p.d2 = d2; p.out_rs = N; p.out_bs = nq * N; p.n = c->N;
        ProfScope ps(LGPU_KCLASS_TENSOR, st, 8.0 * c->N * nq * batch * 7, 1);
        dim3 grid((c->N / 2 + 255) / 256, (unsigned)nq, batch);
        ckks_tensor_kernel<<<grid, 256, 0, st>>>(p);
        LGPU_CUDA_OK(cudaGetLastError());
    }
    if (rlk.levelP >= 1 && rlk.pw2 == 0 && fz_applicable(c, level, rlk.levelP) && (nb_rescales == 0 || (nb_rescales == 1 && level >= 1))) {
        // fused tail: accumulators -> (ModDown + add of d0/d1) in one chunk-pass epilogue -> fused rescale
        const size_t np = rlk.levelP + 1;
        Scratch accb;
        if (accb.alloc((size_t)2 * batch * (nq + np) * N, st)) return -1;
        AccSpans acc;
        for (int k = 0; k < 2; k++) {
            u64* base = accb.p + (size_t)k * batch * (nq + np) * N;
            acc.q[k] = Span{base, N, (nq + np) * N};
            acc.p[k] = Span{base + nq * N, N, (nq + np) * N};
        }
        if (gadget_product_lazy(c, level, CSpan{d2, N, nq * N}, rlk, acc, batch, st)) return -1;
        // LGPU_FZ_RESCALE (default 1): ModDown and Rescale as one pass (one basis extension and one transform per output row, see
        // moddown_ntt_fused); 0 runs them as two passes through d0
        static const int fz_rescale = [] { const char* e = getenv("LGPU_FZ_RESCALE"); return e ? atoi(e) : 1; }();
        if (nb_rescales == 1 && fz_rescale)
            return moddown_ntt_fused(c, level, rlk.levelP, accb.p, (size_t)batch * (nq + np) * N, (nq + np) * N, d0, (size_t)batch * nq * N, nq * N,
                                     out, (nq - 1) * N, 2 * (nq - 1) * N, 2, batch, st, 1);
        // d0, d1 are consecutive [comp][batch][nq][N] blocks: out = d + ModDown(acc), in place
        if (moddown_ntt_fused(c, level, rlk.levelP, accb.p, (size_t)batch * (nq + np) * N, (nq + np) * N, d0, (size_t)batch * nq * N, nq * N,
                              d0, (size_t)batch * nq * N, nq * N, 2, batch, st)) return -1;
        if (nb_rescales == 1) {
            const size_t nqo = nq - 1;
            return div_round_last_ntt_fused(c, level, d0, (size_t)batch * nq * N, nq * N, out, nqo * N, 2 * nqo * N, 2, batch, st);
        }
        for (int k = 0; k < 2; k++)
            LGPU_CUDA_OK(cudaMemcpy2DAsync(out + (size_t)k * nq * N, ct_stride * 8, d0 + (size_t)k * batch * nq * N, nq * N * 8, nq * N * 8, batch,
                                           cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    if (gadget_product(c, level, CSpan{d2, N, nq * N}, rlk, Span{t0, N, nq * N}, Span{t1, N, nq * N}, batch, st)) return -1;
    RowMap rm = rows_range(0, 0, (int)nq);
    if (nb_rescales == 0) {
        if (launch_vecop(c, rm, LGPU_OP_ADD, CSpan{d0, N, nq * N}, CSpan{t0, N, nq * N}, Span{out, N, ct_stride}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
        return launch_vecop(c, rm, LGPU_OP_ADD, CSpan{d1, N, nq * N}, CSpan{t1, N, nq * N}, Span{out + nq * N, N, ct_stride}, batch, nullptr, nullptr, 0, 0, c->N, st);
    }
    if (launch_vecop(c, rm, LGPU_OP_ADD, CSpan{d0, N, nq * N}, CSpan{t0, N, nq * N}, Span{d0, N, nq * N}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    if (launch_vecop(c, rm, LGPU_OP_ADD, CSpan{d1, N, nq * N}, CSpan{t1, N, nq * N}, Span{d1, N, nq * N}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    const size_t nqo = nq - nb_rescales;
    const size_t out_stride = 2 * nqo * N;
    if (div_by_last_modulus_many(c, LGPU_RING_Q, level, true, true, nb_rescales, CSpan{d0, N, nq * N}, Span{out, N, out_stride}, batch, st)) return -1;
    return div_by_last_modulus_many(c, LGPU_RING_Q, level, true, true, nb_rescales, CSpan{d1, N, nq * N}, Span{out + nqo * N, N, out_stride}, batch, st);
}

}  // namespace lgpu
