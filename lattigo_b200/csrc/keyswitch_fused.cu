// keyswitch_fused.cu -- fused pipeline for gadgetProductMultiplePLazy (core/rlwe/evaluator_gadget_product.go:129-201),
// the dominant loop of every key-switch (relinearisation, rotations):
//
//     for each digit d:  DecomposeSingleNTT(d) -> MulCoeffsMontgomeryLazy[ThenAddLazy](evk[d], .) on Q and P
//
// Unfused this is, per digit and per ciphertext, a basis-extension pass (write l+k rows), a two-pass NTT (read/write
// them twice) and a MAC pass that reads them again and read-modify-writes 2(l+k) accumulator rows. Here:
//
//   K1 ks_prepare   once per ciphertext: y_i = MRed(x_i + half_i, (S/s_i)^-1) for every row and the float64 overflow
//                   count v of every digit (ring/basis_extension.go:504-548) -- the only part of the basis extension
//                   that is shared by all target limbs.
//   K2 ks_strided   one launch for all (digit, target limb): the per-target sum  sum_i y_i (S/s_i mod t) - v S - S/2
//                   is evaluated on the INTEGER pipes for the 16 coefficients a thread owns and fed straight into
//                   the first 4 NTT stages (FP64 pipe for primes < 2^46, Shoup integer butterflies otherwise); the
//                   extended polynomial never exists in memory.
//   K3 ks_chunk_mac one CTA per (ciphertext, limb, 4096-chunk) walks over ALL digits: remaining 12 NTT stages in
//                   shared memory, then the Montgomery MAC against evk[d] with the two accumulators resident in
//                   shared memory; each accumulator row is written once, canonical, instead of 2 x digits times.
//
// Only canonical values leave the pipeline (the accumulators after the reference's trailing Reduce are canonical,
// :179-200), so the arithmetic inside is free-form -- except the float64 `v`, which is computed exactly as the
// reference does, and the single-limb digit rule (:402-436), which is reproduced literally.
#include <cstring>
#include "../../include/lattigo_b200.h"
#include "composite.h"
#include "modarith.cuh"
#include "ntt_arith.cuh"

namespace lgpu {

constexpr int kMaxDigits = 32;

// The integer-pipe rows (primes >= 2^46: q0 and the special primes) and the FP64-pipe rows of one operation are
// independent chains that use different execution pipes, so they are issued on two streams and overlap on the SMs.
struct SideStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
static SideStream* side_stream(int device) {
    static thread_local SideStream ss[16];
    // Opt-in (LGPU_SIDE_STREAM=1): running the integer-row chain next to the FP64-row chain gains ~1 % when one stream
    // drives the GPU, but the shared side stream couples otherwise independent caller streams (the host-buffer
    // pipeline lost a third of its throughput to it), so the default keeps every chain on the caller's stream.
    static const int on = [] { const char* e = getenv("LGPU_SIDE_STREAM"); return e && atoi(e) ? 1 : 0; }();
    if (!on || device < 0 || device >= 16) return nullptr;
    SideStream& x = ss[device];
    if (!x.s) {
        if (cudaStreamCreateWithFlags(&x.s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        cudaEventCreateWithFlags(&x.fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&x.join, cudaEventDisableTiming);
    }
    return &x;
}
// Measured: evaluating the basis extension on the FP64 pipe (fp_src == 2) makes K2 ~25 % slower than the 128-bit integer
// MAC, because the FP64 pipe then carries both the extension and the butterflies while the integer pipes idle.
// Kept selectable for experiments (LGPU_K2_FPSUM=1).
// LGPU_K2_SPLIT (default 1; 0 = the 128-bit Montgomery form everywhere): 23-bit-halves basis extension (ks_ext_split) on the FP64 target rows of
// digits whose sources are all FP64-pipe primes. Measured on the headline step: K2 class 55.6 -> 52.2 ms per 4 steps (profiles/r02_ab_late.txt)
static int k2_split() {
    static const int v = [] { const char* e = getenv("LGPU_K2_SPLIT"); return e ? atoi(e) : 1; }();
    return v;
}
static int k2_fpsum() {
    static const int on = [] { const char* e = getenv("LGPU_K2_FPSUM"); return e && atoi(e) ? 1 : 0; }();
    return on;
}
// returns the stream for the integer chain (forked from `st`), or `st` itself when side streams are unavailable
static cudaStream_t fork_side(const Ctx* c, cudaStream_t st, bool have_both) {
    if (!have_both || profiling_on()) return st;
    SideStream* ss = side_stream(c->device);
    if (!ss) return st;
    cudaEventRecord(ss->fork, st);
    cudaStreamWaitEvent(ss->s, ss->fork, 0);
    return ss->s;
}
static void join_side(const Ctx* c, cudaStream_t st, cudaStream_t side) {
    if (side == st) return;
    SideStream* ss = side_stream(c->device);
    cudaEventRecord(ss->join, side);
    cudaStreamWaitEvent(st, ss->join, 0);
}

// ------------------------------------------------------------------------------------------------------------
// K1
// ------------------------------------------------------------------------------------------------------------
struct KsPrepParams {
    const LimbConst* limbs;
    const u64* cx; size_t cx_rs, cx_bs;
    u64* Y; size_t y_bs;
    unsigned char* V; size_t v_bs;
    int nq, nd, k, n;
    int limb0;        // global limb index of source row 0 (0 for Q sources, nQ for P sources)
    int single_rule;  // 1: one-limb digits follow Decomposer's rule (raw coefficient, :402-436); 0: always ModUpExact
    u64 half_src[64];
    u64 cinv[64];
};
__global__ void __launch_bounds__(256) ks_prepare_kernel(KsPrepParams p) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= p.n) return;
    const int b = blockIdx.y;
    const u64* src = p.cx + (size_t)b * p.cx_bs + x;
    u64* Y = p.Y + (size_t)b * p.y_bs + x;
    unsigned char* V = p.V + (size_t)b * p.v_bs + x;
    for (int d = 0; d < p.nd; d++) {
        const int r0 = d * p.k;
        const int r1 = min(r0 + p.k, p.nq);
        if (r1 - r0 == 1 && p.single_rule) {   // single-limb digit: the raw coefficient is consumed by K2 (:402-436)
            Y[(size_t)r0 * p.n] = src[(size_t)r0 * p.cx_rs];
            V[(size_t)d * p.n] = 0;
            continue;
        }
        double vi = 0.0;
        for (int i = r0; i < r1; i++) {
            const LimbConst& L = p.limbs[p.limb0 + i];
            const u64 yi = mred(src[(size_t)i * p.cx_rs] + p.half_src[i], p.cinv[i], L.q, L.qinv);
            Y[(size_t)i * p.n] = yi;
            vi = __dadd_rn(vi, __ddiv_rn(__ull2double_rn(yi), __ull2double_rn(L.q)));
        }
        V[(size_t)d * p.n] = (unsigned char)__double2ull_rz(vi);
    }
}

// ------------------------------------------------------------------------------------------------------------
// K2
// ------------------------------------------------------------------------------------------------------------
struct KsDigit {
    unsigned int off_c, off_vt, off_half_t;   // blob offsets (words) of qoverqimodp / vtimesqmodp / half_t for this digit
    unsigned int off_cp;                      // plain (non-Montgomery) qoverqimodp, for the FP64 evaluation
    unsigned short ldc, nS;
    unsigned short fp_src;                    // 1: every source prime of the digit is below 2^46 (y_i exact in doubles)
};
struct KsStridedParams {
    const LimbConst* limbs;
    const u64* blob;
    RowMap rm;                      // launch row -> (global limb, row in the QP-stacked buffers)
    const u64* Y; size_t y_bs;
    const unsigned char* V; size_t v_bs;
    u64* P1; size_t p1_ds, p1_bs;   // [batch][digit][nq+np][N]
    int logN, nq, k, nd;
    int skip_own;     // 1: rows that belong to the digit itself are skipped (key-switch); 0: every launch row is a target
    int single_rule;  // see KsPrepParams
    int src_limb0;    // global limb of source row 0 (single-limb rule only)
    int split23;      // 1: full digits whose sources are all FP64-pipe primes take ks_ext_split on the FP64 target rows (LGPU_K2_SPLIT)
    // PRO_BCAST (rescale): e = cred(bc[x] + bc_add, bc_q) + s0[launch row]; PRO_MODUP_BCAST adds the same term to the extension
    const u64* bc; size_t bc_bs; u64 bc_add, bc_q;
    u64 s0[kMaxRows];
    KsDigit dg[kMaxDigits];
};

// ext value of one coefficient for target limb (q, qinv): reference formula of multSum + centring, reduced to < 3q.
// BC: plus a broadcast term bc < 2q, canonical (r + q - half_t < 4q, so the sum is below 6q < 8q, q < 2^61).
template <int NSMAX, bool BC = false>
__device__ __forceinline__ u64 ks_ext(const u64 (&y)[NSMAX], int nS, int v, const u64* c, const u64* vt, u64 half_t, u64 q, u64 qinv,
                                      u64 bc = 0) {
    // 128-bit accumulation through one __int128 so that the partial products chain on IMAD.WIDE / IADD3.X carries
    unsigned __int128 acc = 0;
#pragma unroll
    for (int i = 0; i < NSMAX; i++)
        if (i < nS) acc += (unsigned __int128)y[i] * c[i];
    const u64 rlo = (u64)acc, rhi = (u64)(acc >> 64);
    const u64 hhi = mulhi64(rlo * qinv, q);
    u64 r = rhi - hhi + q + vt[v];
    if (BC) return csub_lt8q(r + q - half_t + bc, q);
    return cred(r + q - half_t, q);
}

// The Rescale broadcast term of PRO_BCAST, (c_L + floor(q_L/2) mod q_L) + (q - floor(q_L/2) mod q) < q_L + q, brought below 2q for the
// merged prologue: reduced when the last modulus is above the target prime, where q_L + q could exceed the 8q the integer butterflies accept
__device__ __forceinline__ u64 bcast_lt2q(u64 c, u64 bc_add, u64 bc_q, u64 s0, u64 q, u64 bred_hi) {
    const u64 e = cred(c + bc_add, bc_q) + s0;
    return bc_q > q ? bred_add(e, q, bred_hi) : e;
}

// The same residue when every source prime of the digit AND the target prime are FP64-pipe primes (below 2^46.3), as a lazy double in
// (-0.66q, 0.66q) for the FP64 butterflies that follow. With 23-bit halves y = y0 + y1 2^23, c = c0 + c1 2^23 and c' = c 2^23 mod q = d0 + d1 2^23:
//   sum_i y_i c_i  ==  A + B 2^23 (mod q),   A = sum_i (y0 c0 + y1 d0),   B = sum_i (y0 c1 + y1 d1),
// every partial product is below 2^48 and both sums over up to 6 sources stay below 2^51, so the 4 products per source are 32 x 32 -> 64 bit
// multiply-adds without carry chains, and the reduction  A + (B 2^23 mod q) + (vt[v] - half_t)  takes 9 FP64 instructions (B 2^23 < 2^74 is an
// exact double, so one fp_reduce brings it below q/2; the 2^52 biases of the integer -> double conversions are folded into the constants)
// instead of a 128-bit Montgomery step plus 64-bit additions on the ALU pipe. `y` holds the two halves of a source word in its 32-bit halves
// (packed when the tile is staged); c (plain, not Montgomery: KsDigit::off_cp) and c' are split the same way. vtb = vt[v] - half_t - 2^52.
__device__ __forceinline__ u64 mad_wide(u32 a, u32 b, u64 c) {
    u64 r;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(a), "r"(b), "l"(c));
    return r;
}
// BC: plus a broadcast term 0 <= bc < 2q < 2^48 before the last reduction; the sum stays an exact integer below 2^52 (A < 2^51,
// |vt - half_t| < q, |t| < 0.66q, see above), so the result keeps the (-0.66q, 0.66q) range.
template <int NSMAX, bool BC = false>
__device__ __forceinline__ double ks_ext_split(const u64 (&y)[NSMAX], const u32 (&c0)[NSMAX], const u32 (&c1)[NSMAX], const u32 (&d0)[NSMAX],
                                               const u32 (&d1)[NSMAX], double vtb, double fq, double fqinv, double bc = 0.0) {
    u64 A = 0, B = 0;
#pragma unroll
    for (int i = 0; i < NSMAX; i++) {
        const u32 y0 = (u32)y[i], y1 = (u32)(y[i] >> 32);
        A = mad_wide(y0, c0[i], A);
        A = mad_wide(y1, d0[i], A);
        B = mad_wide(y0, c1[i], B);
        B = mad_wide(y1, d1[i], B);
    }
    const double ab = __longlong_as_double((long long)(A | 0x4330000000000000ull));                 // 2^52 + A
    const double bb = __longlong_as_double((long long)(B | 0x4330000000000000ull));                 // 2^52 + B
    const double t = fp_reduce(__fma_rn(bb, 8388608.0, -37778931862957161709568.0), fq, fqinv);     // (2^52 + B) 2^23 - 2^75 = B 2^23, exact
    if (BC) return fp_reduce(__dadd_rn(__dadd_rn(__dadd_rn(ab, vtb), t), bc), fq, fqinv);
    return fp_reduce(__dadd_rn(__dadd_rn(ab, vtb), t), fq, fqinv);                                  // (2^52 + A) + (vt - half_t - 2^52), exact
}

// K2 prologues: PRO_MODUP the basis extension, PRO_BCAST the Rescale broadcast of the last row, PRO_MODUP_BCAST their sum (the merged
// ModDown + Rescale tail: P^-1 ModUp with the constants of Ctx::muc_PtoQ_pinv, plus bcast_lt2q; canonical, see ks_ext)
enum { PRO_MODUP = 0, PRO_BCAST = 1, PRO_MODUP_BCAST = 2 };
#ifndef KS_STRIDED_MINB
#define KS_STRIDED_MINB 5
#endif
#ifndef KS_STRIDED_J4_MINB
#define KS_STRIDED_J4_MINB 4
#endif
#ifndef KS_FULL
#define KS_FULL 1
#endif
#ifndef KS_STREAM
#define KS_STREAM 0   // (measured: no gain) P1 tiles and key rows are read once per CTA: streaming loads keep the twiddles in L1
#endif
#ifndef KS_L2_PREFETCH
#define KS_L2_PREFETCH 1
#endif
#ifndef KS_J
#define KS_J 8   // target rows sharing one staged y/v tile
#endif

template <int RL, int NSMAX, bool FP, int PRO, bool CORR = true>
__global__ void __launch_bounds__(256, KS_STRIDED_MINB) ks_strided_kernel(KsStridedParams p) {
    constexpr int R = 1 << RL;
    __shared__ u64 s_c[NSMAX];
    __shared__ u64 s_vt[NSMAX + 1];
    const int limb = p.rm.limb[blockIdx.y];
    const int row = p.rm.drow[blockIdx.y];
    const int d = blockIdx.z % p.nd, b = blockIdx.z / p.nd;
    const KsDigit dg = p.dg[d];
    const int r0 = d * p.k;
    const int nS = dg.nS;
    if (PRO != PRO_BCAST && p.skip_own && row < p.nq && row >= r0 && row < r0 + nS) return;   // own rows come from the NTT input
    const LimbConst L = p.limbs[limb];
    const bool fpsum = FP && PRO == PRO_MODUP && dg.fp_src == 2 && (nS > 1 || !p.single_rule);
    if (PRO != PRO_BCAST) {
        if (threadIdx.x < nS) s_c[threadIdx.x] = p.blob[(fpsum ? dg.off_cp : dg.off_c) + (size_t)limb * dg.ldc + threadIdx.x];
        if (threadIdx.x <= nS) s_vt[threadIdx.x] = p.blob[dg.off_vt + (size_t)limb * (dg.ldc + 1) + threadIdx.x];
    }
    __syncthreads();
    // the strided pass always covers logN - 12 = RL stages, so N and the element stride are compile-time constants:
    // every load/store below addresses base + immediate (no per-access address arithmetic on the ALU pipe)
#ifdef KS_RUNTIME_STRIDE
    const int N = 1 << p.logN;
    const int stride = N >> RL;
#else
    constexpr int N = 4096 << RL;
    constexpr int stride = 4096;
#endif
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= stride) return;
    const u64 q = L.q, qinv = L.qinv;
    u64* out = p.P1 + (size_t)b * p.p1_bs + (size_t)d * p.p1_ds + (size_t)row * N;
    if constexpr (FP && PRO == PRO_MODUP) {
        if (fpsum) {
            // FP64 evaluation of the basis extension (targets and sources below 2^46): 5 FP64 operations per product
            // instead of a 128-bit integer MAC; any representative of the value is fine here, v is the exact one from K1.
            const double fq = L.fq, fqinv = L.fqinv;
            const double* tw = L.ftw_fwd;
            const u64* Y = p.Y + (size_t)b * p.y_bs + (size_t)r0 * N;
            const unsigned char* V = p.V + (size_t)b * p.v_bs + (size_t)d * N;
            const double halfd = (double)p.blob[dg.off_half_t + limb];
            double cj[NSMAX];
#pragma unroll
            for (int i = 0; i < NSMAX; i++) cj[i] = i < nS ? (double)s_c[i] : 0.0;
            double x[R];
#pragma unroll
            for (int k = 0; k < R; k++) {
                const int xi = k * stride + l;
                double acc = __dadd_rn((double)s_vt[V[xi]], -halfd);
#pragma unroll
                for (int i = 0; i < NSMAX; i++)
                    if (i < nS) acc = __dadd_rn(acc, fp_mulmod(u2d(Y[(size_t)i * N + xi]), cj[i], fq, fqinv));
                x[k] = acc;
            }
#pragma unroll
            for (int u = 0; u < RL; u++) {
                const int half = 1 << (RL - 1 - u);
#pragma unroll
                for (int k = 0; k < R; k++) {
                    if (k & half) continue;
                    fp_fwd_bfly(x[k], x[k + half], __ldg(tw + (1 << u) + (k >> (RL - u))), fq, fqinv);
                }
            }
#pragma unroll
            for (int k = 0; k < R; k++) out[(size_t)k * stride + l] = (u64)__double_as_longlong(x[k]);
            return;
        }
    }
    u64 e[R];
    if constexpr (PRO == PRO_BCAST) {
        const u64* bc = p.bc + (size_t)b * p.bc_bs;
        const u64 s0 = p.s0[blockIdx.y];
#pragma unroll
        for (int k = 0; k < R; k++) e[k] = cred(bc[k * stride + l] + p.bc_add, p.bc_q) + s0;
        // a wide last modulus under a narrow row (mixed 40 / 60-bit chains): bring the value into the range the butterflies
        // assume (< 2^52 for the FP64 rows, < 8q for the integer ones); only its residue matters
        if (p.bc_q >> 50) {
#pragma unroll
            for (int k = 0; k < R; k++) e[k] = bred_add(e[k], q, L.bred_hi);
        }
    } else {
    constexpr bool BC = PRO == PRO_MODUP_BCAST;
    const bool multi = nS > 1 || !p.single_rule;
    const u64 half_t = multi ? p.blob[dg.off_half_t + limb] : 0;
    const u64* Y = p.Y + (size_t)b * p.y_bs + (size_t)r0 * N;
    const unsigned char* V = p.V + (size_t)b * p.v_bs + (size_t)d * N;
    const u64* bc = BC ? p.bc + (size_t)b * p.bc_bs : nullptr;
    const u64 s0 = BC ? p.s0[blockIdx.y] : 0;
    if (multi) {
#pragma unroll
        for (int k = 0; k < R; k++) {
            const int x = k * stride + l;
            u64 y[NSMAX];
#pragma unroll
            for (int i = 0; i < NSMAX; i++) y[i] = i < nS ? Y[(size_t)i * N + x] : 0;
            const u64 t = BC ? bcast_lt2q(bc[x], p.bc_add, p.bc_q, s0, q, L.bred_hi) : 0;
            e[k] = ks_ext<NSMAX, BC>(y, nS, (int)V[x], s_c, s_vt, half_t, q, qinv, t);
        }
    } else {
        // single-limb digit (ring/basis_extension.go:402-436): centre around q_src/2, reduce, restore the sign
        const u64 qs = p.limbs[p.src_limb0 + r0].q;
#pragma unroll
        for (int k = 0; k < R; k++) {
            u64 c = Y[k * stride + l];
            const bool neg = c >= (qs >> 1);
            if (neg) c = qs - c;
            const u64 t = bred_add(c, q, L.bred_hi);
            e[k] = neg ? q - t : t;
            if (BC) e[k] += bcast_lt2q(bc[k * stride + l], p.bc_add, p.bc_q, s0, q, L.bred_hi);     // < 3q
        }
    }
    }
    if constexpr (FP) {
        const double fq = L.fq, fqinv = L.fqinv;
        const double* tw = L.ftw_fwd;
        double x[R];
#pragma unroll
        for (int k = 0; k < R; k++) x[k] = u2d(e[k]);
#pragma unroll
        for (int u = 0; u < RL; u++) {
            const int half = 1 << (RL - 1 - u);
#pragma unroll
            for (int k = 0; k < R; k++) {
                if (k & half) continue;
                fp_fwd_bfly(x[k], x[k + half], __ldg(tw + (1 << u) + (k >> (RL - u))), fq, fqinv);
            }
        }
#pragma unroll
        for (int k = 0; k < R; k++) out[(size_t)k * stride + l] = (u64)__double_as_longlong(x[k]);
    } else {
        const ulonglong2* tw = L.tw_fwd;
        const u64 nq = 0ull - q, twoq = q << 1, kq = L.kq;
        const unsigned mask = L.fwd_mask;     // per-prime lazy-correction schedule (0 below 2^57; every stage for 61-bit primes)
#pragma unroll
        for (int u = 0; u < RL; u++) {
            const int half = 1 << (RL - 1 - u);
            const bool corr = CORR && ((mask >> u) & 1u);
#pragma unroll
            for (int k = 0; k < R; k++) {
                if (k & half) continue;
                fast_fwd_bfly(e[k], e[k + half], __ldg(tw + (1 << u) + (k >> (RL - u))), nq, twoq, kq, corr);
            }
        }
#pragma unroll
        for (int k = 0; k < R; k++) out[(size_t)k * stride + l] = e[k];
    }
}

// ------------------------------------------------------------------------------------------------------------
// K2, row-sharing variant. The plain kernel reads the digit's y_i (nS x 8 B) + v (1 B) once per TARGET ROW, i.e.
// ~33 B from L2 per 8 B written: 73 GB of L2->SM traffic per 64-ciphertext step at L=44, which is what bounds it.
// Here a CTA owns 64 strided columns (l) x all R strided coefficients and stages that y/v tile in shared memory once
// for J = 4 target rows (thread = (column, target row)): L2 traffic drops 4x, the y reads become conflict-free /
// broadcast shared-memory loads. Multi-source digits only (the single-limb rule keeps the plain kernel).
// BC: prologue PRO_MODUP_BCAST (one digit: the ModDown extension, plus the Rescale broadcast term of the column).
// ------------------------------------------------------------------------------------------------------------
template <int RL, int NSMAX, bool FP, bool CORR = true, bool BC = false>
__global__ void __launch_bounds__(256, KS_STRIDED_J4_MINB) ks_strided_j4_kernel(KsStridedParams p) {
    constexpr int R = 1 << RL, J = KS_J, LB = 256 / J;
    extern __shared__ u64 dsm[];
    u64* s_y = dsm;                                                        // [NSMAX][R][LB]
    unsigned char* s_v = reinterpret_cast<unsigned char*>(dsm + NSMAX * R * LB);   // [R][LB]
    // BC: this thread's broadcast terms [R][256], formed before the extension so that their operands are not live across it (with them
    // live the R = 16 instantiations spill several times more than without)
    u64* s_bt = dsm + NSMAX * R * LB + R * LB / 8;
    __shared__ u64 s_c[J][NSMAX];
    __shared__ u64 s_vt[J][NSMAX + 1];
    __shared__ u64 s_c2[FP ? J : 1][NSMAX];              // split path: c 2^23 mod q
    __shared__ double s_vtd[FP ? J : 1][NSMAX + 1];      // split path: vt[v] - half_t - 2^52
    const int tid = threadIdx.x, lx = tid % LB, jj = tid / LB;
    const int jrow = blockIdx.y * J + jj;
    const bool valid = jrow < p.rm.nrows;
    const int limb = valid ? p.rm.limb[jrow] : 0;
    const int row = valid ? p.rm.drow[jrow] : 0;
    const int d = blockIdx.z % p.nd, b = blockIdx.z / p.nd;
    const KsDigit dg = p.dg[d];
    const int r0 = d * p.k;
    const int nS = dg.nS;
    constexpr int N = 4096 << RL;
    constexpr int stride = 4096;
    const int l0 = blockIdx.x * LB;
    const u64* Y = p.Y + (size_t)b * p.y_bs + (size_t)r0 * N;
    const unsigned char* V = p.V + (size_t)b * p.v_bs + (size_t)d * N;
    const bool split = FP && p.split23 && dg.fp_src != 0 && nS == NSMAX;      // CTA-uniform
    for (int idx = tid; idx < nS * R * LB; idx += 256) {
        const int i = idx / (R * LB), k = (idx / LB) % R, x = idx % LB;
        u64 w = Y[(size_t)i * N + k * stride + l0 + x];
        if (split) w = (w & 0x7FFFFFull) | ((w >> 23) << 32);                  // 23-bit halves for ks_ext_split (w < 2^46.3)
        s_y[idx] = w;
    }
    for (int idx = tid; idx < R * LB / 4; idx += 256) {      // 4 bytes per thread: 16-column groups are 4-byte aligned
        const int k = (idx * 4) / LB, x = (idx * 4) % LB;
        reinterpret_cast<unsigned int*>(s_v)[idx] = *reinterpret_cast<const unsigned int*>(V + k * stride + l0 + x);
    }
    if (valid) {
        if (split) {
            // plain constants c, c' = c 2^23 mod q and the double table vt[v] - half_t of this target row
            const double fq = p.limbs[limb].fq, fqinv = p.limbs[limb].fqinv;
            if (lx < nS) {
                const u64 cp = p.blob[dg.off_cp + (size_t)limb * dg.ldc + lx];
                const double w = u2d(fp_canon(8388608.0, fq, fqinv));
                s_c[jj][lx] = cp;
                s_c2[jj][lx] = fp_canon(fp_mulmod(u2d(cp), w, fq, fqinv), fq, fqinv);
            }
            if (lx <= nS)
                s_vtd[jj][lx] = __dadd_rn(__dadd_rn(u2d(p.blob[dg.off_vt + (size_t)limb * (dg.ldc + 1) + lx]), -u2d(p.blob[dg.off_half_t + limb])), -FP_TWO52);
        } else {
            if (lx < nS) s_c[jj][lx] = p.blob[dg.off_c + (size_t)limb * dg.ldc + lx];
            if (lx <= nS) s_vt[jj][lx] = p.blob[dg.off_vt + (size_t)limb * (dg.ldc + 1) + lx];
        }
        if (BC) {
            const u64* bc = p.bc + (size_t)b * p.bc_bs + l0 + lx;
            const u64 q = p.limbs[limb].q, bh = p.limbs[limb].bred_hi, s0 = p.s0[jrow];
#pragma unroll
            for (int k = 0; k < R; k++) s_bt[k * 256 + tid] = bcast_lt2q(bc[k * stride], p.bc_add, p.bc_q, s0, q, bh);
        }
    }
    __syncthreads();
    if (!valid) return;
    if (p.skip_own && row < p.nq && row >= r0 && row < r0 + nS) return;   // own rows come from the NTT input
    const LimbConst L = p.limbs[limb];
    const u64 q = L.q, qinv = L.qinv;
    const u64 half_t = p.blob[dg.off_half_t + limb];
    const int l = l0 + lx;
    u64* out = p.P1 + (size_t)b * p.p1_bs + (size_t)d * p.p1_ds + (size_t)row * N + l;
    u64 e[R];
    if constexpr (FP) {
        if (split) {
            const double fq = L.fq, fqinv = L.fqinv;
            const double* tw = L.ftw_fwd;
            u32 c0[NSMAX], c1[NSMAX], d0[NSMAX], d1[NSMAX];
#pragma unroll
            for (int i = 0; i < NSMAX; i++) {
                const u64 cw = s_c[jj][i], dw = s_c2[jj][i];
                c0[i] = (u32)cw & 0x7FFFFFu; c1[i] = (u32)(cw >> 23);
                d0[i] = (u32)dw & 0x7FFFFFu; d1[i] = (u32)(dw >> 23);
            }
            double x[R];
#pragma unroll
            for (int k = 0; k < R; k++) {
                u64 y[NSMAX];
#pragma unroll
                for (int i = 0; i < NSMAX; i++) y[i] = s_y[(i * R + k) * LB + lx];
                const double t = BC ? u2d(s_bt[k * 256 + tid]) : 0.0;
                x[k] = ks_ext_split<NSMAX, BC>(y, c0, c1, d0, d1, s_vtd[jj][s_v[k * LB + lx]], fq, fqinv, t);
            }
#pragma unroll
            for (int u = 0; u < RL; u++) {
                const int half = 1 << (RL - 1 - u);
#pragma unroll
                for (int k = 0; k < R; k++) {
                    if (k & half) continue;
                    fp_fwd_bfly(x[k], x[k + half], __ldg(tw + (1 << u) + (k >> (RL - u))), fq, fqinv);
                }
            }
#pragma unroll
            for (int k = 0; k < R; k++) out[(size_t)k * stride] = (u64)__double_as_longlong(x[k]);
            return;
        }
    }
    if (KS_FULL && nS == NSMAX) {          // full digit (every digit but possibly the last): no per-source predication
#pragma unroll
        for (int k = 0; k < R; k++) {
            u64 y[NSMAX];
#pragma unroll
            for (int i = 0; i < NSMAX; i++) y[i] = s_y[(i * R + k) * LB + lx];
            const u64 t = BC ? s_bt[k * 256 + tid] : 0;
            e[k] = ks_ext<NSMAX, BC>(y, NSMAX, (int)s_v[k * LB + lx], s_c[jj], s_vt[jj], half_t, q, qinv, t);
        }
    } else {
#pragma unroll
        for (int k = 0; k < R; k++) {
            u64 y[NSMAX];
#pragma unroll
            for (int i = 0; i < NSMAX; i++) y[i] = i < nS ? s_y[(i * R + k) * LB + lx] : 0;
            const u64 t = BC ? s_bt[k * 256 + tid] : 0;
            e[k] = ks_ext<NSMAX, BC>(y, nS, (int)s_v[k * LB + lx], s_c[jj], s_vt[jj], half_t, q, qinv, t);
        }
    }
    if constexpr (FP) {
        const double fq = L.fq, fqinv = L.fqinv;
        const double* tw = L.ftw_fwd;
        double x[R];
#pragma unroll
        for (int k = 0; k < R; k++) x[k] = u2d(e[k]);
#pragma unroll
        for (int u = 0; u < RL; u++) {
            const int half = 1 << (RL - 1 - u);
#pragma unroll
            for (int k = 0; k < R; k++) {
                if (k & half) continue;
                fp_fwd_bfly(x[k], x[k + half], __ldg(tw + (1 << u) + (k >> (RL - u))), fq, fqinv);
            }
        }
#pragma unroll
        for (int k = 0; k < R; k++) out[(size_t)k * stride] = (u64)__double_as_longlong(x[k]);
    } else {
        const ulonglong2* tw = L.tw_fwd;
        const u64 nq = 0ull - q, twoq = q << 1, kq = L.kq;
        const unsigned mask = L.fwd_mask;     // per-prime lazy-correction schedule (0 below 2^57; every stage for 61-bit primes)
#pragma unroll
        for (int u = 0; u < RL; u++) {
            const int half = 1 << (RL - 1 - u);
            const bool corr = CORR && ((mask >> u) & 1u);
#pragma unroll
            for (int k = 0; k < R; k++) {
                if (k & half) continue;
                fast_fwd_bfly(e[k], e[k + half], __ldg(tw + (1 << u) + (k >> (RL - u))), nq, twoq, kq, corr);
            }
        }
#pragma unroll
        for (int k = 0; k < R; k++) out[(size_t)k * stride] = e[k];
    }
}

// ------------------------------------------------------------------------------------------------------------
// K3
// ------------------------------------------------------------------------------------------------------------
struct KsChunkParams {
    const LimbConst* limbs;
    RowMap rm;
    const u64* P1; size_t p1_ds, p1_bs;
    const u64* cx; size_t cx_rs, cx_bs;     // NTT-domain input (the digit's own rows)
    const u64* evk; size_t evk_ds, evk_cs;  // digit stride, component stride (words); row r of the key at r_key * N
    int nQk;                                // Q rows in the key
    u64* acc; size_t acc_cs, acc_bs;        // [batch][2][nq+np][N]
    int logN, nq, k, nd;
    int wide;                               // 1: key / own rows are 32-byte aligned -> 256-bit loads in the register-MAC kernels (LGPU_K3_WIDE)
};

template <bool FP>
__global__ void __launch_bounds__(256, 2) ks_chunk_mac_kernel(KsChunkParams p) {
    constexpr int CL = 12, T = 256;
    extern __shared__ u64 smem[];
    u64* sm = smem;                         // (4096 + 256 + 1) words: transform buffer (padded)
    u64* a0 = smem + 4096 + 256 + 8;        // 4096 words
    u64* a1 = a0 + 4096;
    const int b = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
    const int limb = p.rm.limb[blockIdx.z];
    const int row = p.rm.drow[blockIdx.z];
    const LimbConst L = p.limbs[limb];
    const int s1 = p.logN - CL;
    const int N = 1 << p.logN;
    const u64 q = L.q, qinv = L.qinv, twoq = q << 1;
    const size_t erow = (size_t)(row < p.nq ? row : p.nQk + (row - p.nq)) * N + ((size_t)chunk << CL);
    const u64* P1row = p.P1 + (size_t)b * p.p1_bs + (size_t)row * N + ((size_t)chunk << CL);
    const u64* xin = p.cx + (size_t)b * p.cx_bs + (size_t)row * p.cx_rs + ((size_t)chunk << CL);
    // digits whose limbs contain this row contribute the NTT-domain input itself; at most one such digit exists
    const int own_d = row < p.nq ? row / p.k : -1;
    // software pipeline: the tile of the next digit is fetched into registers while the current one is transformed
    u64 raw[16];
    {
        const int d0 = own_d == 0 ? 1 : 0;
        if (d0 < p.nd) {
#pragma unroll
            for (int k = 0; k < 16; k++) raw[k] = P1row[(size_t)d0 * p.p1_ds + k * T + tid];
        }
    }
    for (int d = 0; d < p.nd; d++) {
        const bool own = d == own_d;
        const u64* e0 = p.evk + (size_t)d * p.evk_ds + erow;
        const u64* e1 = e0 + p.evk_cs;
        int dn = d + 1;
        if (dn == own_d) dn++;
        // first half of this thread's key words: requested before the last transform round so that the L2 latency
        // is covered by that round instead of stalling the MAC
        u64 k0[8], k1[8];
        if (!own) {
            if constexpr (FP) {
                double* fsm = reinterpret_cast<double*>(sm);
                const double fq = L.fq, fqinv = L.fqinv;
                const double* tw = L.ftw_fwd;
                {
                    double x[16];
#pragma unroll
                    for (int k = 0; k < 16; k++) x[k] = __longlong_as_double((long long)raw[k]);
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int half = 1 << (3 - u);
                        const int twbase = (1 << (s1 + u)) + (chunk << u);
#pragma unroll
                        for (int k = 0; k < 16; k++) {
                            if (k & half) continue;
                            fp_fwd_bfly(x[k], x[k + half], __ldg(tw + twbase + (k >> (4 - u))), fq, fqinv);
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 16; k++) fsm[fpad(k * T + tid)] = x[k];
                }
                double t2[15];
                fp_load_tw<CL, 4, 4>(t2, tw, s1, chunk, tid);
                __syncthreads();
                fp_fwd_round_tw<CL, 4, 4>(fsm, t2, fq, fqinv, tid);
                double t3[15];
                fp_load_tw<CL, 8, 4>(t3, tw, s1, chunk, tid);
#pragma unroll
                for (int j = 0; j < 8; j++) { k0[j] = __ldg(e0 + j * T + tid); k1[j] = __ldg(e1 + j * T + tid); }
                __syncthreads();
                fp_fwd_round_tw<CL, 8, 4>(fsm, t3, fq, fqinv, tid);
            } else {
                const ulonglong2* tw = L.tw_fwd;
                const u64 nq = 0ull - q;
                {
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int half = 1 << (3 - u);
                        const int twbase = (1 << (s1 + u)) + (chunk << u);
                        const bool corr = (L.fwd_mask >> (s1 + u)) & 1u;
#pragma unroll
                        for (int k = 0; k < 16; k++) {
                            if (k & half) continue;
                            fast_fwd_bfly(raw[k], raw[k + half], __ldg(tw + twbase + (k >> (4 - u))), nq, twoq, L.kq, corr);
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 16; k++) sm[pad_idx(k * T + tid)] = raw[k];
                }
                __syncthreads();
                fwd_round<CL, 4, 4, false, 1>(sm, nullptr, L, s1, p.logN, chunk, tid);
#pragma unroll
                for (int j = 0; j < 8; j++) { k0[j] = __ldg(e0 + j * T + tid); k1[j] = __ldg(e1 + j * T + tid); }
                __syncthreads();
                fwd_round<CL, 8, 4, false, 1>(sm, nullptr, L, s1, p.logN, chunk, tid);
            }
            __syncthreads();
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) { k0[j] = __ldg(e0 + j * T + tid); k1[j] = __ldg(e1 + j * T + tid); }
        }
        // the tile of the next digit travels while the MAC runs
        if (!own && dn < p.nd) {
#pragma unroll
            for (int k = 0; k < 16; k++) raw[k] = P1row[(size_t)dn * p.p1_ds + k * T + tid];
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            u64 n0[8], n1[8];
            if (h == 0) {   // second half of the key words, requested while the first half is consumed
#pragma unroll
                for (int j = 0; j < 8; j++) { n0[j] = __ldg(e0 + (8 + j) * T + tid); n1[j] = __ldg(e1 + (8 + j) * T + tid); }
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int idx = (h * 8 + j) * T + tid;
                u64 x;
                if (own) x = xin[idx];
                else if (FP) x = fp_canon(reinterpret_cast<double*>(sm)[fpad(idx)], L.fq, L.fqinv);
                else x = sm[pad_idx(idx)];
                const u64 m0 = mred_lazy(k0[j], x, q, qinv);
                const u64 m1 = mred_lazy(k1[j], x, q, qinv);
                if (d == 0) { a0[idx] = m0; a1[idx] = m1; }
                else {
                    u64 v0 = a0[idx] + m0, v1 = a1[idx] + m1;
                    a0[idx] = v0 >= twoq ? v0 - twoq : v0;
                    a1[idx] = v1 >= twoq ? v1 - twoq : v1;
                }
            }
            if (h == 0) {
#pragma unroll
                for (int j = 0; j < 8; j++) { k0[j] = n0[j]; k1[j] = n1[j]; }
            }
        }
        __syncthreads();
    }
    u64* o0 = p.acc + (size_t)b * p.acc_bs + (size_t)row * N + ((size_t)chunk << CL);
    u64* o1 = o0 + p.acc_cs;
#pragma unroll 4
    for (int kk = 0; kk < 16; kk++) {
        const int idx = kk * T + tid;
        const u64 v0 = a0[idx], v1 = a1[idx];
        o0[idx] = cred(v0 >= twoq ? v0 - twoq : v0, q);
        o1[idx] = cred(v1 >= twoq ? v1 - twoq : v1, q);
    }
}

// ------------------------------------------------------------------------------------------------------------
// K3, high-occupancy FP64 variant: 512 threads x 8 elements (four radix-8 rounds), <= 64 registers, 2 CTAs = 32 warps
// per SM. The FP64 butterfly only reaches its pipe rate (0.46 warp-instr/clk/SMSP, tools/ubench/fp64_operands.cu) with
// >= 4 warps per scheduler issuing it; the 256-thread variant leaves 2 warps per scheduler per CTA and half of them
// sit in the integer MAC phase or at a barrier.
// ------------------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------------------
// K3, register-MAC variant of the 512 x 8 kernel. The last radix-8 round leaves every thread with 8 CONSECUTIVE
// coefficients in registers (stages 9..11 act inside aligned groups of 8), so the MAC consumes them right there:
//   * no store / barrier / reload of the transformed tile before the MAC,
//   * key rows, own rows and results move as 128-bit accesses (64 contiguous bytes per thread),
//   * the accumulators of those 8 coefficients are private to the thread (shared memory is only their spill space,
//     laid out so that 128-bit accesses are conflict-free), hence the MAC phase has no barrier at all,
//   * the only ordering the next digit needs -- "everybody has read the tile before I overwrite it" -- is a split
//     mbarrier: arrive right after the last-round reads, wait just before the next digit's first-round stores.
// Warps therefore drift apart inside a CTA and the integer MAC of one warp overlaps the FP64 butterflies of another.
// ------------------------------------------------------------------------------------------------------------
// The integer consumers of a transformed coefficient (MRedLazy with a key word, the ModDown / Rescale MRed) accept ANY
// representative below 2^64, so the canonicalisation (3 FP64 + compare + add + conversion) is replaced by one biased
// conversion: |x| < (10 + logN) q < 2^51 (the fp_ok bound), hence x + (10 + logN) q lies in [0, 2^52) and
// bits(x + (10 + logN) q + 2^52) & (2^52 - 1) is that value as an integer.
#ifndef KS_LAZY_X
#define KS_LAZY_X 1
#endif
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u64 mbar_arrive(unsigned bar) {
    u64 tok;
    asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(tok) : "r"(bar) : "memory");
    return tok;
}
__device__ __forceinline__ void mbar_wait(unsigned bar, u64 tok) {
    unsigned done;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.test_wait.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "l"(tok) : "memory");
    } while (!done);
}
__device__ __forceinline__ ulonglong2 ldg128(const u64* p) {
    return KS_STREAM ? __ldcs(reinterpret_cast<const ulonglong2*>(p)) : __ldg(reinterpret_cast<const ulonglong2*>(p));
}
// 4 consecutive words in one request. Every thread of the register-MAC kernels reads its own 64 contiguous bytes of a key row, so a warp-wide load
// touches all 16 lines of a 2 KB span whatever its width: four 128-bit loads cost 4 x 16 tag look-ups in the L1 that bounds the kernel, two 256-bit
// loads 2 x 16 for the same bytes.
__device__ __forceinline__ void ldg256(const u64* p, u64& a, u64& b, u64& c, u64& d) {
    asm("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
}
// coherent forms for buffers the same kernel writes (the epilogue's operands may alias its output)
__device__ __forceinline__ void ld256(const u64* p, u64& a, u64& b, u64& c, u64& d) {
    asm volatile("ld.global.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void st256(u64* p, u64 a, u64 b, u64 c, u64 d) {
    asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" :: "l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

// MACV selects the pipe of the multiply-accumulate (LGPU_K3_VARIANT = 10 + MACV):
//   0  integer pipes: MRedLazy(key, x) with the biased-integer x, u64 sums, one Barrett step at the end;
//   1  FP64 pipe: acc += fp_mulmod(x, double(key)) with x left as the double the last round produced -- 8 FP64 instructions per term instead of
//      ~21 integer ones. The key is in Montgomery form (key * 2^64), so the sum carries a factor 2^64 that one fp_mulmod by 2^-64 mod q removes
//      per output coefficient; |acc| <= kMaxDigits * q < 2^52 stays an exact integer. Key / own-row words at or above 2^46 (never produced by the
//      reference: both are canonical residues) are Barrett-reduced first;
//   2  component 0 as in 1, component 1 as in 0 (both pipes busy in the MAC phase).
template <int MACV>
__global__ void __launch_bounds__(512, 2) ks_chunk_mac_fp8r_kernel(KsChunkParams p) {
    constexpr int CL = 12, T = 512;
    constexpr bool F0 = MACV >= 1, F1 = MACV == 1 || MACV == 3, R1 = MACV == 3;
    extern __shared__ u64 smem[];
    __shared__ __align__(8) u64 s_bar;
    double* fsm = reinterpret_cast<double*>(smem);
    // accumulators: component c, pair j (coefficients 8*tid + 2j, 2j+1) at acc + ((c*4 + j) * T + tid) * 2
    ulonglong2* accs = reinterpret_cast<ulonglong2*>(smem + 4096);       // the transform tile is XOR-swizzled, not padded
    double2* accd = reinterpret_cast<double2*>(smem + 4096);
    const int b = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
    const int limb = p.rm.limb[blockIdx.z];
    const int row = p.rm.drow[blockIdx.z];
    const LimbConst L = p.limbs[limb];
    const int s1 = p.logN - CL;
    const int N = 1 << p.logN;
    const u64 q = L.q, qinv = L.qinv;
    const double fq = L.fq, fqinv = L.fqinv;
    const double off52 = __dmul_rn((double)(10 + p.logN), fq) + 4503599627370496.0;   // (10 + logN) q + 2^52, exact
    const double* tw = L.ftw_fwd;
    const size_t erow = (size_t)(row < p.nq ? row : p.nQk + (row - p.nq)) * N + ((size_t)chunk << CL);
    const u64* P1row = p.P1 + (size_t)b * p.p1_bs + (size_t)row * N + ((size_t)chunk << CL);
    const u64* xin = p.cx + (size_t)b * p.cx_bs + (size_t)row * p.cx_rs + ((size_t)chunk << CL) + 8 * tid;
    const int own_d = row < p.nq ? row / p.k : -1;
    const unsigned bar = smem_addr(&s_bar);
    if (tid == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(T) : "memory");
    __syncthreads();
    u64 raw[8];
    u64 tok = 0;
    bool pending = false;      // a tile read phase is outstanding: wait for it before overwriting the tile
    double acc1[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};       // MACV == 3: component 1 accumulates in registers
    for (int d = 0; d < p.nd; d++) {
        const bool own = d == own_d;
        const u64* e0 = p.evk + (size_t)d * p.evk_ds + erow + 8 * tid;
        const u64* e1 = e0 + p.evk_cs;
        int dn = d + 1;
        if (dn == own_d) dn++;
        u64 xv[8];
        double xd[8];
        // the twiddle addresses are loop-invariant too; left alone the compiler hoists the 12 pointers out of the loop and spills them. Laundering the
        // base and the thread index makes it recompute them here (a few integer instructions on pipes that are idle) instead of reloading them from
        // local memory through the L1 that bounds this kernel
        const double* twl = tw;
        int tl = tid;
        asm volatile("" : "+l"(twl), "+r"(tl));
        if (!own) {
            {
                double x[8];
                {
#pragma unroll
                    for (int k = 0; k < 8; k++) raw[k] = KS_STREAM ? __ldcs(P1row + (size_t)d * p.p1_ds + k * T + tid) : P1row[(size_t)d * p.p1_ds + k * T + tid];
                    // pull the next digit's tile (32 KB = 256 lines) from HBM into L2 while this digit is processed
                    if (KS_L2_PREFETCH && dn < p.nd && tid < 256)
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(P1row + (size_t)dn * p.p1_ds + tid * 16));
                }
                {
                    double t1[7];
                    fp8_load_tw<0, true>(t1, twl, s1, chunk, tl);       // CTA-uniform: hi = 0
#pragma unroll
                    for (int k = 0; k < 8; k++) x[k] = __longlong_as_double((long long)raw[k]);
                    fp8_bflys(x, t1, fq, fqinv);
                }
                if (pending) { mbar_wait(bar, tok); pending = false; }
                fp8s_store_r1(fsm, x, tid);
            }
            double t[7];
            fp8_load_tw<3, true>(t, twl, s1, chunk, tl);
            __syncthreads();
            fp8s_round2(fsm, t, fq, fqinv, tid);
            fp8_load_tw<6, true>(t, twl, s1, chunk, tl);
            fp8s_pair_sync(tid);
            fp8s_round3(fsm, t, fq, fqinv, tid);
            fp8_load_tw<9, true>(t, twl, s1, chunk, tl);
            __syncwarp();
            {   // last round stays in registers: coefficients 8*tid .. 8*tid+7
                double x[8];
                fp8s_load_r4(fsm, x, tid);
                tok = mbar_arrive(bar);
                pending = true;
                fp8_bflys(x, t, fq, fqinv);
                if (!F1) {
#pragma unroll
                    for (int k = 0; k < 8; k++) xv[k] = KS_LAZY_X ? fp_biased_u64(x[k], off52) : fp_canon(x[k], fq, fqinv);
                }
                if (F0) {
#pragma unroll
                    for (int k = 0; k < 8; k++) xd[k] = x[k];
                }
            }
        } else {
            if (p.wide) {
                ldg256(xin, xv[0], xv[1], xv[2], xv[3]);
                ldg256(xin + 4, xv[4], xv[5], xv[6], xv[7]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) { const ulonglong2 v = ldg128(xin + 2 * j); xv[2 * j] = v.x; xv[2 * j + 1] = v.y; }
            }
            if (F0) {
                if ((xv[0] | xv[1] | xv[2] | xv[3] | xv[4] | xv[5] | xv[6] | xv[7]) >> 46) {
#pragma unroll
                    for (int k = 0; k < 8; k++) xv[k] = bred_add(xv[k], q, L.bred_hi);
                }
#pragma unroll
                for (int k = 0; k < 8; k++) xd[k] = u2d(xv[k]);
            }
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            ulonglong2 k0[2], k1[2];
            if (p.wide) {
                ldg256(e0 + 4 * h, k0[0].x, k0[0].y, k0[1].x, k0[1].y);
                ldg256(e1 + 4 * h, k1[0].x, k1[0].y, k1[1].x, k1[1].y);
            } else {
#pragma unroll
                for (int j = 0; j < 2; j++) { k0[j] = ldg128(e0 + 4 * h + 2 * j); k1[j] = ldg128(e1 + 4 * h + 2 * j); }
            }
            if (F0) {
                u64 g = k0[0].x | k0[0].y | k0[1].x | k0[1].y;
                if (F1) g |= k1[0].x | k1[0].y | k1[1].x | k1[1].y;
                if (g >> 46) {
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        k0[j].x = bred_add(k0[j].x, q, L.bred_hi); k0[j].y = bred_add(k0[j].y, q, L.bred_hi);
                        if (F1) { k1[j].x = bred_add(k1[j].x, q, L.bred_hi); k1[j].y = bred_add(k1[j].y, q, L.bred_hi); }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int pj = 2 * h + j;
                if (F0) {
                    double2 m0;
                    m0.x = fp_mulmod(xd[2 * pj], u2d(k0[j].x), fq, fqinv); m0.y = fp_mulmod(xd[2 * pj + 1], u2d(k0[j].y), fq, fqinv);
                    double2* A0 = accd + (size_t)(0 * 4 + pj) * T + tid;
                    if (d != 0) { const double2 c0 = *A0; m0.x = __dadd_rn(m0.x, c0.x); m0.y = __dadd_rn(m0.y, c0.y); }
                    *A0 = m0;
                } else {
                    ulonglong2 m0;
                    m0.x = mred_lazy(k0[j].x, xv[2 * pj], q, qinv); m0.y = mred_lazy(k0[j].y, xv[2 * pj + 1], q, qinv);
                    ulonglong2* A0 = accs + (size_t)(0 * 4 + pj) * T + tid;
                    // plain adds: every term is < 2q < 2^47 and there are at most kMaxDigits of them, so the u64 sums cannot
                    // overflow; one Barrett step in the epilogue gives the canonical residue the reference's Reduce leaves
                    if (d != 0) { const ulonglong2 c0 = *A0; m0.x += c0.x; m0.y += c0.y; }
                    *A0 = m0;
                }
                if (R1) {
                    acc1[2 * pj] = __dadd_rn(acc1[2 * pj], fp_mulmod(xd[2 * pj], u2d(k1[j].x), fq, fqinv));
                    acc1[2 * pj + 1] = __dadd_rn(acc1[2 * pj + 1], fp_mulmod(xd[2 * pj + 1], u2d(k1[j].y), fq, fqinv));
                } else if (F1) {
                    double2 m1;
                    m1.x = fp_mulmod(xd[2 * pj], u2d(k1[j].x), fq, fqinv); m1.y = fp_mulmod(xd[2 * pj + 1], u2d(k1[j].y), fq, fqinv);
                    double2* A1 = accd + (size_t)(1 * 4 + pj) * T + tid;
                    if (d != 0) { const double2 c1 = *A1; m1.x = __dadd_rn(m1.x, c1.x); m1.y = __dadd_rn(m1.y, c1.y); }
                    *A1 = m1;
                } else {
                    ulonglong2 m1;
                    m1.x = mred_lazy(k1[j].x, xv[2 * pj], q, qinv); m1.y = mred_lazy(k1[j].y, xv[2 * pj + 1], q, qinv);
                    ulonglong2* A1 = accs + (size_t)(1 * 4 + pj) * T + tid;
                    if (d != 0) { const ulonglong2 c1 = *A1; m1.x += c1.x; m1.y += c1.y; }
                    *A1 = m1;
                }
            }
        }
    }
    u64* o0 = p.acc + (size_t)b * p.acc_bs + (size_t)row * N + ((size_t)chunk << CL) + 8 * tid;
    u64* o1 = o0 + p.acc_cs;
    const double rinv = u2d(mred(1, 1, q, qinv));      // 2^-64 mod q: takes the Montgomery factor of the key out of the FP64 sums
#pragma unroll
    for (int pj = 0; pj < 4; pj++) {
        ulonglong2 r0, r1;
        if (F0) {
            const double2 c0 = accd[(size_t)(0 * 4 + pj) * T + tid];
            r0.x = fp_canon(fp_mulmod(c0.x, rinv, fq, fqinv), fq, fqinv); r0.y = fp_canon(fp_mulmod(c0.y, rinv, fq, fqinv), fq, fqinv);
        } else {
            const ulonglong2 c0 = accs[(size_t)(0 * 4 + pj) * T + tid];
            r0.x = bred_add(c0.x, q, L.bred_hi); r0.y = bred_add(c0.y, q, L.bred_hi);
        }
        if (R1) {
            r1.x = fp_canon(fp_mulmod(acc1[2 * pj], rinv, fq, fqinv), fq, fqinv); r1.y = fp_canon(fp_mulmod(acc1[2 * pj + 1], rinv, fq, fqinv), fq, fqinv);
        } else if (F1) {
            const double2 c1 = accd[(size_t)(1 * 4 + pj) * T + tid];
            r1.x = fp_canon(fp_mulmod(c1.x, rinv, fq, fqinv), fq, fqinv); r1.y = fp_canon(fp_mulmod(c1.y, rinv, fq, fqinv), fq, fqinv);
        } else {
            const ulonglong2 c1 = accs[(size_t)(1 * 4 + pj) * T + tid];
            r1.x = bred_add(c1.x, q, L.bred_hi); r1.y = bred_add(c1.y, q, L.bred_hi);
        }
        *reinterpret_cast<ulonglong2*>(o0 + 2 * pj) = r0;
        *reinterpret_cast<ulonglong2*>(o1 + 2 * pj) = r1;
    }
}

// ------------------------------------------------------------------------------------------------------------
// K3 for the integer rows (primes above 2^46: q0, the 56 / 60-bit levels of the bootstrapping chains, the 61-bit special primes), same
// structure as ks_chunk_mac_fp8r_kernel: 512 threads x 8 coefficients, swizzled tile, pair / warp level exchanges, the last radix-8 round
// and the MAC in registers, split mbarrier between digits. The 256 x 16 kernel it replaces (ks_chunk_mac_kernel<false>, kept as
// LGPU_K3_INT_VARIANT=0) ran 16 warps per SM with CTA-wide barriers and cost 3.3x an FP64 row per row (profiles/r02_configs.json).
// ------------------------------------------------------------------------------------------------------------
template <bool CORR>
__global__ void __launch_bounds__(512, 2) ks_chunk_mac_int8r_kernel(KsChunkParams p) {
    constexpr int CL = 12, T = 512;
    extern __shared__ u64 smem[];
    __shared__ __align__(8) u64 s_bar;
    u64* sm = smem;
    ulonglong2* accs = reinterpret_cast<ulonglong2*>(smem + 4096);
    const int b = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
    const int limb = p.rm.limb[blockIdx.z];
    const int row = p.rm.drow[blockIdx.z];
    const LimbConst L = p.limbs[limb];
    const int s1 = p.logN - CL;
    const int N = 1 << p.logN;
    const u64 q = L.q, qinv = L.qinv, twoq = q << 1, nq = 0ull - q, kq = L.kq;
    const unsigned mask = L.fwd_mask;
    const ulonglong2* tw = L.tw_fwd;
    const size_t erow = (size_t)(row < p.nq ? row : p.nQk + (row - p.nq)) * N + ((size_t)chunk << CL);
    const u64* P1row = p.P1 + (size_t)b * p.p1_bs + (size_t)row * N + ((size_t)chunk << CL);
    const u64* xin = p.cx + (size_t)b * p.cx_bs + (size_t)row * p.cx_rs + ((size_t)chunk << CL) + 8 * tid;
    const int own_d = row < p.nq ? row / p.k : -1;
    const unsigned bar = smem_addr(&s_bar);
    if (tid == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(T) : "memory");
    __syncthreads();
    u64 tok = 0;
    bool pending = false;
    for (int d = 0; d < p.nd; d++) {
        const bool own = d == own_d;
        const u64* e0 = p.evk + (size_t)d * p.evk_ds + erow + 8 * tid;
        const u64* e1 = e0 + p.evk_cs;
        int dn = d + 1;
        if (dn == own_d) dn++;
        u64 xv[8];
        if (!own) {
            {
                u64 x[8];
#pragma unroll
                for (int k = 0; k < 8; k++) x[k] = P1row[(size_t)d * p.p1_ds + k * T + tid];
                if (KS_L2_PREFETCH && dn < p.nd && tid < 256)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(P1row + (size_t)dn * p.p1_ds + tid * 16));
                int8_bflys<0, CORR>(x, tw, s1, chunk, 0, nq, twoq, kq, mask);
                if (pending) { mbar_wait(bar, tok); pending = false; }
                i8s_store_r1(sm, x, tid);
            }
            __syncthreads();
            i8s_round2<CORR>(sm, tw, s1, chunk, tid, nq, twoq, kq, mask);
            fp8s_pair_sync(tid);
            i8s_round3<CORR>(sm, tw, s1, chunk, tid, nq, twoq, kq, mask);
            __syncwarp();
            i8s_load_r4(sm, xv, tid);
            tok = mbar_arrive(bar);
            pending = true;
            int8_bflys<9, CORR>(xv, tw, s1, chunk, tid, nq, twoq, kq, mask);     // lazy values below 2 kq: any u64 is a valid MRedLazy operand
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) { const ulonglong2 v = ldg128(xin + 2 * j); xv[2 * j] = v.x; xv[2 * j + 1] = v.y; }
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            ulonglong2 k0[2], k1[2];
#pragma unroll
            for (int j = 0; j < 2; j++) { k0[j] = ldg128(e0 + 4 * h + 2 * j); k1[j] = ldg128(e1 + 4 * h + 2 * j); }
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int pj = 2 * h + j;
                const u64 xa = xv[2 * pj], xb = xv[2 * pj + 1];
                ulonglong2 m0, m1;
                m0.x = mred_lazy(k0[j].x, xa, q, qinv); m0.y = mred_lazy(k0[j].y, xb, q, qinv);
                m1.x = mred_lazy(k1[j].x, xa, q, qinv); m1.y = mred_lazy(k1[j].y, xb, q, qinv);
                ulonglong2* A0 = accs + (size_t)(0 * 4 + pj) * T + tid;
                ulonglong2* A1 = accs + (size_t)(1 * 4 + pj) * T + tid;
                if (d != 0) {
                    // terms are below 2q and q reaches 2^61: keep the running sums below 2q (4q fits 64 bits)
                    const ulonglong2 c0 = *A0, c1 = *A1;
                    m0.x += c0.x; m0.y += c0.y; m1.x += c1.x; m1.y += c1.y;
                    m0.x = m0.x >= twoq ? m0.x - twoq : m0.x; m0.y = m0.y >= twoq ? m0.y - twoq : m0.y;
                    m1.x = m1.x >= twoq ? m1.x - twoq : m1.x; m1.y = m1.y >= twoq ? m1.y - twoq : m1.y;
                }
                *A0 = m0; *A1 = m1;
            }
        }
    }
    u64* o0 = p.acc + (size_t)b * p.acc_bs + (size_t)row * N + ((size_t)chunk << CL) + 8 * tid;
    u64* o1 = o0 + p.acc_cs;
#pragma unroll
    for (int pj = 0; pj < 4; pj++) {
        const ulonglong2 c0 = accs[(size_t)(0 * 4 + pj) * T + tid], c1 = accs[(size_t)(1 * 4 + pj) * T + tid];
        ulonglong2 r0, r1;
        r0.x = cred(c0.x, q); r0.y = cred(c0.y, q); r1.x = cred(c1.x, q); r1.y = cred(c1.y, q);
        *reinterpret_cast<ulonglong2*>(o0 + 2 * pj) = r0;
        *reinterpret_cast<ulonglong2*>(o1 + 2 * pj) = r1;
    }
}

// ------------------------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------------------------
bool ks_fused_applicable(const Ctx* c, int levelQ, const GadgetCt& evk) {
    static const int off = [] { const char* e = getenv("LGPU_NO_FUSED_KS"); return e && atoi(e) ? 1 : 0; }();
    if (off || c->ring_type != 0) return false;
    if (c->logN < 13 || c->logN > 16) return false;            // two-pass transforms with a 4096-element chunk pass; validated sizes only (2^17 takes the unfused kernels)
    if (evk.levelP < 1 || evk.pw2 != 0) return false;          // multiple-P path only
    const int k = evk.levelP + 1;
    const int nd = base_rns_decomposition_vector_size(levelQ, evk.levelP);
    // digit sizes 2..6 (the reference's parameter sets use up to 6 special primes: circuits/ckks/bootstrapping/default_parameters.go:118-134);
    // the 128-bit sum of ks_ext holds k products of a source word and a target constant: k * 2^61 * t < t * 2^64 needs k < 8
    if (levelQ + 1 > 64 || nd > kMaxDigits || k > 6) return false;
    return true;
}

template <int RL, int NSMAX, bool FP, bool CORR, bool BC>
static int ks_launch_j4(const KsStridedParams& p, dim3 grid, cudaStream_t st) {
    constexpr int R = 1 << RL;
    constexpr int LB = 256 / KS_J;
    const size_t smem = (size_t)NSMAX * R * LB * sizeof(u64) + (size_t)R * LB + (BC ? (size_t)R * 256 * sizeof(u64) : 0);
    LGPU_CUDA_OK(cudaFuncSetAttribute(ks_strided_j4_kernel<RL, NSMAX, FP, CORR, BC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ks_strided_j4_kernel<RL, NSMAX, FP, CORR, BC><<<dim3(grid.x * KS_J, (grid.y + KS_J - 1) / KS_J, grid.z), 256, smem, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

// CORR: the integer rows of the launch need the lazy-correction schedule (some prime above 2^57); ignored for FP64 rows
template <bool FP, int PRO = PRO_MODUP, bool CORR = true>
static int ks_launch_strided(int rl, int nsmax, const KsStridedParams& p, dim3 grid, cudaStream_t st) {
    if constexpr (PRO != PRO_BCAST) {
        constexpr bool BC = PRO == PRO_MODUP_BCAST;
        static const int j4 = [] { const char* e = getenv("LGPU_K2_J4"); return e ? atoi(e) : 1; }();
        bool multi = j4 != 0 && rl <= 4;                       // R = 32 (N = 2^17) would need 2 x 66 KB of shared memory
        for (int d = 0; d < p.nd; d++) multi = multi && (p.dg[d].nS > 1 || !p.single_rule);
        if (multi) {
#define KS_J4(RLV) case RLV: return nsmax <= 4 ? ks_launch_j4<RLV, 4, FP, CORR, BC>(p, grid, st) : ks_launch_j4<RLV, 8, FP, CORR, BC>(p, grid, st);
            switch (rl) { KS_J4(1) KS_J4(2) KS_J4(3) KS_J4(4) default: break; }
#undef KS_J4
        }
    }
#define KS_CASE(RLV) \
    case RLV: if (nsmax <= 4) ks_strided_kernel<RLV, 4, FP, PRO, CORR><<<grid, 256, 0, st>>>(p); else ks_strided_kernel<RLV, 8, FP, PRO, CORR><<<grid, 256, 0, st>>>(p); break;
    switch (rl) {
        KS_CASE(1) KS_CASE(2) KS_CASE(3) KS_CASE(4) KS_CASE(5)
        default: set_error("unsupported strided radix"); return -1;
    }
#undef KS_CASE
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

// integer rows whose prime needs the lazy-correction schedule (fwd_mask != 0: above 2^57) vs rows that never correct: the second class
// runs instantiations with the correction compiled out
static void split_by_corr(const Ctx* c, const RowMap& in, RowMap& corr, RowMap& plain) {
    corr.nrows = plain.nrows = 0;
    for (int r = 0; r < in.nrows; r++) {
        RowMap& d = c->h_limbs[in.limb[r]].fwd_mask != 0 ? corr : plain;
        d.limb[d.nrows] = in.limb[r]; d.drow[d.nrows] = in.drow[r]; d.nrows++;
    }
}

// acc: QP-stacked accumulators (component c, batch b at acc + c*acc_cs + b*acc_bs, rows 0..nq-1 Q then P; canonical).
// cx: NTT-domain input, cxInv: its INTT (coefficient domain).
int gadget_product_multiple_p_fused(const Ctx* c, int levelQ, CSpan cx, CSpan cxInv, const GadgetCt& evk, u64* acc, size_t acc_cs, size_t acc_bs,
                                    int batch, cudaStream_t st) {
    const int levelP = evk.levelP;
    const int k = levelP + 1, nq = levelQ + 1, np = levelP + 1, nrows = nq + np;
    const int nd = base_rns_decomposition_vector_size(levelQ, levelP);
    const size_t N = c->N;
    const int s1 = c->logN - 12;
    // scratch: Y [batch][nq][N] | P1 [batch][nd][nrows][N] | V [batch][nd][N] bytes
    const size_t y_words = (size_t)batch * nq * N;
    const size_t p1_words = (size_t)batch * nd * nrows * N;
    const size_t v_words = ((size_t)batch * nd * N + 7) / 8;
    u64* buf = nullptr;
    LGPU_CUDA_OK(cudaMallocAsync((void**)&buf, (y_words + p1_words + v_words) * sizeof(u64), st));
    struct Free { u64* p; cudaStream_t s; ~Free() { cudaFreeAsync(p, s); } } guard{buf, st};
    u64* Y = buf;
    u64* P1 = buf + y_words;
    unsigned char* V = reinterpret_cast<unsigned char*>(P1 + p1_words);

    // ---- K1
    KsPrepParams pp;
    memset(&pp, 0, sizeof(pp));
    pp.limbs = c->d_limbs; pp.cx = cxInv.p; pp.cx_rs = cxInv.row_stride; pp.cx_bs = cxInv.batch_stride;
    pp.Y = Y; pp.y_bs = (size_t)nq * N; pp.V = V; pp.v_bs = (size_t)nd * N;
    pp.nq = nq; pp.nd = nd; pp.k = k; pp.n = c->N; pp.limb0 = 0; pp.single_rule = 1;
    KsStridedParams sp;
    memset(&sp, 0, sizeof(sp));
    int nsmax = 1;
    for (int d = 0; d < nd; d++) {
        const int r0 = d * k, r1 = std::min(r0 + k, nq), nS = r1 - r0;
        sp.dg[d].nS = (unsigned short)nS;
        if (nS > nsmax) nsmax = nS;
        if (nS == 1) continue;
        if (k - 2 >= (int)c->muc_dec.size() || d >= (int)c->muc_dec[k - 2].size() || nS - 2 >= (int)c->muc_dec[k - 2][d].size()) {
            set_error("no decomposer constants for this (nbPi, digit, level)");
            return -1;
        }
        const ModUpSet& m = c->muc_dec[k - 2][d][nS - 2];
        for (int i = 0; i < nS; i++) {
            pp.half_src[r0 + i] = c->h_blob[m.off_half_s + i];
            pp.cinv[r0 + i] = c->h_blob[m.off_qoverqiinvqi + i];
        }
        sp.dg[d].off_c = (unsigned)m.off_qoverqimodp; sp.dg[d].off_vt = (unsigned)m.off_vtimesqmodp;
        sp.dg[d].off_half_t = (unsigned)m.off_half_t; sp.dg[d].ldc = (unsigned short)m.nS;
        sp.dg[d].off_cp = (unsigned)m.off_c_plain;
        bool fps = true;
        for (int i = r0; i < r1; i++) fps = fps && c->h_limbs[i].fp_ok;
        sp.dg[d].fp_src = fps ? (unsigned short)(1 + k2_fpsum()) : 0;
    }
    {
        ProfScope ps(LGPU_KCLASS_MODUP, st, 8.0 * N * batch * (2.0 * nq), 1);
        dim3 grid((unsigned)((N + 255) / 256), batch);
        ks_prepare_kernel<<<grid, 256, 0, st>>>(pp);
        LGPU_CUDA_OK(cudaGetLastError());
    }
    // row classes
    RowMap fp, in;
    fp.nrows = in.nrows = 0;
    for (int r = 0; r < nrows; r++) {
        const int limb = r < nq ? r : c->nQ + (r - nq);
        RowMap& dst = (c->h_limbs[limb].fp_ok && fp64_ntt_supported(c)) ? fp : in;
        dst.limb[dst.nrows] = (unsigned char)limb; dst.drow[dst.nrows] = (unsigned char)r; dst.nrows++;
    }
    // ---- K2 + K3: FP64 rows on `st`, integer rows on the side stream
    sp.limbs = c->d_limbs; sp.blob = c->d_blob; sp.Y = Y; sp.y_bs = (size_t)nq * N; sp.V = V; sp.v_bs = (size_t)nd * N;
    sp.P1 = P1; sp.p1_ds = (size_t)nrows * N; sp.p1_bs = (size_t)nd * nrows * N;
    sp.logN = c->logN; sp.nq = nq; sp.k = k; sp.nd = nd; sp.skip_own = 1; sp.single_rule = 1; sp.src_limb0 = 0; sp.split23 = k2_split();
    KsChunkParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.limbs = c->d_limbs; cp.P1 = P1; cp.p1_ds = sp.p1_ds; cp.p1_bs = sp.p1_bs;
    cp.cx = cx.p; cp.cx_rs = cx.row_stride; cp.cx_bs = cx.batch_stride;
    const size_t key_rows = (size_t)(evk.levelQ + 1) + (size_t)(evk.levelP + 1);
    cp.evk = evk.data; cp.evk_cs = key_rows * N; cp.evk_ds = (size_t)evk.npw2max * 2 * key_rows * N; cp.nQk = evk.levelQ + 1;
    cp.acc = acc; cp.acc_cs = acc_cs; cp.acc_bs = acc_bs;
    cp.logN = c->logN; cp.nq = nq; cp.k = k; cp.nd = nd;
    // LGPU_K3_WIDE (default 1): 256-bit key / own-row loads when everything is 32-byte aligned (the ABI only asks for 16)
    static const int k3wide = [] { const char* e = getenv("LGPU_K3_WIDE"); return e ? atoi(e) : 1; }();
    cp.wide = k3wide && ((reinterpret_cast<uintptr_t>(cp.evk) | reinterpret_cast<uintptr_t>(cp.cx)) & 31u) == 0 &&
              ((cp.evk_ds | cp.evk_cs | cp.cx_rs | cp.cx_bs) & 3u) == 0;
    const size_t smem = (size_t)(4096 + 256 + 8 + 2 * 4096) * sizeof(u64);
    const unsigned gx = (unsigned)(((N >> s1) + 255) / 256);
    const unsigned chunks = (unsigned)(N >> 12);
    cudaStream_t sint = fork_side(c, st, fp.nrows > 0 && in.nrows > 0);
    RowMap in_c, in_n;
    split_by_corr(c, in, in_c, in_n);
    for (int pass = 0; pass < 2; pass++) {
        const RowMap& ir = pass ? in_n : in_c;
        if (!ir.nrows) continue;
        sp.rm = ir; cp.rm = ir;
        {
            ProfScope ps(LGPU_KCLASS_FUSED, sint, 8.0 * N * batch * nd * (double)ir.nrows, 1);
            if (pass ? ks_launch_strided<false, PRO_MODUP, false>(s1, nsmax, sp, dim3(gx, ir.nrows, nd * batch), sint)
                     : ks_launch_strided<false, PRO_MODUP, true>(s1, nsmax, sp, dim3(gx, ir.nrows, nd * batch), sint)) return -1;
        }
        ProfScope ps(LGPU_KCLASS_MAC, sint, 8.0 * N * ir.nrows * (batch * (double)(nd + 2) + 2.0 * nd), 1);
        // LGPU_K3_INT_VARIANT=0 selects the 256 x 16 shared-memory-MAC kernel (cross-check of the default 512 x 8 register-MAC one)
        static const int k3i = [] { const char* e = getenv("LGPU_K3_INT_VARIANT"); return e ? atoi(e) : 8; }();
        if (k3i != 0 && pass) {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_int8r_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_int8r_kernel<false><<<dim3(batch, chunks, ir.nrows), 512, smem, sint>>>(cp);
        } else if (k3i != 0) {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_int8r_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_int8r_kernel<true><<<dim3(batch, chunks, ir.nrows), 512, smem, sint>>>(cp);
        } else {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_kernel<false><<<dim3(batch, chunks, ir.nrows), 256, smem, sint>>>(cp);
        }
        LGPU_CUDA_OK(cudaGetLastError());
    }
    if (fp.nrows) {
        sp.rm = fp; cp.rm = fp;
        {
            ProfScope ps(LGPU_KCLASS_FUSED, st, 8.0 * N * batch * nd * (double)fp.nrows, 1);
            if (ks_launch_strided<true>(s1, nsmax, sp, dim3(gx, fp.nrows, nd * batch), st)) return -1;
        }
        // algorithmic bytes: P1 read once + accumulators written once + evk once per launch
        ProfScope ps(LGPU_KCLASS_MAC, st, 8.0 * N * fp.nrows * (batch * (double)(nd + 2) + 2.0 * nd), 1);
        // LGPU_K3_VARIANT: 11 (default) = 512 x 8 kernel with the FP64-pipe MAC, 10 = integer-pipe MAC, 12 = one component each (measured 64.3 / 65.3 /
        // 66.3 ms per 4 steps for the class, profiles/r02_ab_late.txt), 0 = the 256 x 16 shared-memory-MAC kernel (kept as a cross-check)
        static const int k3v = [] { const char* e = getenv("LGPU_K3_VARIANT"); return e ? atoi(e) : 11; }();
        if (k3v == 11) {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_fp8r_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_fp8r_kernel<1><<<dim3(batch, chunks, fp.nrows), 512, smem, st>>>(cp);
        } else if (k3v == 13) {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_fp8r_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_fp8r_kernel<3><<<dim3(batch, chunks, fp.nrows), 512, smem, st>>>(cp);
        } else if (k3v == 12) {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_fp8r_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_fp8r_kernel<2><<<dim3(batch, chunks, fp.nrows), 512, smem, st>>>(cp);
        } else if (k3v != 0) {      // 10
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_fp8r_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_fp8r_kernel<0><<<dim3(batch, chunks, fp.nrows), 512, smem, st>>>(cp);
        } else {
            LGPU_CUDA_OK(cudaFuncSetAttribute(ks_chunk_mac_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ks_chunk_mac_kernel<true><<<dim3(batch, chunks, fp.nrows), 256, smem, st>>>(cp);
        }
        LGPU_CUDA_OK(cudaGetLastError());
    }
    join_side(c, st, sint);
    return 0;
}


// ------------------------------------------------------------------------------------------------------------
// chunk pass with an element-wise epilogue: out = CRed( MRed(x + 2q - a, s) [+ d] ), x = NTT(P1 row).
// Used by the fused ModDown (a = accumulator Q rows, s = -P^-1, d = the other summand of the ciphertext) and the
// fused rescale (a = input rows, s = RescaleConstants): SubThenMulScalarMontgomeryTwoModulus, ring/vec_ops.go:752.
// RS (merged ModDown + Rescale tail): out = CRed( MRed(x + 2q - d, s) + MRed(a, s2) ) = ((d - x) q_L^-1 + a P^-1 q_L^-1) mod q with
// s = RescaleConstants, s2 = MForm(P^-1 q_L^-1), x = NTT(P^-1 ModUp + broadcast term), a the accumulator, d the other summand (or 0).
// Both MReds are canonical (a < q, s < q), so the sum is below 2q.
// Buffers with a (component, batch) structure are addressed as  z -> (z / nb) * cs + (z % nb) * bs.
// ------------------------------------------------------------------------------------------------------------
struct FzChunkParams {
    const LimbConst* limbs;
    RowMap rm;
    const u64* P1; size_t p1_bs;
    const u64* A; size_t a_cs, a_bs;
    const u64* D; size_t d_cs, d_bs;
    u64* out; size_t o_cs, o_bs;
    int nb, logN;
    int wide;                 // 1: A / D / out are 32-byte aligned -> 256-bit accesses in fz_chunk_epi_fp8_kernel (LGPU_K3_WIDE)
    u64 s[kMaxRows];
    u64 s2[kMaxRows];         // RS only
};

template <bool RS>
__device__ __forceinline__ u64 fz_epi(u64 x, u64 a, u64 d, bool has_d, u64 sc, u64 sc2, u64 q, u64 qinv) {
    if (RS) return cred(mred(x + (q << 1) - d, sc, q, qinv) + mred(a, sc2, q, qinv), q);
    const u64 r = mred(x + (q << 1) - a, sc, q, qinv);
    return has_d ? cred(r + d, q) : r;
}

template <bool FP, bool RS>
__global__ void __launch_bounds__(256, 2) fz_chunk_epi_kernel(FzChunkParams p) {
    constexpr int CL = 12, T = 256;
    extern __shared__ u64 smem[];
    u64* sm = smem;
    const int chunk = blockIdx.x, z = blockIdx.z, tid = threadIdx.x;
    const int limb = p.rm.limb[blockIdx.y];
    const int row = p.rm.drow[blockIdx.y];
    const LimbConst L = p.limbs[limb];
    const int s1 = p.logN - CL;
    const int N = 1 << p.logN;
    const u64 q = L.q, qinv = L.qinv;
    const u64 sc = p.s[blockIdx.y], sc2 = RS ? p.s2[blockIdx.y] : 0;
    const int zc = z / p.nb, zb = z % p.nb;
    const size_t roff = (size_t)row * N + ((size_t)chunk << CL);
    const u64* src = p.P1 + (size_t)z * p.p1_bs + roff;
    const u64* A = p.A + (size_t)zc * p.a_cs + (size_t)zb * p.a_bs + roff;
    const u64* D = p.D ? p.D + (size_t)zc * p.d_cs + (size_t)zb * p.d_bs + roff : nullptr;
    u64* out = p.out + (size_t)zc * p.o_cs + (size_t)zb * p.o_bs + roff;
    if constexpr (FP) {
        double* fsm = reinterpret_cast<double*>(sm);
        fp_fwd_round<CL, 0, 4, 2>(fsm, src, L, s1, chunk, tid);
        double t2[15];
        fp_load_tw<CL, 4, 4>(t2, L.ftw_fwd, s1, chunk, tid);
        __syncthreads();
        fp_fwd_round_tw<CL, 4, 4>(fsm, t2, L.fq, L.fqinv, tid);
        double t3[15];
        fp_load_tw<CL, 8, 4>(t3, L.ftw_fwd, s1, chunk, tid);
        __syncthreads();
        fp_fwd_round_tw<CL, 8, 4>(fsm, t3, L.fq, L.fqinv, tid);
    } else {
        fwd_round<CL, 0, 4, true, 1>(sm, src, L, s1, p.logN, chunk, tid);
        __syncthreads();
        fwd_round<CL, 4, 4, false, 1>(sm, nullptr, L, s1, p.logN, chunk, tid);
        __syncthreads();
        fwd_round<CL, 8, 4, false, 1>(sm, nullptr, L, s1, p.logN, chunk, tid);
    }
    __syncthreads();
    // loads of a whole batch are issued before any store (out may alias A or D, so the compiler cannot hoist them itself)
    constexpr int EB = 8;
#pragma unroll 1
    for (int k0 = 0; k0 < 16; k0 += EB) {
        u64 a[EB], d[EB];
#pragma unroll
        for (int j = 0; j < EB; j++) {
            const int idx = (k0 + j) * T + tid;
            a[j] = A[idx];
            d[j] = D ? D[idx] : 0;
        }
#pragma unroll
        for (int j = 0; j < EB; j++) {
            const int idx = (k0 + j) * T + tid;
            u64 x;
            if (FP) x = fp_canon(reinterpret_cast<double*>(sm)[fpad(idx)], L.fq, L.fqinv);
            else {
                // lazy transform output: below 2 kq, i.e. up to ~2^64 for 60/61-bit primes -- one correction keeps x + 2q - a
                // inside 64 bits (kq is a multiple of q)
                x = sm[pad_idx(idx)];
                x = x >= L.kq ? x - L.kq : x;
            }
            out[idx] = fz_epi<RS>(x, a[j], d[j], D != nullptr, sc, sc2, q, qinv);
        }
    }
}

// high-occupancy FP64 variant of the same kernel (512 threads x 8 elements, last round and epilogue in registers,
// see ks_chunk_mac_fp8r_kernel)
template <bool RS>
__global__ void __launch_bounds__(512, 2) fz_chunk_epi_fp8_kernel(FzChunkParams p) {
    constexpr int CL = 12, T = 512;
    extern __shared__ u64 smem[];
    double* fsm = reinterpret_cast<double*>(smem);
    const int chunk = blockIdx.x, z = blockIdx.z, tid = threadIdx.x;
    const int limb = p.rm.limb[blockIdx.y];
    const int row = p.rm.drow[blockIdx.y];
    const LimbConst L = p.limbs[limb];
    const int s1 = p.logN - CL;
    const int N = 1 << p.logN;
    const u64 q = L.q, qinv = L.qinv;
    const double fq = L.fq, fqinv = L.fqinv;
    const double off52 = __dmul_rn((double)(10 + p.logN), fq) + 4503599627370496.0;   // (10 + logN) q + 2^52, exact
    const double* tw = L.ftw_fwd;
    const u64 sc = p.s[blockIdx.y], sc2 = RS ? p.s2[blockIdx.y] : 0;
    const int zc = z / p.nb, zb = z % p.nb;
    const size_t roff = (size_t)row * N + ((size_t)chunk << CL);
    const u64* src = p.P1 + (size_t)z * p.p1_bs + roff;
    const u64* A = p.A + (size_t)zc * p.a_cs + (size_t)zb * p.a_bs + roff;
    const u64* D = p.D ? p.D + (size_t)zc * p.d_cs + (size_t)zb * p.d_bs + roff : nullptr;
    u64* out = p.out + (size_t)zc * p.o_cs + (size_t)zb * p.o_bs + roff;
    {
        double x[8];
#pragma unroll
        for (int k = 0; k < 8; k++) x[k] = __longlong_as_double((long long)src[k * T + tid]);
        {
            double t1[7];
            fp8_load_tw<0>(t1, tw, s1, chunk, tid);       // CTA-uniform: hi = 0
            fp8_bflys(x, t1, fq, fqinv);
        }
        fp8s_store_r1(fsm, x, tid);
    }
    double t[7];
    fp8_load_tw<3>(t, tw, s1, chunk, tid);
    __syncthreads();
    fp8s_round2(fsm, t, fq, fqinv, tid);
    fp8_load_tw<6>(t, tw, s1, chunk, tid);
    fp8s_pair_sync(tid);
    fp8s_round3(fsm, t, fq, fqinv, tid);
    fp8_load_tw<9>(t, tw, s1, chunk, tid);
    // the operands of the epilogue for this thread's 8 consecutive coefficients (last round: stages 9..11 act inside
    // aligned groups of 8), issued before the warp-level exchange so that their latency overlaps it
    ulonglong2 a[4], d[4];
    if (p.wide) {
        ld256(A + 8 * tid, a[0].x, a[0].y, a[1].x, a[1].y);
        ld256(A + 8 * tid + 4, a[2].x, a[2].y, a[3].x, a[3].y);
        if (D) {
            ld256(D + 8 * tid, d[0].x, d[0].y, d[1].x, d[1].y);
            ld256(D + 8 * tid + 4, d[2].x, d[2].y, d[3].x, d[3].y);
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) d[j] = make_ulonglong2(0, 0);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            a[j] = *reinterpret_cast<const ulonglong2*>(A + 8 * tid + 2 * j);
            d[j] = D ? *reinterpret_cast<const ulonglong2*>(D + 8 * tid + 2 * j) : make_ulonglong2(0, 0);
        }
    }
    __syncwarp();
    double x[8];
    fp8s_load_r4(fsm, x, tid);
    fp8_bflys(x, t, fq, fqinv);
    ulonglong2 r[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const u64 xa = KS_LAZY_X ? fp_biased_u64(x[2 * j], off52) : fp_canon(x[2 * j], fq, fqinv);
        const u64 xb = KS_LAZY_X ? fp_biased_u64(x[2 * j + 1], off52) : fp_canon(x[2 * j + 1], fq, fqinv);
        r[j].x = fz_epi<RS>(xa, a[j].x, d[j].x, D != nullptr, sc, sc2, q, qinv);
        r[j].y = fz_epi<RS>(xb, a[j].y, d[j].y, D != nullptr, sc, sc2, q, qinv);
    }
    if (p.wide) {
        st256(out + 8 * tid, r[0].x, r[0].y, r[1].x, r[1].y);
        st256(out + 8 * tid + 4, r[2].x, r[2].y, r[3].x, r[3].y);
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) *reinterpret_cast<ulonglong2*>(out + 8 * tid + 2 * j) = r[j];
    }
}

// integer-row variant of fz_chunk_epi_fp8_kernel (512 threads x 8 elements, last round and epilogue in registers)
template <bool CORR, bool RS>
__global__ void __launch_bounds__(512, 2) fz_chunk_epi_int8_kernel(FzChunkParams p) {
    constexpr int CL = 12, T = 512;
    extern __shared__ u64 smem[];
    u64* sm = smem;
    const int chunk = blockIdx.x, z = blockIdx.z, tid = threadIdx.x;
    const int limb = p.rm.limb[blockIdx.y];
    const int row = p.rm.drow[blockIdx.y];
    const LimbConst L = p.limbs[limb];
    const int s1 = p.logN - CL;
    const int N = 1 << p.logN;
    const u64 q = L.q, qinv = L.qinv, twoq = q << 1, nq = 0ull - q, kq = L.kq;
    const unsigned mask = L.fwd_mask;
    const ulonglong2* tw = L.tw_fwd;
    const u64 sc = p.s[blockIdx.y], sc2 = RS ? p.s2[blockIdx.y] : 0;
    const int zc = z / p.nb, zb = z % p.nb;
    const size_t roff = (size_t)row * N + ((size_t)chunk << CL);
    const u64* src = p.P1 + (size_t)z * p.p1_bs + roff;
    const u64* A = p.A + (size_t)zc * p.a_cs + (size_t)zb * p.a_bs + roff;
    const u64* D = p.D ? p.D + (size_t)zc * p.d_cs + (size_t)zb * p.d_bs + roff : nullptr;
    u64* out = p.out + (size_t)zc * p.o_cs + (size_t)zb * p.o_bs + roff;
    {
        u64 x[8];
#pragma unroll
        for (int k = 0; k < 8; k++) x[k] = src[k * T + tid];
        int8_bflys<0, CORR>(x, tw, s1, chunk, 0, nq, twoq, kq, mask);
        i8s_store_r1(sm, x, tid);
    }
    __syncthreads();
    i8s_round2<CORR>(sm, tw, s1, chunk, tid, nq, twoq, kq, mask);
    fp8s_pair_sync(tid);
    i8s_round3<CORR>(sm, tw, s1, chunk, tid, nq, twoq, kq, mask);
    ulonglong2 a[4], d[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        a[j] = *reinterpret_cast<const ulonglong2*>(A + 8 * tid + 2 * j);
        d[j] = D ? *reinterpret_cast<const ulonglong2*>(D + 8 * tid + 2 * j) : make_ulonglong2(0, 0);
    }
    __syncwarp();
    u64 x[8];
    i8s_load_r4(sm, x, tid);
    int8_bflys<9, CORR>(x, tw, s1, chunk, tid, nq, twoq, kq, mask);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        // lazy transform output below 2 kq (up to ~2^64 for 60 / 61-bit primes): one correction keeps x + 2q - a inside 64 bits
        u64 xa = x[2 * j], xb = x[2 * j + 1];
        xa = xa >= kq ? xa - kq : xa; xb = xb >= kq ? xb - kq : xb;
        ulonglong2 r;
        r.x = fz_epi<RS>(xa, a[j].x, d[j].x, D != nullptr, sc, sc2, q, qinv);
        r.y = fz_epi<RS>(xb, a[j].y, d[j].y, D != nullptr, sc, sc2, q, qinv);
        *reinterpret_cast<ulonglong2*>(out + 8 * tid + 2 * j) = r;
    }
}

template <bool FP, bool CORR = true, bool RS = false>
static int fz_launch_chunk(const FzChunkParams& p, dim3 grid, cudaStream_t st) {
    const size_t smem = (size_t)(4096 + 256 + 8) * sizeof(u64);
    static const int v8 = [] { const char* e = getenv("LGPU_FZ_VARIANT"); return e ? atoi(e) : 8; }();
    const bool vec_ok = aligned16(p.A) && aligned16(p.D) && aligned16(p.out) && even_words(p.a_cs, p.a_bs) && even_words(p.d_cs, p.d_bs) &&
                        even_words(p.o_cs, p.o_bs);
    if (FP && v8 == 8 && vec_ok) {
        static const int k3wide = [] { const char* e = getenv("LGPU_K3_WIDE"); return e ? atoi(e) : 1; }();
        FzChunkParams pw = p;
        pw.wide = k3wide && ((reinterpret_cast<uintptr_t>(p.A) | reinterpret_cast<uintptr_t>(p.D) | reinterpret_cast<uintptr_t>(p.out)) & 31u) == 0 &&
                  ((p.a_cs | p.a_bs | p.d_cs | p.d_bs | p.o_cs | p.o_bs) & 3u) == 0;
        fz_chunk_epi_fp8_kernel<RS><<<grid, 512, smem, st>>>(pw);
        LGPU_CUDA_OK(cudaGetLastError());
        return 0;
    }
    if (!FP && v8 == 8 && vec_ok) {
        fz_chunk_epi_int8_kernel<CORR, RS><<<grid, 512, smem, st>>>(p);
        LGPU_CUDA_OK(cudaGetLastError());
        return 0;
    }
    fz_chunk_epi_kernel<FP, RS><<<grid, 256, smem, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

// Splits `rows` into FP64-pipe rows and integer rows.
static void split_fp(const Ctx* c, const RowMap& rows, RowMap& fp, RowMap& in) {
    fp.nrows = in.nrows = 0;
    for (int r = 0; r < rows.nrows; r++) {
        RowMap& dst = (c->h_limbs[rows.limb[r]].fp_ok && fp64_ntt_supported(c)) ? fp : in;
        dst.limb[dst.nrows] = rows.limb[r]; dst.drow[dst.nrows] = rows.drow[r]; dst.nrows++;
    }
}

static RowMap q_rows(int limb0, int nrows) {
    RowMap rm;
    rm.nrows = nrows;
    for (int r = 0; r < nrows; r++) { rm.limb[r] = (unsigned char)(limb0 + r); rm.drow[r] = (unsigned char)r; }
    return rm;
}

bool fz_applicable(const Ctx* c, int levelQ, int levelP) {
    static const int off = [] { const char* e = getenv("LGPU_NO_FUSED_KS"); return e && atoi(e) ? 1 : 0; }();
    if (off || c->ring_type != 0 || c->logN < 13 || c->logN > 16) return false;
    if (levelQ + 1 > kMaxRows || levelP + 1 > 6) return false;   // source counts 1..6 (see ks_fused_applicable)
    return true;
}

// K2 strided pass with prologue PRO into sp.P1, then the chunk-pass epilogue (cp) over the Q rows `rows`: FP64 rows on `st`, integer rows
// on the side stream. consts(rm) fills the per-launch-row constants (sp.s0, cp.s, cp.s2) of one row class before its launches;
// epi_words: algorithmic words per coefficient of the epilogue.
template <int PRO, bool RS, class F>
static int fz_tail(const Ctx* c, const RowMap& rows, int nsmax, KsStridedParams& sp, FzChunkParams& cp, int Z, double epi_words, F consts,
                   cudaStream_t st) {
    const size_t N = c->N;
    const int s1 = c->logN - 12;
    const unsigned gx = (unsigned)(((N >> s1) + 255) / 256);
    const unsigned chunks = (unsigned)(N >> 12);
    RowMap fp, in;
    split_fp(c, rows, fp, in);
    cudaStream_t sint = fork_side(c, st, fp.nrows > 0 && in.nrows > 0);
    RowMap in_c, in_n;
    split_by_corr(c, in, in_c, in_n);
    for (int pass = 0; pass < 2; pass++) {
        const RowMap& ir = pass ? in_n : in_c;
        if (!ir.nrows) continue;
        consts(ir);
        { ProfScope ps(LGPU_KCLASS_FUSED, sint, 8.0 * N * Z * ir.nrows, 1);
          sp.rm = ir;
          if (pass ? ks_launch_strided<false, PRO, false>(s1, nsmax, sp, dim3(gx, ir.nrows, Z), sint)
                   : ks_launch_strided<false, PRO, true>(s1, nsmax, sp, dim3(gx, ir.nrows, Z), sint)) return -1; }
        ProfScope ps(LGPU_KCLASS_EPILOGUE, sint, 8.0 * N * Z * ir.nrows * epi_words, 1);
        cp.rm = ir;
        if (pass ? fz_launch_chunk<false, false, RS>(cp, dim3(chunks, ir.nrows, Z), sint)
                 : fz_launch_chunk<false, true, RS>(cp, dim3(chunks, ir.nrows, Z), sint)) return -1;
    }
    if (fp.nrows) {
        consts(fp);
        { ProfScope ps(LGPU_KCLASS_FUSED, st, 8.0 * N * Z * fp.nrows, 1);
          sp.rm = fp; if (ks_launch_strided<true, PRO>(s1, nsmax, sp, dim3(gx, fp.nrows, Z), st)) return -1; }
        ProfScope ps(LGPU_KCLASS_EPILOGUE, st, 8.0 * N * Z * fp.nrows * epi_words, 1);
        cp.rm = fp; if (fz_launch_chunk<true, true, RS>(cp, dim3(chunks, fp.nrows, Z), st)) return -1;
    }
    join_side(c, st, sint);
    return 0;
}

// Fused Evaluator.ModDown (NTT -> NTT, core/rlwe/evaluator_gadget_product.go:39-52 = 2 x ModDownQPtoQNTT,
// ring/basis_extension.go:235-256) for ncomp x batch QP-stacked accumulators, with an optional addend:
//     out[c][b] = (accQ[c][b] - NTT(ModUpPtoQ(INTT(accP[c][b])))) * P^-1  (+ D[c][b])
// rescale = 1: followed by Ring.DivRoundByLastModulusNTT (ring/scaling.go:101-122), out receiving rows 0..levelQ-1. Only row L = levelQ of
// the ModDown output is formed (a one-row pass into scratch, then its INTT c_L); every other row j takes ONE extension and ONE transform:
//     out_j = ((acc_j - NTT(E_j)) P^-1 + D_j - NTT(ext_L,j)) q_L^-1  =  (acc_j P^-1 + D_j - NTT(P^-1 E_j + ext_L,j)) q_L^-1   (mod q_j)
// with E_j the P -> Q extension and ext_L,j = (c_L + floor(q_L/2)) mod q_L - floor(q_L/2) mod q_j the Rescale broadcast term: the K2 prologue
// PRO_MODUP_BCAST (constants Ctx::muc_PtoQ_pinv) and the RS epilogue. Every step is exact mod q_j, so the output words equal those of the
// two separate passes.
int moddown_ntt_fused(const Ctx* c, int levelQ, int levelP, const u64* acc, size_t acc_cs, size_t acc_bs, const u64* D, size_t d_cs, size_t d_bs,
                      u64* out, size_t o_cs, size_t o_bs, int ncomp, int batch, cudaStream_t st, int rescale) {
    if (rescale && levelQ < 1) { set_error("cannot Rescale at level 0"); return -1; }
    const int nq = levelQ + 1, np = levelP + 1;
    const size_t N = c->N;
    const int Z = ncomp * batch;
    // scratch: INTT of the P rows | y | P1 (one row per output row) | v bytes | rescale: ModDown row L and its INTT
    const size_t bp_words = (size_t)Z * np * N, y_words = bp_words, p1_words = (size_t)Z * (nq - rescale) * N, v_words = ((size_t)Z * N + 7) / 8;
    const size_t l_words = rescale ? 2 * (size_t)Z * N : 0;
    u64* buf = nullptr;
    LGPU_CUDA_OK(cudaMallocAsync((void**)&buf, (bp_words + y_words + p1_words + v_words + l_words) * sizeof(u64), st));
    struct Free { u64* p; cudaStream_t s; ~Free() { cudaFreeAsync(p, s); } } guard{buf, st};
    u64* buffP = buf; u64* Y = buffP + bp_words; u64* P1 = Y + y_words;
    unsigned char* V = reinterpret_cast<unsigned char*>(P1 + p1_words);
    u64* mdL = P1 + p1_words + v_words; u64* cL = mdL + (size_t)Z * N;
    // A: INTT of the P rows
    const RowMap rp = q_rows(c->nQ, np);
    for (int cc = 0; cc < ncomp; cc++) {
        CSpan in{acc + (size_t)cc * acc_cs + (size_t)nq * N, N, acc_bs};
        Span o{buffP + (size_t)cc * batch * np * N, N, (size_t)np * N};
        if (launch_intt(c, rp, in, o, batch, NTT_CANONICAL, st)) return -1;
    }
    // B: y_i, v
    const ModUpSet& m = c->muc_PtoQ[levelP];
    KsPrepParams pp;
    memset(&pp, 0, sizeof(pp));
    pp.limbs = c->d_limbs; pp.cx = buffP; pp.cx_rs = N; pp.cx_bs = (size_t)np * N;
    pp.Y = Y; pp.y_bs = (size_t)np * N; pp.V = V; pp.v_bs = N;
    pp.nq = np; pp.nd = 1; pp.k = np; pp.n = c->N; pp.limb0 = c->nQ; pp.single_rule = 0;
    for (int i = 0; i < np; i++) { pp.half_src[i] = c->h_blob[m.off_half_s + i]; pp.cinv[i] = c->h_blob[m.off_qoverqiinvqi + i]; }
    {
        ProfScope ps(LGPU_KCLASS_MODUP, st, 8.0 * N * Z * (2.0 * np), 1);
        ks_prepare_kernel<<<dim3((unsigned)((N + 255) / 256), Z), 256, 0, st>>>(pp);
        LGPU_CUDA_OK(cudaGetLastError());
    }
    // C: basis extension folded into the strided pass, then the chunk-pass epilogue
    KsStridedParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.limbs = c->d_limbs; sp.blob = c->d_blob; sp.Y = Y; sp.y_bs = (size_t)np * N; sp.V = V; sp.v_bs = N;
    sp.logN = c->logN; sp.k = np; sp.nd = 1; sp.skip_own = 0; sp.single_rule = 0; sp.src_limb0 = c->nQ; sp.split23 = k2_split();
    auto set_digit = [&](const ModUpSet& s) {
        sp.dg[0].nS = (unsigned short)np; sp.dg[0].ldc = (unsigned short)s.nS;
        sp.dg[0].off_c = (unsigned)s.off_qoverqimodp; sp.dg[0].off_vt = (unsigned)s.off_vtimesqmodp; sp.dg[0].off_half_t = (unsigned)s.off_half_t;
        sp.dg[0].off_cp = (unsigned)s.off_c_plain;
        bool fps = true;
        for (int j = 0; j < np; j++) fps = fps && c->h_limbs[c->nQ + j].fp_ok;
        sp.dg[0].fp_src = fps ? (unsigned short)(1 + k2_fpsum()) : 0;
    };
    set_digit(m);
    FzChunkParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.limbs = c->d_limbs; cp.nb = batch; cp.logN = c->logN;
    const u64* mdc = &c->mdc_PtoQ[(size_t)levelP * c->nQ];
    auto md_consts = [&](const RowMap& rm) { for (int r = 0; r < rm.nrows; r++) { const int i = rm.limb[r]; cp.s[r] = c->Q[i] - mdc[i]; } };
    const double md_words = D ? 4.0 : 3.0;      // P1 + accumulator (+ D) read, out written
    if (!rescale) {
        sp.P1 = P1; sp.p1_ds = sp.p1_bs = (size_t)nq * N; sp.nq = nq;
        cp.P1 = P1; cp.p1_bs = (size_t)nq * N;
        cp.A = acc; cp.a_cs = acc_cs; cp.a_bs = acc_bs; cp.D = D; cp.d_cs = d_cs; cp.d_bs = d_bs;
        cp.out = out; cp.o_cs = o_cs; cp.o_bs = o_bs;
        return fz_tail<PRO_MODUP, false>(c, q_rows(0, nq), np, sp, cp, Z, md_words, md_consts, st);
    }
    const int L = levelQ;
    // C1: ModDown of row L alone into mdL [Z][N] (launch row 0: the row offsets are folded into the pointers), then c_L = INTT(mdL)
    RowMap rl;
    rl.nrows = 1; rl.limb[0] = (unsigned char)L; rl.drow[0] = 0;
    sp.P1 = P1; sp.p1_ds = sp.p1_bs = N; sp.nq = 1;
    cp.P1 = P1; cp.p1_bs = N;
    cp.A = acc + (size_t)L * N; cp.a_cs = acc_cs; cp.a_bs = acc_bs;
    cp.D = D ? D + (size_t)L * N : nullptr; cp.d_cs = d_cs; cp.d_bs = d_bs;
    cp.out = mdL; cp.o_cs = (size_t)batch * N; cp.o_bs = N;
    if (fz_tail<PRO_MODUP, false>(c, rl, np, sp, cp, Z, md_words, md_consts, st)) return -1;
    if (launch_intt(c, rl, CSpan{mdL, N, N}, Span{cL, N, N}, Z, NTT_CANONICAL, st)) return -1;
    // C2: rows 0..L-1, one extension (P^-1 E_j + ext_L,j) and one transform each, straight into out
    const u64 qL = c->Q[L];
    const u64 pHalf = (qL - 1) >> 1;
    set_digit(c->muc_PtoQ_pinv[levelP]);
    sp.P1 = P1; sp.p1_ds = sp.p1_bs = (size_t)L * N; sp.nq = L;
    sp.bc = cL; sp.bc_bs = N; sp.bc_add = pHalf; sp.bc_q = qL;
    cp.P1 = P1; cp.p1_bs = (size_t)L * N;
    cp.A = acc; cp.D = D;
    cp.out = out; cp.o_cs = o_cs; cp.o_bs = o_bs;
    const u64* resc = &c->rescaleQ[(size_t)(L - 1) * c->nQ];
    auto rs_consts = [&](const RowMap& rm) {
        for (int r = 0; r < rm.nrows; r++) {
            const int i = rm.limb[r];
            const u64 qi = c->Q[i];
            sp.s0[r] = qi - (pHalf % qi);
            cp.s[r] = resc[i];
            // MForm(P^-1 q_L^-1) = MForm(P^-1) * (-RescaleConstant) * 2^-64: both are Montgomery forms
            cp.s2[r] = h_mulmod(h_mulmod(mdc[i], (qi - resc[i]) % qi, qi), h_invmod(h_mform(1, qi), qi), qi);
        }
    };
    return fz_tail<PRO_MODUP_BCAST, true>(c, q_rows(0, L), np, sp, cp, Z, md_words, rs_consts, st);
}

// Fused Ring.DivRoundByLastModulusNTT (ring/scaling.go:101-122) for ncomp x batch polynomials at level `level`:
// X rows 0..level -> out rows 0..level-1.
int div_round_last_ntt_fused(const Ctx* c, int level, const u64* X, size_t x_cs, size_t x_bs, u64* out, size_t o_cs, size_t o_bs,
                             int ncomp, int batch, cudaStream_t st) {
    const size_t N = c->N;
    const int Z = ncomp * batch;
    u64* buf = nullptr;
    LGPU_CUDA_OK(cudaMallocAsync((void**)&buf, ((size_t)Z * N + (size_t)Z * level * N) * sizeof(u64), st));
    struct Free { u64* p; cudaStream_t s; ~Free() { cudaFreeAsync(p, s); } } guard{buf, st};
    u64* r = buf; u64* P1 = buf + (size_t)Z * N;
    RowMap rl;
    rl.nrows = 1; rl.limb[0] = (unsigned char)level; rl.drow[0] = 0;
    for (int cc = 0; cc < ncomp; cc++) {
        CSpan in{X + (size_t)cc * x_cs + (size_t)level * N, N, x_bs};
        Span o{r + (size_t)cc * batch * N, N, N};
        if (launch_intt(c, rl, in, o, batch, NTT_CANONICAL, st)) return -1;
    }
    const u64 qL = c->Q[level];
    const u64 pHalf = (qL - 1) >> 1;
    KsStridedParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.limbs = c->d_limbs; sp.blob = c->d_blob; sp.P1 = P1; sp.p1_ds = (size_t)level * N; sp.p1_bs = (size_t)level * N;
    sp.logN = c->logN; sp.nq = level; sp.k = 1; sp.nd = 1;
    sp.bc = r; sp.bc_bs = N; sp.bc_add = pHalf; sp.bc_q = qL;
    FzChunkParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.limbs = c->d_limbs; cp.P1 = P1; cp.p1_bs = (size_t)level * N;
    cp.A = X; cp.a_cs = x_cs; cp.a_bs = x_bs; cp.D = nullptr;
    cp.out = out; cp.o_cs = o_cs; cp.o_bs = o_bs; cp.nb = batch; cp.logN = c->logN;
    auto consts = [&](const RowMap& rm) {
        for (int k = 0; k < rm.nrows; k++) {
            const u64 qi = c->Q[rm.drow[k]];
            sp.s0[k] = qi - (pHalf % qi);
            cp.s[k] = c->rescaleQ[(size_t)(level - 1) * c->nQ + rm.drow[k]];
        }
    };
    return fz_tail<PRO_BCAST, false>(c, q_rows(0, level), 1, sp, cp, Z, 3.0, consts, st);
}

}  // namespace lgpu
