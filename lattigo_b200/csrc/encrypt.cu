// encrypt.cu -- the encryptor / key-generator inner loops and the samplers on the device (SURVEY 8(f) rank 3).
//
// Deterministic part (bit-exact with the reference given the same sampled polynomials; restated for tests in oracle/encryptor.py):
//   Encryptor.encryptZeroPk (Element[ring.Poly])          core/rlwe/encryptor.go:204-299
//   Encryptor.encryptZeroPkNoP                            :301-341
//   Encryptor.encryptZeroSkFromC1QP / encryptZeroSk       :346-430
//   KeyGenerator.genEvaluationKey                         core/rlwe/keygenerator.go:287-330
//   AddPolyTimesGadgetVectorToGadgetCiphertext            core/rlwe/gadgetciphertext.go:171-241
//   ringqp.Ring.ExtendBasisSmallNormAndCenter             ring/ringqp/operations.go:325-351 (folded into small_to_rns)
// Samplers (ring/sampler_uniform.go, sampler_ternary.go, sampler_gaussian.go): same DISTRIBUTIONS, own random streams -- the
// reference reads a blake2b XOF sequentially (sampling/prng.go), which has no parallel form; here every coefficient owns a
// Philox4x32-10 counter (seed, stream, sampler kind, polynomial, coefficient, attempt), so a batch of polynomials is sampled in
// one launch and the result does not depend on the launch geometry. tests/sampler_model.py restates these kernels bit for bit.
#include <cmath>
#include <cstring>
#include <vector>
#include "../../include/lattigo_b200.h"
#include "capi_common.h"
#include "composite.h"
#include "modarith.cuh"

namespace lgpu {

// ---------------------------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11): counter-based, 128-bit counter, 64-bit key
// ---------------------------------------------------------------------------------------------------------------------
struct Ph4 { unsigned x, y, z, w; };
__device__ __forceinline__ Ph4 philox4x32_10(Ph4 c, unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = Ph4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c;
}
// Counter layout {coefficient or draw index, kind << 30 | polynomial, low half of the stream id, attempt} under the key
// (seed, high half of the stream id): every (seed, stream id, sampler kind, polynomial) has its own counter space, so no two
// samplers, rings or batch elements ever read the same block. polynomial < 2^30: batch * kMaxRows + limb for the uniform
// sampler, the batch index otherwise.
enum SampleKind : unsigned { kUniform = 0, kTernaryP = 1, kTernaryH = 2, kGaussian = 3 };
struct SampleKey { unsigned k0, k1, stream, kind; };
__device__ __forceinline__ Ph4 draw(const SampleKey& k, unsigned poly, unsigned coeff, unsigned attempt) {
    return philox4x32_10(Ph4{coeff, k.kind << 30 | poly, k.stream, attempt}, k.k0, k.k1);
}

// uniform in [0, q) per row: masked 64-bit words, rejected until below q (ring/sampler_uniform.go:48-100). A row draws from the
// stream of its global limb (Q limbs, then P limbs), so the Q and P rows of one stream id differ and a row does not depend on
// the level it is drawn at.
struct UniformParams {
    const LimbConst* limbs; RowMap rm;
    u64* out; size_t rs, bs;
    SampleKey key; int n;
};
__global__ void __launch_bounds__(256) sample_uniform_kernel(UniformParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const int r = blockIdx.y, b = blockIdx.z;
    const u64 q = p.limbs[p.rm.limb[r]].q;
    const u64 mask = ~0ull >> __clzll((long long)(q - 1));
    const unsigned poly = (unsigned)b * kMaxRows + p.rm.limb[r];
    u64 v = 0;
    for (unsigned a = 0;; a++) {
        const Ph4 d = draw(p.key, poly, (unsigned)i, a);
        v = (((u64)d.x << 32) | d.y) & mask;
        if (v < q) break;
        v = (((u64)d.z << 32) | d.w) & mask;
        if (v < q) break;
    }
    p.out[(size_t)b * p.bs + (size_t)p.rm.drow[r] * p.rs + i] = v;
}

// ternary with P(+-1) = prob / 2 each (ring.Ternary{P}, ring/sampler_ternary.go:136-201)
__global__ void __launch_bounds__(256) sample_ternary_p_kernel(long long* out, int n, double prob, SampleKey key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Ph4 d = draw(key, blockIdx.y, (unsigned)i, 0);
    const double u = ((double)d.x * 4294967296.0 + (double)d.y) * (1.0 / 18446744073709551616.0);
    out[(size_t)blockIdx.y * n + i] = u < prob ? ((d.z & 1u) ? 1 : -1) : 0;
}
// ternary with exactly h non-zero coefficients, uniform positions and signs (ring.Ternary{H}, :203-260): one CTA per polynomial,
// positions drawn by rejection against a bitmap in shared memory
__global__ void __launch_bounds__(256) sample_ternary_h_kernel(long long* out, int n, int h, SampleKey key) {
    extern __shared__ unsigned bitmap[];
    long long* o = out + (size_t)blockIdx.x * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) o[i] = 0;
    for (int i = threadIdx.x; i < (n + 31) / 32; i += blockDim.x) bitmap[i] = 0;
    __syncthreads();
    if (threadIdx.x != 0) return;
    int placed = 0;
    for (unsigned a = 0; placed < h; a++) {
        const Ph4 d = draw(key, blockIdx.x, a, 0);
        const unsigned cand[2] = {d.x & (unsigned)(n - 1), d.z & (unsigned)(n - 1)};
        const unsigned sgn[2] = {d.y & 1u, d.w & 1u};
        for (int t = 0; t < 2 && placed < h; t++) {
            const unsigned pos = cand[t];
            if (bitmap[pos >> 5] & (1u << (pos & 31))) continue;
            bitmap[pos >> 5] |= 1u << (pos & 31);
            o[pos] = sgn[t] ? 1 : -1;
            placed++;
        }
    }
}
// truncated discrete Gaussian: round(|N(0,1)| * sigma) with a random sign, redrawn while |N(0,1)| * sigma > bound
// (ring/sampler_gaussian.go:160-182); the normal deviate comes from Box-Muller on two 53-bit uniforms
__global__ void __launch_bounds__(256) sample_gaussian_kernel(long long* out, int n, double sigma, double bound, SampleKey key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long v = 0;
    for (unsigned a = 0;; a++) {
        const Ph4 d = draw(key, blockIdx.y, (unsigned)i, a);
        const double u1 = ((double)(((u64)d.x << 21) | (d.y >> 11)) + 1.0) * (1.0 / 9007199254740992.0);   // (0, 1]
        const double u2 = (double)(((u64)d.z << 21) | (d.w >> 11)) * (1.0 / 9007199254740992.0);            // [0, 1)
        const double z = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        const double m = fabs(z) * sigma;
        if (m <= bound) {
            v = (long long)(m + 0.5);
            if (d.w & 1u) v = -v;      // bit 0 of d.w is not part of u2
            break;
        }
    }
    out[(size_t)blockIdx.y * n + i] = v;
}

// signed small coefficients -> residues on the launch rows: Sampler.Read on the Q rows followed by ExtendBasisSmallNormAndCenter on
// the P rows leaves exactly v mod q_i / v mod p_j (|v| < q_0 / 2)
struct SmallParams {
    const LimbConst* limbs; RowMap rm;
    const long long* in; size_t in_bs;
    u64* out; size_t rs, bs;
    int n;
};
__global__ void __launch_bounds__(256) small_to_rns_kernel(SmallParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const int r = blockIdx.y, b = blockIdx.z;
    const u64 q = p.limbs[p.rm.limb[r]].q;
    const long long v = p.in[(size_t)b * p.in_bs + i];
    p.out[(size_t)b * p.bs + (size_t)p.rm.drow[r] * p.rs + i] = v < 0 ? q - (u64)(-v) : (u64)v;
}

// AddPolyTimesGadgetVectorToGadgetCiphertext: evk[i][j][0][index] += pt[index] * (P w^j) on the limbs of digit i
struct GadgetAddParams {
    const LimbConst* limbs;
    u64* evk; size_t ds, js;          // digit stride, pw2 stride (words); component 0 first
    const u64* pt;                    // rows 0..levelQ, NTT + Montgomery
    int nq, k, n, npw2;
    const u64* f;                     // device, [index][j]: MForm(P * 2^(pw2 j) mod q_index)
    unsigned char npw2_of_digit[kMaxRows];
};
__global__ void __launch_bounds__(256) gadget_add_kernel(GadgetAddParams p) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= p.n) return;
    const int index = blockIdx.y, j = blockIdx.z;
    const int i = index / p.k;
    if (j >= p.npw2_of_digit[i]) return;
    const LimbConst& L = p.limbs[index];
    u64* dst = p.evk + (size_t)i * p.ds + (size_t)j * p.js + (size_t)index * p.n + w;
    const u64 t = mred(p.pt[(size_t)index * p.n + w], p.f[index * p.npw2 + j], L.q, L.qinv);
    *dst = cred(*dst + t, L.q);
}

static SampleKey make_key(u64 seed, u64 stream, SampleKind kind) {
    SampleKey k;
    k.k0 = (unsigned)seed; k.k1 = (unsigned)(seed >> 32) ^ (unsigned)(stream >> 32) * 0x85EBCA6Bu; k.stream = (unsigned)stream;
    k.kind = kind;
    return k;
}

static int small_to_rns(const Ctx* c, const RowMap& rm, const long long* in, size_t in_bs, Span out, int batch, cudaStream_t st) {
    SmallParams p;
    p.limbs = c->d_limbs; p.rm = rm; p.in = in; p.in_bs = in_bs; p.out = out.p; p.rs = out.row_stride; p.bs = out.batch_stride; p.n = c->N;
    count_launch(1);
    small_to_rns_kernel<<<dim3((c->N + 255) / 256, rm.nrows, batch), 256, 0, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}
static RowMap one_row(int limb) { RowMap r; r.nrows = 1; r.limb[0] = (unsigned char)limb; r.drow[0] = 0; return r; }

// encryptZeroSkFromC1QP (:404-430). sk: rows of the secret key at the context's maximum levels ([nQ + nP][N], NTT + Montgomery).
// c1 / c0: QP-stacked blocks ([levelQ+1 + levelP+1][N]) with the given batch strides; c1 is only rewritten when !is_ntt.
int encrypt_zero_sk(const Ctx* c, int levelQ, int levelP, const u64* sk, u64* c1, size_t c1_bs, const long long* e, u64* c0, size_t c0_bs,
                    bool is_ntt, bool is_mont, int batch, cudaStream_t st) {
    if (levelQ < 0 || levelQ >= c->nQ || levelP < -1 || levelP >= c->nP) { set_error("level out of range"); return -1; }
    const size_t N = c->N;
    const int nq = levelQ + 1, np = levelP + 1;
    const RowMap rqp = rows_qp(c, nq, np);
    Span s0{c0, N, c0_bs};
    if (small_to_rns(c, rqp, e, N, s0, batch, st)) return -1;
    if (launch_ntt(c, rqp, CSpan{c0, N, c0_bs}, s0, batch, NTT_CANONICAL, st)) return -1;
    if (is_mont && launch_vecop(c, rqp, LGPU_OP_MFORM, CSpan{c0, N, c0_bs}, CSpan{nullptr, 0, 0}, s0, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    // c0 -= c1 * sk: Q rows, then P rows (the key's P rows start at row nQ)
    if (launch_vecop(c, rows_range(0, 0, nq), LGPU_OP_MULCOEFFSMONTGOMERYTHENSUB, CSpan{c1, N, c1_bs}, CSpan{sk, N, 0}, s0, batch, nullptr, nullptr, 0, 0,
                     c->N, st)) return -1;
    if (np > 0 && launch_vecop(c, rows_range(c->nQ, 0, np), LGPU_OP_MULCOEFFSMONTGOMERYTHENSUB, CSpan{c1 + (size_t)nq * N, N, c1_bs},
                               CSpan{sk + (size_t)c->nQ * N, N, 0}, Span{c0 + (size_t)nq * N, N, c0_bs}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    if (!is_ntt) {
        if (launch_intt(c, rqp, CSpan{c0, N, c0_bs}, s0, batch, NTT_CANONICAL, st)) return -1;
        if (launch_intt(c, rqp, CSpan{c1, N, c1_bs}, Span{c1, N, c1_bs}, batch, NTT_CANONICAL, st)) return -1;
    }
    return 0;
}

// encryptZeroPk for an Element[ring.Poly] (:204-299; levelP = 0 there) and encryptZeroPkNoP (:301-341) when the context has no P.
// pk: [2][nQ + nP][N] (rlwe.PublicKey.Value at the maximum levels); u, e0, e1: [batch][N] signed; ct_out: [batch][2][levelQ+1][N].
int encrypt_zero_pk(const Ctx* c, int levelQ, const u64* pk, const long long* u, const long long* e0, const long long* e1, u64* ct_out,
                    bool is_ntt, bool is_mont, int batch, cudaStream_t st) {
    if (levelQ < 0 || levelQ >= c->nQ) { set_error("level out of range"); return -1; }
    const size_t N = c->N;
    const int nq = levelQ + 1;
    const size_t key_rows = (size_t)c->nQ + c->nP, ct_bs = (size_t)2 * nq * N;
    const RowMap rq = rows_range(0, 0, nq);
    const long long* es[2] = {e0, e1};
    if (c->nP == 0) {
        if (is_mont) { set_error("encryptZeroPkNoP has no Montgomery-form output"); return -1; }
        Scratch buf;
        if (buf.alloc((size_t)2 * batch * nq * N, st)) return -1;
        u64* U = buf.p; u64* E = buf.p + (size_t)batch * nq * N;
        if (small_to_rns(c, rq, u, N, Span{U, N, nq * N}, batch, st)) return -1;
        if (launch_ntt(c, rq, CSpan{U, N, nq * N}, Span{U, N, nq * N}, batch, NTT_CANONICAL, st)) return -1;
        for (int k = 0; k < 2; k++) {
            Span o{ct_out + (size_t)k * nq * N, N, ct_bs};
            if (launch_vecop(c, rq, LGPU_OP_MULCOEFFSMONTGOMERY, CSpan{U, N, nq * N}, CSpan{pk + (size_t)k * key_rows * N, N, 0}, o, batch, nullptr, nullptr, 0, 0,
                             c->N, st)) return -1;
            if (small_to_rns(c, rq, es[k], N, Span{E, N, nq * N}, batch, st)) return -1;
            if (is_ntt) { if (launch_ntt(c, rq, CSpan{E, N, nq * N}, Span{E, N, nq * N}, batch, NTT_CANONICAL, st)) return -1; }
            else if (launch_intt(c, rq, CSpan{o.p, N, ct_bs}, o, batch, NTT_CANONICAL, st)) return -1;
            if (launch_vecop(c, rq, LGPU_OP_ADD, CSpan{o.p, N, ct_bs}, CSpan{E, N, nq * N}, o, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
        }
        return 0;
    }
    const int levelP = 0, np = 1;
    const RowMap rqp = rows_qp(c, nq, np);
    const size_t qp = (size_t)(nq + np) * N;
    Scratch buf;
    if (buf.alloc((size_t)3 * batch * qp, st)) return -1;
    u64* U = buf.p; u64* C = U + (size_t)batch * qp; u64* E = C + (size_t)batch * qp;
    if (small_to_rns(c, rqp, u, N, Span{U, N, qp}, batch, st)) return -1;
    if (launch_ntt(c, rqp, CSpan{U, N, qp}, Span{U, N, qp}, batch, NTT_CANONICAL, st)) return -1;
    for (int k = 0; k < 2; k++) {
        const u64* pkk = pk + (size_t)k * key_rows * N;
        if (launch_vecop(c, rq, LGPU_OP_MULCOEFFSMONTGOMERY, CSpan{U, N, qp}, CSpan{pkk, N, 0}, Span{C, N, qp}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
        if (launch_vecop(c, one_row(c->nQ), LGPU_OP_MULCOEFFSMONTGOMERY, CSpan{U + (size_t)nq * N, N, qp}, CSpan{pkk + (size_t)c->nQ * N, N, 0},
                         Span{C + (size_t)nq * N, N, qp}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
        if (launch_intt(c, rqp, CSpan{C, N, qp}, Span{C, N, qp}, batch, NTT_CANONICAL, st)) return -1;
        if (small_to_rns(c, rqp, es[k], N, Span{E, N, qp}, batch, st)) return -1;
        if (launch_vecop(c, rqp, LGPU_OP_ADD, CSpan{C, N, qp}, CSpan{E, N, qp}, Span{C, N, qp}, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
        Span o{ct_out + (size_t)k * nq * N, N, ct_bs};
        if (moddown_qp_to_q(c, levelQ, levelP, CSpan{C, N, qp}, CSpan{C + (size_t)nq * N, N, qp}, o, batch, st)) return -1;
        if (is_ntt && launch_ntt(c, rq, CSpan{o.p, N, ct_bs}, o, batch, NTT_CANONICAL, st)) return -1;
        if (is_mont && launch_vecop(c, rq, LGPU_OP_MFORM, CSpan{o.p, N, ct_bs}, CSpan{nullptr, 0, 0}, o, batch, nullptr, nullptr, 0, 0, c->N, st)) return -1;
    }
    return 0;
}

// KeyGenerator.genEvaluationKey (keygenerator.go:287-330) at the maximum levels: on entry component 1 of every evk[i][j] holds the
// uniform polynomial `a` (QP rows, NTT domain); on return component 0 = -a sk_out + e_ij + P w^j sk_in on the limbs of digit i.
int gen_evaluation_key(const Ctx* c, int pw2, const u64* sk_in, const u64* sk_out, u64* evk, int n_digits, int n_pw2_max, const int* pw2_sizes,
                       const long long* e, cudaStream_t st) {
    const int levelQ = c->nQ - 1, levelP = c->nP - 1;
    const size_t N = c->N, rows = (size_t)c->nQ + c->nP;
    const int nd = levelP >= 0 ? base_rns_decomposition_vector_size(levelQ, levelP) : levelQ + 1;
    if (n_digits != nd) { set_error("evaluation key: n_digits != BaseRNSDecompositionVectorSize(levelQ, levelP)"); return -1; }
    if (n_pw2_max < 1 || n_pw2_max > 64) { set_error("evaluation key: n_pw2_max out of [1, 64]"); return -1; }
    if (pw2 < 0 || pw2 > 62) { set_error("evaluation key: BaseTwoDecomposition out of [0, 62]"); return -1; }
    for (int i = 0; pw2_sizes && i < n_digits; i++)
        if (pw2_sizes[i] < 1 || pw2_sizes[i] > n_pw2_max) { set_error("evaluation key: pw2_sizes[i] out of [1, n_pw2_max]"); return -1; }
    const int entries = n_digits * n_pw2_max;
    const size_t ebs = 2 * rows * N;
    if (encrypt_zero_sk(c, levelQ, levelP, sk_out, evk + rows * N, ebs, e, evk, ebs, true, true, entries, st)) return -1;
    GadgetAddParams p;
    memset(&p, 0, sizeof(p));
    p.limbs = c->d_limbs; p.evk = evk; p.ds = (size_t)n_pw2_max * ebs; p.js = ebs; p.pt = sk_in;
    p.nq = c->nQ; p.k = levelP >= 0 ? levelP + 1 : 1; p.n = c->N; p.npw2 = n_pw2_max;
    for (int i = 0; i < n_digits; i++) p.npw2_of_digit[i] = (unsigned char)(pw2_sizes ? pw2_sizes[i] : n_pw2_max);
    std::vector<u64> hf((size_t)c->nQ * n_pw2_max);
    for (int idx = 0; idx < c->nQ; idx++) {
        const u64 q = c->Q[idx];
        u64 f = 1;
        for (int j = 0; j <= levelP; j++) f = h_mulmod(f, c->P[j] % q, q);
        for (int j = 0; j < n_pw2_max; j++) {
            hf[(size_t)idx * n_pw2_max + j] = h_mform(f, q);
            f = h_mulmod(f, (1ull << pw2) % q, q);
        }
    }
    Scratch fbuf;
    if (fbuf.alloc(hf.size(), st)) return -1;
    LGPU_CUDA_OK(cudaMemcpyAsync(fbuf.p, hf.data(), hf.size() * sizeof(u64), cudaMemcpyHostToDevice, st));   // pageable source: staged before return
    p.f = fbuf.p;
    count_launch(1);
    gadget_add_kernel<<<dim3((c->N + 255) / 256, c->nQ, n_pw2_max), 256, 0, st>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace lgpu

using namespace lgpu;

extern "C" {

int lgpu_sample_uniform(lgpu_ctx* ctx, int ring, int level, uint64_t seed, uint64_t stream_id, uint64_t* out, int batch, size_t batch_stride, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(out && batch >= 1 && batch <= 65535, "bad argument");
    UniformParams p;
    if (make_rowmap(ctx->c, ring, level, p.rm)) return -1;
    p.limbs = ctx->c.d_limbs; p.out = (u64*)out; p.rs = ctx->c.N; p.bs = batch_stride; p.key = make_key(seed, stream_id, kUniform); p.n = ctx->c.N;
    count_launch(1);
    sample_uniform_kernel<<<dim3((ctx->c.N + 255) / 256, p.rm.nrows, batch), 256, 0, (cudaStream_t)stream>>>(p);
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

int lgpu_sample_ternary(lgpu_ctx* ctx, double p, int hamming_weight, uint64_t seed, uint64_t stream_id, int64_t* out, int batch, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(out && batch >= 1 && batch <= 65535, "bad argument");
    const int N = ctx->c.N;
    count_launch(1);
    if (hamming_weight > 0) {
        REQUIRE(hamming_weight <= N, "ternary sampler: Hamming weight above N");
        const size_t smem = (size_t)((N + 31) / 32) * sizeof(unsigned);
        sample_ternary_h_kernel<<<batch, 256, smem, (cudaStream_t)stream>>>((long long*)out, N, hamming_weight, make_key(seed, stream_id, kTernaryH));
    } else {
        REQUIRE(p > 0.0 && p <= 1.0, "ternary sampler: P must be in (0, 1]");
        sample_ternary_p_kernel<<<dim3((N + 255) / 256, batch), 256, 0, (cudaStream_t)stream>>>((long long*)out, N, p, make_key(seed, stream_id, kTernaryP));
    }
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

int lgpu_sample_gaussian(lgpu_ctx* ctx, double sigma, double bound, uint64_t seed, uint64_t stream_id, int64_t* out, int batch, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(out && batch >= 1 && batch <= 65535, "bad argument");
    REQUIRE(sigma > 0.0 && bound >= 1.0 && bound < 9.0e18, "gaussian sampler: sigma / bound out of range");
    const int N = ctx->c.N;
    count_launch(1);
    sample_gaussian_kernel<<<dim3((N + 255) / 256, batch), 256, 0, (cudaStream_t)stream>>>((long long*)out, N, sigma, bound, make_key(seed, stream_id, kGaussian));
    LGPU_CUDA_OK(cudaGetLastError());
    return 0;
}

int lgpu_small_poly_to_rns(lgpu_ctx* ctx, int level_q, int level_p, const int64_t* small, uint64_t* out_q, uint64_t* out_p, int batch, size_t stride_q,
                           size_t stride_p, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(small && (out_q || out_p) && batch >= 1 && batch <= 65535, "bad argument");
    const Ctx& c = ctx->c;
    RowMap rm;
    if (out_q) {
        if (make_rowmap(c, LGPU_RING_Q, level_q, rm)) return -1;
        if (small_to_rns(&c, rm, (const long long*)small, c.N, Span{(u64*)out_q, (size_t)c.N, stride_q}, batch, (cudaStream_t)stream)) return -1;
    }
    if (out_p && level_p >= 0) {
        if (make_rowmap(c, LGPU_RING_P, level_p, rm)) return -1;
        if (small_to_rns(&c, rm, (const long long*)small, c.N, Span{(u64*)out_p, (size_t)c.N, stride_p}, batch, (cudaStream_t)stream)) return -1;
    }
    return 0;
}

int lgpu_encrypt_zero_pk(lgpu_ctx* ctx, int level_q, const uint64_t* pk, const int64_t* u, const int64_t* e0, const int64_t* e1, uint64_t* ct_out,
                         int is_ntt, int is_montgomery, int batch, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(pk && u && e0 && e1 && ct_out, "null argument");
    REQUIRE(batch >= 1 && batch <= 65535, "batch out of range");
    return encrypt_zero_pk(&ctx->c, level_q, (const u64*)pk, (const long long*)u, (const long long*)e0, (const long long*)e1, (u64*)ct_out, is_ntt != 0,
                           is_montgomery != 0, batch, (cudaStream_t)stream);
}

int lgpu_encrypt_zero_sk(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* sk, uint64_t* c1, const int64_t* e, uint64_t* c0, int is_ntt,
                         int is_montgomery, int batch, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(sk && c1 && e && c0, "null argument");
    REQUIRE(batch >= 1 && batch <= 65535, "batch out of range");
    const size_t bs = (size_t)(level_q + 1 + level_p + 1) * ctx->c.N;
    return encrypt_zero_sk(&ctx->c, level_q, level_p, (const u64*)sk, (u64*)c1, bs, (const long long*)e, (u64*)c0, bs, is_ntt != 0, is_montgomery != 0, batch,
                           (cudaStream_t)stream);
}

int lgpu_gen_evaluation_key(lgpu_ctx* ctx, const uint64_t* sk_in, const uint64_t* sk_out, lgpu_gadget_ct* evk, const int64_t* e, void* stream) {
    REQUIRE_DEVICE(ctx);
    REQUIRE(sk_in && sk_out && evk && evk->data && e, "null argument");
    REQUIRE_ALIGNED(AL(evk->data));
    REQUIRE(evk->level_q == ctx->c.nQ - 1 && evk->level_p == ctx->c.nP - 1, "evaluation keys are generated at the maximum levels");
    return gen_evaluation_key(&ctx->c, evk->base_two_decomposition, (const u64*)sk_in, (const u64*)sk_out, (u64*)evk->data, evk->n_digits,
                              evk->n_pw2_max > 0 ? evk->n_pw2_max : 1, evk->pw2_sizes, (const long long*)e, (cudaStream_t)stream);
}

}  // extern "C"
