// engine.h -- host-side structures of the B200 RNS ring engine (C++ mirror of the reference's
// ring.Ring / ring.BasisExtender / ring.Decomposer / rlwe.Evaluator state for the hot path).
//
// Data layout in HBM: a polynomial is a contiguous (limb, coeff) row-major block of uint64,
// row stride >= N words (ring/poly.go:13-15 keeps one Go slice per limb; the cgo shim makes those
// slices views of the rows of one such block). Batches are arrays of polynomials with a constant
// batch stride. Constants live once per context in device memory (LimbConst table + root tables +
// basis-extension matrices) and are addressed through a "global limb index": Q limbs 0..nQ-1 followed
// by P limbs nQ..nQ+nP-1, so that one kernel launch can cover the Q and P parts of a ringqp.Poly.
#pragma once
#include <cstddef>
#include <cstdint>
#include <mutex>
#include <string>
#include <vector>
#include <cuda_runtime.h>

typedef unsigned long long u64;

namespace lgpu {

constexpr int kMaxRows = 128;  // max limbs (rows) handled by one launch

// Per-limb device constants. ring/subring.go:15-35 + ring/ntt.go:38-44.
struct LimbConst {
    u64 q;        // Modulus
    u64 qinv;     // MRedConstant = q^-1 mod 2^64
    u64 bred_hi;  // BRedConstant[0]
    u64 bred_lo;  // BRedConstant[1]
    u64 ninv;     // NInv = MForm(N^-1 mod q)
    const u64* roots_fwd;  // RootsForward  (device, NthRoot/2 entries)
    const u64* roots_bwd;  // RootsBackward (device)
    // ---- free-form fast path (canonical outputs only; see ntt.cu) ----
    const ulonglong2* tw_fwd;  // {psi^j, floor(psi^j * 2^64 / q)} (plain, not Montgomery), same bit-reversed indexing
    const ulonglong2* tw_bwd;  // {psi^-j, floor(.)}
    ulonglong2 ninv_s;         // {N^-1, floor(N^-1 * 2^64 / q)}
    ulonglong2 last_inv_s;     // {psi^-(N/2)... = tw_bwd[1] * N^-1, floor(.)}: last inverse stage with the scaling folded in
    u64 kq;                    // K*q, K the largest power of two with K*q <= 2^63 (forward lazy correction)
    unsigned int fwd_mask;     // bit s: correct U (if U >= kq: U -= kq) before stage s of the forward transform
    unsigned int inv_lazy;     // 1: q * 2^(logN+1) < 2^64 -> the inverse transform needs no per-stage correction
    // ---- FP64-pipe path (ntt_fp64.cu), primes below ~2^46 ----
    unsigned int fp_ok;        // 1: (10 + logN) * q < 2^51 -> exact FP64 butterflies are valid for this prime
    double fq, fqinv;          // q and fl(1/q)
    double fninv, flast_inv;   // N^-1 mod q and psi_bwd[1] * N^-1 mod q as doubles
    const double* ftw_fwd;     // psi^j as doubles (same bit-reversed indexing as roots_fwd)
    const double* ftw_bwd;
};

// Which global limb each row of a launch uses.
struct RowMap {
    int nrows;
    unsigned char limb[kMaxRows];  // global limb index of launch row r
    unsigned char drow[kMaxRows];  // data row (within the polynomial) of launch row r
};

struct HostSubRing {
    u64 q, qinv, bred_hi, bred_lo, ninv, primitive_root;
    std::vector<u64> roots_fwd, roots_bwd;  // host copies (also returned through the C ABI for cross-checks)
    u64* d_tw = nullptr;                    // device: tw_fwd (2*half words) followed by tw_bwd
};

// ring.ModUpConstants for a (source chain, target chain) pair -- ring/basis_extension.go:90-98.
// Device layout: qoverqiinvqi[nS] | qoverqimodp[nT][nS] | vtimesqmodp[nT][nS+1], offsets into the blob.
struct ModUpSet {
    int nS = 0, nT = 0;
    size_t off_qoverqiinvqi = 0, off_qoverqimodp = 0, off_vtimesqmodp = 0;
    size_t off_half_s = 0, off_half_t = 0;  // floor(S/2) mod s_i (nS words) and mod t_j (nT words), S = prod(sources)
    size_t off_c_plain = 0;                 // (S/s_i mod t_j) NOT in Montgomery form, [nT][nS] (FP64 basis extension)
};

struct Ctx {
    int device = 0;
    int logN = 0, N = 0;
    int ring_type = 0;  // 0 = Standard, 1 = ConjugateInvariant
    u64 nthroot = 0;
    int nQ = 0, nP = 0;
    std::vector<u64> Q, P;
    std::vector<HostSubRing> sub;  // nQ + nP (global limb index)
    // device tables
    LimbConst* d_limbs = nullptr;
    u64* d_roots = nullptr;        // 2 * (nQ+nP) * (nthroot/2) words
    u64* d_tw = nullptr;           // Shoup twiddle pairs: 4 * (nQ+nP) * (nthroot/2) words
    double* d_ftw = nullptr;       // FP64 twiddles: 2 * (nQ+nP) * (nthroot/2) doubles
    std::vector<LimbConst> h_limbs;
    // rescale constants, ring/ring.go:329-346: rescale[(j-1)*nQ + i] = MForm(q_i - q_j^-1 mod q_i)  (Q ring)
    std::vector<u64> rescaleQ, rescaleP;
    // basis-extension constant blob (host mirror + device)
    std::vector<u64> h_blob;
    u64* d_blob = nullptr;
    std::vector<ModUpSet> muc_QtoP;  // [levelQ]: Q[:levelQ+1] -> P (all)
    std::vector<ModUpSet> muc_PtoQ;  // [levelP]: P[:levelP+1] -> Q (all)
    // [levelP]: muc_PtoQ with every target-side constant (qoverqimodp, vtimesqmodp, half_t, c_plain) multiplied by
    // P^-1 mod q_j, P = p_0..p_levelP; source-side offsets are those of muc_PtoQ. The extension it evaluates is P^-1 ModUp(x)
    // (used by the ModDown + Rescale tail, which needs that product and nothing else)
    std::vector<ModUpSet> muc_PtoQ_pinv;
    // decomposer sets, ring/basis_extension.go:333-373: index (nbPi-2, digit, decompLvl)
    std::vector<std::vector<std::vector<ModUpSet>>> muc_dec;
    // modDownConstants: [levelP][i] (PtoQ) and [levelQ][j] (QtoP), Montgomery form  (:25-49)
    std::vector<u64> mdc_PtoQ, mdc_QtoP;
    // half-moduli: floor(Q_l/2) mod q_i, mod p_j etc. are computed on the fly from prefix products
    cudaStream_t stream = nullptr;  // default stream of the context
    // scratch arena (device), grown on demand; used by composite ops (ModDown, GadgetProduct, ...)
    u64* d_scratch = nullptr;
    size_t scratch_words = 0;
    // automorphism index cache: galEl -> device index table (u32[N])
    std::vector<std::pair<u64, unsigned int*>> auto_index;
    // staging state of the *_host entry points, created on first use and kept for the life of the context (allocating
    // and freeing ~2 GB of device staging per call was a visible, noisy part of the end-to-end time)
    struct HostPipe {
        static constexpr int kStreams = 3;   // capacity; two are used by default (capi2.cu)
        cudaStream_t st[kStreams] = {nullptr, nullptr, nullptr};
        u64* buf[kStreams][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};   // [stream][A, B, out]
        size_t cap[3] = {0, 0, 0};                                                       // words per buffer kind
        std::mutex mu;                                                                   // one host-pipeline call at a time PER CONTEXT (contexts on other GPUs run concurrently)
    } host_pipe;
};

// 128-bit vector accesses need 16-byte aligned bases and even strides (in words); callers that hand in odd row offsets
// are routed to the 64-bit kernels instead.
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool even_words(size_t a, size_t b = 0, size_t c = 0) { return ((a | b | c) & 1u) == 0; }

// ---- error handling --------------------------------------------------------------------------------
void set_error(const std::string& msg);
const char* last_error();
#define LGPU_CUDA_OK(expr)                                                                       \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            lgpu::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                 \
            return -1;                                                                           \
        }                                                                                        \
    } while (0)

// ---- host number theory (tables.cu) ------------------------------------------------------------------
u64 h_mulmod(u64 a, u64 b, u64 m);
u64 h_powmod(u64 a, u64 e, u64 m);
u64 h_invmod(u64 a, u64 m);  // m prime
bool h_is_prime(u64 n);
u64 h_mform(u64 a, u64 q);   // a * 2^64 mod q
int build_context(Ctx* c, int device, int logN, int ring_type, const u64* q, int nq, const u64* p, int np);
void destroy_context(Ctx* c);
int ensure_scratch(Ctx* c, size_t words);
// (re)derives the fast-path tables of global limb g from its Montgomery root tables and uploads them
int upload_limb_tables(Ctx* c, int g);
// half modulus of the product of `mods[0..n)` reduced mod m: floor(prod/2) mod m
u64 h_half_prod_mod(const u64* mods, int n, u64 m);

// ---- launchers (ntt.cu / vecops.cu / basisext.cu / keyswitch.cu) ---------------------------------------
// All launchers are asynchronous on `st`. rows: RowMap; data: base pointer, row stride, batch count/stride.
struct Span {
    u64* p;
    size_t row_stride;    // words between consecutive rows (limbs)
    size_t batch_stride;  // words between consecutive batch elements
};
struct CSpan {
    const u64* p;
    size_t row_stride;
    size_t batch_stride;
};

enum NttMode { NTT_CANONICAL = 0, NTT_EXACT_LAZY = 1, NTT_REFERENCE_ARITH = 2 };

int launch_ntt(const Ctx* c, const RowMap& rm, CSpan in, Span out, int batch, int mode, cudaStream_t st);
int launch_intt(const Ctx* c, const RowMap& rm, CSpan in, Span out, int batch, int mode, cudaStream_t st);

int launch_vecop(const Ctx* c, const RowMap& rm, int op, CSpan p1, CSpan p2, Span p3, int batch,
                 const u64* h_s0, const u64* h_s1, u64 s0, u64 s1, int n, cudaStream_t st);

// ntt_fp64.cu
bool fp64_ntt_supported(const Ctx* c);
// conjugate-invariant ring (ntt_ci.cu); lazy selects NTTConjugateInvariantLazy / INTTConjugateInvariantLazy
int launch_ntt_ci(const Ctx* c, const RowMap& rm, bool inverse, CSpan in, Span out, int batch, int lazy, cudaStream_t st);
int launch_ntt_fp64(const Ctx* c, const RowMap& rm, bool inverse, CSpan in, Span out, int batch, cudaStream_t st);

// ntt_persist.cu: single-launch, single-HBM-pass transforms (2^13 <= N <= 2^16); kind 0 = FP64-pipe rows, 1 / 2 = integer rows
bool ntt_persist_supported(const Ctx* c, bool inverse);
int launch_ntt_persist(const Ctx* c, const RowMap& rm, bool inverse, int kind, CSpan in, Span out, int batch, cudaStream_t st,
                       CSpan mul = CSpan{nullptr, 0, 0});
// Ring.NTT followed by Ring.MulCoeffsMontgomery(., other, out) (ring/ntt.go:127-131 + ring/operations.go:88-92): fused into the
// transform's last pass where the persistent kernels apply, two launches otherwise (ntt.cu)
int launch_ntt_mul_montgomery(const Ctx* c, const RowMap& rm, CSpan in, CSpan other, Span out, int batch, cudaStream_t st);

// basisext.cu
int launch_modup_qp(const Ctx* c, bool toP, int levelQ, int levelP, CSpan in, Span out, int batch, cudaStream_t st);
int launch_decompose_and_split(const Ctx* c, int levelQ, int levelP, int nbPi, int digit, CSpan p0Q, Span p1Q, Span p1P,
                               int batch, cudaStream_t st);

bool profiling_on();   // event profiler active: kernel chains are kept on ONE stream so that class times do not overlap
// prof.cu: launch accounting + optional event profiling (kernel classes = LGPU_KCLASS_* of the public header)
void count_launch(int n);
class ProfScope {
  public:
    ProfScope(int kclass, cudaStream_t st, double alg_bytes, int kernels);
    ~ProfScope();
  private:
    int k_; cudaStream_t st_; bool on_; double bytes_; int kernels_;
    cudaEvent_t a_ = nullptr, b_ = nullptr;
};

// capi.cu helpers
int make_rowmap(const Ctx& c, int ring, int level, RowMap& rm);
int make_rowmap_single(const Ctx& c, int ring, int limb, RowMap& rm);

}  // namespace lgpu
