// tables.cu -- host-side constant generation and context life-cycle.
//
// Regenerates, with 128-bit modular arithmetic only (no big integers), every table the reference
// builds at ring construction time:
//   SubRing constants        ring/subring.go:40-80,99-159   (BRed/MRed constants, NInv, root tables)
//   primitive root choice    ring/subring.go:161-194        (smallest primitive root >= 3)
//   RescaleConstants         ring/ring.go:329-346
//   ModUpConstants           ring/basis_extension.go:101-172
//   modDownConstants         ring/basis_extension.go:25-49
//   Decomposer constants     ring/basis_extension.go:318-377
// The tests cross-check all of them against the oracle's independent big-integer generation.
#include <algorithm>
#include <cstring>
#include <numeric>
#include "engine.h"

namespace lgpu {

typedef unsigned __int128 u128;

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }

u64 h_mulmod(u64 a, u64 b, u64 m) { return (u64)((u128)a * b % m); }
u64 h_powmod(u64 a, u64 e, u64 m) {
    u64 r = 1 % m;
    a %= m;
    while (e) {
        if (e & 1) r = h_mulmod(r, a, m);
        a = h_mulmod(a, a, m);
        e >>= 1;
    }
    return r;
}
u64 h_invmod(u64 a, u64 m) { return h_powmod(a % m, m - 2, m); }
u64 h_mform(u64 a, u64 q) { return (u64)(((u128)a << 64) % q); }

bool h_is_prime(u64 n) {
    if (n < 2) return false;
    static const u64 bases[] = {2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37};
    for (u64 p : bases) {
        if (n % p == 0) return n == p;
    }
    u64 d = n - 1;
    int s = 0;
    while ((d & 1) == 0) { d >>= 1; s++; }
    for (u64 a : bases) {
        u64 x = h_powmod(a, d, n);
        if (x == 1 || x == n - 1) continue;
        bool comp = true;
        for (int i = 1; i < s; i++) {
            x = h_mulmod(x, x, n);
            if (x == n - 1) { comp = false; break; }
        }
        if (comp) return false;
    }
    return true;
}

static u64 pollard_rho(u64 n) {
    if ((n & 1) == 0) return 2;
    for (u64 c = 1;; c++) {
        u64 x = 2, y = 2, d = 1;
        auto f = [&](u64 v) { return (u64)(((u128)v * v + c) % n); };
        while (d == 1) {
            x = f(x);
            y = f(f(y));
            d = std::gcd(x > y ? x - y : y - x, n);
        }
        if (d != n) return d;
    }
}
static void factor_rec(u64 n, std::vector<u64>& out) {
    if (n == 1) return;
    if (h_is_prime(n)) { out.push_back(n); return; }
    for (u64 p : {2ull, 3ull, 5ull, 7ull, 11ull, 13ull}) {
        if (n % p == 0) {
            out.push_back(p);
            while (n % p == 0) n /= p;
            factor_rec(n, out);
            return;
        }
    }
    u64 d = pollard_rho(n);
    factor_rec(d, out);
    factor_rec(n / d, out);
}
// PrimitiveRoot, ring/subring.go:161-194: g = 2; loop { g++; test } -> smallest candidate tested is 3.
static u64 primitive_root(u64 q) {
    std::vector<u64> f;
    factor_rec(q - 1, f);
    std::sort(f.begin(), f.end());
    f.erase(std::unique(f.begin(), f.end()), f.end());
    for (u64 g = 3;; g++) {
        bool ok = true;
        for (u64 p : f) {
            if (h_powmod(g, (q - 1) / p, q) == 1) { ok = false; break; }
        }
        if (ok) return g;
    }
}

static u64 bitrev(u64 x, int bits) {
    u64 r = 0;
    for (int i = 0; i < bits; i++) { r = (r << 1) | ((x >> i) & 1); }
    return r;
}

static int build_subring(HostSubRing& s, u64 q, u64 nthroot) {
    if (!h_is_prime(q)) { set_error("invalid modulus: not prime"); return -1; }
    if ((q & (nthroot - 1)) != 1) { set_error("invalid modulus: != 1 mod NthRoot"); return -1; }
    if (q >> 61) { set_error("invalid modulus: must be < 2^61 (lazy Montgomery ranges, ring/ntt.go:169)"); return -1; }
    s.q = q;
    u128 R = (~(u128)0) / q;  // floor((2^128-1)/q) == floor(2^128/q) since q is odd
    s.bred_hi = (u64)(R >> 64);
    s.bred_lo = (u64)R;
    // q^-1 mod 2^64 (GenMRedConstant, ring/modular_reduction.go:68-75)
    u64 inv = 1, t = q;
    for (int i = 0; i < 63; i++) { inv *= t; t *= t; }
    s.qinv = inv;
    s.primitive_root = primitive_root(q);
    const u64 half = nthroot >> 1;
    int log = 0;
    while ((1ull << log) < half) log++;
    s.ninv = h_mform(h_invmod(half % q, q), q);
    const u64 psi = h_powmod(s.primitive_root, (q - 1) / nthroot, q);
    const u64 psi_inv = h_invmod(psi, q);
    s.roots_fwd.assign(half, 0);
    s.roots_bwd.assign(half, 0);
    u64 cf = 1, cb = 1;
    for (u64 j = 0; j < half; j++) {
        const u64 r = bitrev(j, log);
        s.roots_fwd[r] = h_mform(cf, q);
        s.roots_bwd[r] = h_mform(cb, q);
        cf = h_mulmod(cf, psi, q);
        cb = h_mulmod(cb, psi_inv, q);
    }
    return 0;
}

u64 h_half_prod_mod(const u64* mods, int n, u64 m) {
    // floor(prod/2) mod m with prod odd: (prod - 1) * 2^-1 mod m
    u64 pr = 1 % m;
    for (int i = 0; i < n; i++) pr = h_mulmod(pr, mods[i] % m, m);
    u64 inv2 = (m + 1) >> 1;
    return h_mulmod((pr + m - 1) % m, inv2, m);
}

// GenModUpConstants (ring/basis_extension.go:101-172) appended to the blob.
static ModUpSet gen_modup(std::vector<u64>& blob, const u64* S, int nS, const u64* T, int nT) {
    ModUpSet m;
    m.nS = nS; m.nT = nT;
    m.off_qoverqiinvqi = blob.size();
    for (int i = 0; i < nS; i++) {
        u64 qi = S[i], pr = 1;
        for (int j = 0; j < nS; j++) if (j != i) pr = h_mulmod(pr, S[j] % qi, qi);
        blob.push_back(h_mform(h_invmod(pr, qi), qi));
    }
    m.off_qoverqimodp = blob.size();
    for (int j = 0; j < nT; j++) {
        u64 pj = T[j];
        for (int i = 0; i < nS; i++) {
            u64 pr = 1 % pj;
            for (int u = 0; u < nS; u++) if (u != i) pr = h_mulmod(pr, S[u] % pj, pj);
            blob.push_back(h_mform(pr, pj));
        }
    }
    m.off_vtimesqmodp = blob.size();
    for (int j = 0; j < nT; j++) {
        u64 pj = T[j], pr = 1 % pj;
        for (int i = 0; i < nS; i++) pr = h_mulmod(pr, S[i] % pj, pj);
        u64 v = pj - pr, acc = 0;
        blob.push_back(0);
        for (int i = 1; i < nS + 1; i++) {
            acc += v;
            if (acc >= pj) acc -= pj;
            blob.push_back(acc);
        }
    }
    m.off_half_s = blob.size();
    for (int i = 0; i < nS; i++) blob.push_back(h_half_prod_mod(S, nS, S[i]));
    m.off_half_t = blob.size();
    for (int j = 0; j < nT; j++) blob.push_back(h_half_prod_mod(S, nS, T[j]));
    m.off_c_plain = blob.size();
    for (int j = 0; j < nT; j++) {
        const u64 pj = T[j];
        for (int i = 0; i < nS; i++) {
            u64 pr = 1 % pj;
            for (int u = 0; u < nS; u++) if (u != i) pr = h_mulmod(pr, S[u] % pj, pj);
            blob.push_back(pr);
        }
    }
    return m;
}

// A copy of the target-side constants of `m` multiplied by s[j] mod T[j], appended to the blob. The basis extension is linear in
// them (sum_i y_i (S/s_i mod t_j) - v S - S/2), so the copy evaluates s[j] times the extension.
static ModUpSet scale_modup_targets(std::vector<u64>& blob, const ModUpSet& m, const u64* s, const u64* T) {
    ModUpSet r = m;
    auto scaled = [&](size_t off, int per_target) {
        const size_t out = blob.size();
        for (int j = 0; j < m.nT; j++)
            for (int i = 0; i < per_target; i++) blob.push_back(h_mulmod(blob[off + (size_t)j * per_target + i], s[j], T[j]));
        return out;
    };
    r.off_qoverqimodp = scaled(m.off_qoverqimodp, m.nS);
    r.off_vtimesqmodp = scaled(m.off_vtimesqmodp, m.nS + 1);
    r.off_half_t = scaled(m.off_half_t, 1);
    r.off_c_plain = scaled(m.off_c_plain, m.nS);
    return r;
}

int ensure_scratch(Ctx* c, size_t words) {
    if (words <= c->scratch_words) return 0;
    if (c->d_scratch) {
        LGPU_CUDA_OK(cudaStreamSynchronize(c->stream));
        LGPU_CUDA_OK(cudaFree(c->d_scratch));
        c->d_scratch = nullptr;
        c->scratch_words = 0;
    }
    LGPU_CUDA_OK(cudaMalloc(&c->d_scratch, words * sizeof(u64)));
    c->scratch_words = words;
    return 0;
}

static inline u64 shoup_q(u64 w, u64 q) { return (u64)(((u128)w << 64) / q); }

int upload_limb_tables(Ctx* c, int i) {
    const size_t half = (size_t)(c->nthroot >> 1);
    HostSubRing& s = c->sub[i];
    const u64 q = s.q;
    u64* rf = c->d_roots + (size_t)(2 * i) * half;
    u64* rb = rf + half;
    LGPU_CUDA_OK(cudaMemcpy(rf, s.roots_fwd.data(), half * sizeof(u64), cudaMemcpyHostToDevice));
    LGPU_CUDA_OK(cudaMemcpy(rb, s.roots_bwd.data(), half * sizeof(u64), cudaMemcpyHostToDevice));
    // Shoup pairs derived from the (possibly caller-supplied) Montgomery tables: w = IMForm(root)
    const u64 rinv = h_invmod(h_mform(1, q), q);   // 2^-64 mod q
    std::vector<u64> tw(4 * half);
    for (size_t j = 0; j < half; j++) {
        const u64 wf = h_mulmod(s.roots_fwd[j], rinv, q), wb = h_mulmod(s.roots_bwd[j], rinv, q);
        tw[2 * j] = wf; tw[2 * j + 1] = shoup_q(wf, q);
        tw[2 * half + 2 * j] = wb; tw[2 * half + 2 * j + 1] = shoup_q(wb, q);
    }
    u64* dtw = c->d_tw + (size_t)(4 * i) * half;
    LGPU_CUDA_OK(cudaMemcpy(dtw, tw.data(), tw.size() * sizeof(u64), cudaMemcpyHostToDevice));
    LimbConst& L = c->h_limbs[i];
    L.q = q; L.qinv = s.qinv; L.bred_hi = s.bred_hi; L.bred_lo = s.bred_lo;
    L.ninv = s.ninv; L.roots_fwd = rf; L.roots_bwd = rb;
    L.tw_fwd = reinterpret_cast<const ulonglong2*>(dtw);
    L.tw_bwd = reinterpret_cast<const ulonglong2*>(dtw + 2 * half);
    const u64 ninv = h_mulmod(s.ninv, rinv, q);
    L.ninv_s = make_ulonglong2(ninv, shoup_q(ninv, q));
    const u64 last = h_mulmod(tw[2 * half + 2], ninv, q);   // tw_bwd[1] * N^-1
    L.last_inv_s = make_ulonglong2(last, shoup_q(last, q));
    // forward lazy-correction schedule: values are kept below 2K*q <= 2^64; a stage adds at most 2q.
    u64 K = 1;
    while ((u128)(2 * K) * q <= ((u128)1 << 63)) K *= 2;
    L.kq = K * q;
    unsigned mask = 0;
    u64 b = 2 * K < 8 ? 2 * K : 8;   // assumed input bound (in units of q)
    for (int st = 0; st < c->logN + (c->ring_type ? 1 : 0); st++) {
        if (b + 2 > 2 * K) { mask |= 1u << st; b = K; }
        b += 2;
    }
    L.fwd_mask = mask;
    L.inv_lazy = ((u128)q << (c->logN + 1)) < ((u128)1 << 64) ? 1u : 0u;
    // FP64 path
    L.fp_ok = ((u128)q * (u64)(10 + c->logN) < ((u128)1 << 51)) ? 1u : 0u;
    L.fq = (double)q; L.fqinv = 1.0 / (double)q;
    L.fninv = (double)ninv; L.flast_inv = (double)last;
    double* dft = c->d_ftw + (size_t)(2 * i) * half;
    L.ftw_fwd = dft; L.ftw_bwd = dft + half;
    if (L.fp_ok) {
        std::vector<double> ft(2 * half);
        for (size_t j = 0; j < half; j++) { ft[j] = (double)tw[2 * j]; ft[half + j] = (double)tw[2 * half + 2 * j]; }
        LGPU_CUDA_OK(cudaMemcpy(dft, ft.data(), ft.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    return 0;
}

int build_context(Ctx* c, int device, int logN, int ring_type, const u64* q, int nq, const u64* p, int np) {
    if (logN < 4 || logN > 17) { set_error("invalid ring degree: need 16 <= N <= 2^17"); return -1; }
    if (nq <= 0 || !q) { set_error("invalid ModuliChain (must be non-empty)"); return -1; }
    if (nq + np > kMaxRows) { set_error("too many moduli"); return -1; }
    if (ring_type != 0 && ring_type != 1) { set_error("invalid ring type"); return -1; }
    c->device = device;
    c->logN = logN;
    c->N = 1 << logN;
    c->ring_type = ring_type;
    c->nthroot = (u64)c->N << (ring_type == 0 ? 1 : 2);
    c->nQ = nq;
    c->nP = np;
    c->Q.assign(q, q + nq);
    if (np) c->P.assign(p, p + np);
    {
        std::vector<u64> all(c->Q);
        all.insert(all.end(), c->P.begin(), c->P.end());
        std::sort(all.begin(), all.end());
        if (std::adjacent_find(all.begin(), all.end()) != all.end()) { set_error("invalid ModuliChain (moduli are not distinct)"); return -1; }
    }
    const int nl = nq + np;
    c->sub.resize(nl);
    for (int i = 0; i < nl; i++) {
        if (build_subring(c->sub[i], i < nq ? q[i] : p[i - nq], c->nthroot)) return -1;
    }
    // RescaleConstants, ring/ring.go:329-346
    auto rescale = [&](const std::vector<u64>& M, std::vector<u64>& out) {
        const int n = (int)M.size();
        out.assign((size_t)n * n, 0);
        for (int j = 1; j < n; j++)
            for (int i = 0; i < j; i++)
                out[(size_t)(j - 1) * n + i] = h_mform(M[i] - h_invmod(M[j] % M[i], M[i]), M[i]);
    };
    rescale(c->Q, c->rescaleQ);
    if (np) rescale(c->P, c->rescaleP);

    // basis-extension constants
    c->h_blob.clear();
    if (np) {
        c->muc_QtoP.resize(nq);
        for (int i = 0; i < nq; i++) c->muc_QtoP[i] = gen_modup(c->h_blob, q, i + 1, p, np);
        c->muc_PtoQ.resize(np);
        for (int i = 0; i < np; i++) c->muc_PtoQ[i] = gen_modup(c->h_blob, p, i + 1, q, nq);
        c->muc_PtoQ_pinv.resize(np);
        for (int i = 0; i < np; i++) {
            std::vector<u64> pinv(nq);
            for (int j = 0; j < nq; j++) {
                u64 pr = 1;
                for (int u = 0; u <= i; u++) pr = h_mulmod(pr, p[u] % q[j], q[j]);
                pinv[j] = h_invmod(pr, q[j]);
            }
            c->muc_PtoQ_pinv[i] = scale_modup_targets(c->h_blob, c->muc_PtoQ[i], pinv.data(), q);
        }
        // genmodDownConstants: [j][i] = MForm((p_0..p_j)^-1 mod q_i)
        c->mdc_PtoQ.assign((size_t)np * nq, 0);
        for (int i = 0; i < nq; i++) {
            u64 acc = 1;
            for (int j = 0; j < np; j++) {
                acc = h_mulmod(acc, p[j] % q[i], q[i]);
                c->mdc_PtoQ[(size_t)j * nq + i] = h_mform(h_invmod(acc, q[i]), q[i]);
            }
        }
        c->mdc_QtoP.assign((size_t)nq * np, 0);
        for (int i = 0; i < np; i++) {
            u64 acc = 1;
            for (int j = 0; j < nq; j++) {
                acc = h_mulmod(acc, q[j] % p[i], p[i]);
                c->mdc_QtoP[(size_t)j * np + i] = h_mform(h_invmod(acc, p[i]), p[i]);
            }
        }
        // Decomposer, ring/basis_extension.go:333-373
        c->muc_dec.clear();
        for (int lvlP = 0; lvlP < np - 1; lvlP++) {
            const int nbPi = lvlP + 2;
            const int ndig = (nq + nbPi - 1) / nbPi;
            std::vector<std::vector<ModUpSet>> per_digit(ndig);
            std::vector<u64> T(c->Q);
            T.insert(T.end(), p, p + nbPi);
            for (int i = 0; i < ndig; i++) {
                int x = nbPi;
                if (i == ndig - 1 && nq % nbPi != 0) x = nq % nbPi;
                for (int j = 0; j < x - 1; j++)
                    per_digit[i].push_back(gen_modup(c->h_blob, q + (size_t)i * nbPi, j + 2, T.data(), (int)T.size()));
            }
            c->muc_dec.push_back(std::move(per_digit));
        }
    }

    if (device < 0) return 0;  // host-only context (tables only)
    // upload
    LGPU_CUDA_OK(cudaSetDevice(device));
    const size_t half = (size_t)(c->nthroot >> 1);
    LGPU_CUDA_OK(cudaMalloc(&c->d_roots, 2 * (size_t)nl * half * sizeof(u64)));
    LGPU_CUDA_OK(cudaMalloc(&c->d_tw, 4 * (size_t)nl * half * sizeof(u64)));
    LGPU_CUDA_OK(cudaMalloc(&c->d_ftw, 2 * (size_t)nl * half * sizeof(double)));
    c->h_limbs.resize(nl);
    for (int i = 0; i < nl; i++) {
        if (upload_limb_tables(c, i)) return -1;
    }
    LGPU_CUDA_OK(cudaMalloc(&c->d_limbs, nl * sizeof(LimbConst)));
    LGPU_CUDA_OK(cudaMemcpy(c->d_limbs, c->h_limbs.data(), nl * sizeof(LimbConst), cudaMemcpyHostToDevice));
    if (!c->h_blob.empty()) {
        LGPU_CUDA_OK(cudaMalloc(&c->d_blob, c->h_blob.size() * sizeof(u64)));
        LGPU_CUDA_OK(cudaMemcpy(c->d_blob, c->h_blob.data(), c->h_blob.size() * sizeof(u64), cudaMemcpyHostToDevice));
    }
    LGPU_CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    {
        // scratch comes from the stream-ordered allocator: keep freed blocks cached in the pool instead of returning
        // them to the driver at every synchronisation (default release threshold is 0)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    return 0;
}

void destroy_context(Ctx* c) {
    if (!c || c->device < 0) return;
    cudaSetDevice(c->device);
    if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
    for (auto& kv : c->auto_index) cudaFree(kv.second);
    for (int i = 0; i < Ctx::HostPipe::kStreams; i++) {
        if (c->host_pipe.st[i]) { cudaStreamSynchronize(c->host_pipe.st[i]); cudaStreamDestroy(c->host_pipe.st[i]); }
        for (int k = 0; k < 3; k++) cudaFree(c->host_pipe.buf[i][k]);
    }
    cudaFree(c->d_scratch);
    cudaFree(c->d_blob);
    cudaFree(c->d_limbs);
    cudaFree(c->d_roots);
    cudaFree(c->d_tw);
    cudaFree(c->d_ftw);
}

}  // namespace lgpu
