// composite.h -- prototypes of composite.cu (multi-kernel operations of the hot path).
#pragma once
#include "engine.h"

namespace lgpu {

struct GadgetCt {          // device-side view of a rlwe.GadgetCiphertext (mirror of lgpu_gadget_ct)
    const u64* data;       // [digit][pw2][2][nQk + nPk][N], NTT + Montgomery (core/rlwe/gadgetciphertext.go:19-45)
    int levelQ, levelP;    // of the key
    int pw2;               // BaseTwoDecomposition
    int ndigits, npw2max;
    const int* pw2_sizes;  // host, per digit (nullptr => all 1)
    const u64* at(int d, int j, int comp, size_t N) const {
        const size_t rows = (size_t)(levelQ + 1) + (size_t)(levelP + 1);
        return data + ((((size_t)d * npw2max + j) * 2 + comp) * rows) * N;
    }
};
struct AccSpans {  // the four accumulator polynomials of a ctQP: [comp].Q (levelQ+1 rows) and [comp].P (levelP+1 rows)
    Span q[2];
    Span p[2];
};

struct Scratch {
    u64* p = nullptr;
    cudaStream_t st = nullptr;
    int alloc(size_t words, cudaStream_t s) {
        st = s;
        LGPU_CUDA_OK(cudaMallocAsync((void**)&p, words * sizeof(u64), s));
        return 0;
    }
    ~Scratch() { if (p) cudaFreeAsync(p, st); }
};

inline RowMap rows_range(int limb0, int drow0, int count) {
    RowMap rm;
    rm.nrows = count;
    for (int i = 0; i < count; i++) { rm.limb[i] = (unsigned char)(limb0 + i); rm.drow[i] = (unsigned char)(drow0 + i); }
    return rm;
}
// QP-stacked buffer: data rows [0, nq) are Q limbs 0.., rows [nq, nq+np) are P limbs 0..
inline RowMap rows_qp(const Ctx* c, int nq, int np) {
    RowMap rm;
    rm.nrows = nq + np;
    for (int i = 0; i < nq; i++) { rm.limb[i] = (unsigned char)i; rm.drow[i] = (unsigned char)i; }
    for (int j = 0; j < np; j++) { rm.limb[nq + j] = (unsigned char)(c->nQ + j); rm.drow[nq + j] = (unsigned char)(nq + j); }
    return rm;
}

int base_rns_decomposition_vector_size(int levelQ, int levelP);
int moddown_qp_to_q(const Ctx* c, int levelQ, int levelP, CSpan p1Q, CSpan p1P, Span p2Q, int batch, cudaStream_t st);
int moddown_qp_to_q_ntt(const Ctx* c, int levelQ, int levelP, CSpan p1Q, CSpan p1P, Span p2Q, int batch, cudaStream_t st);
int moddown_qp_to_p(const Ctx* c, int levelQ, int levelP, CSpan p1Q, CSpan p1P, Span p2P, int batch, cudaStream_t st);
int div_by_last_modulus_ntt(const Ctx* c, int ring, int level, bool round, CSpan p0, Span p1, int batch, cudaStream_t st);
int div_by_last_modulus(const Ctx* c, int ring, int level, bool round, CSpan p0, Span p1, int batch, cudaStream_t st);
int div_by_last_modulus_many(const Ctx* c, int ring, int level, bool round, bool ntt, int nb, CSpan p0, Span p1, int batch, cudaStream_t st);
int automorphism_ntt_index(const Ctx* c, u64 galEl, u64* d_index, cudaStream_t st);
int automorphism_ntt_with_index(const Ctx* c, int rows, CSpan in, const u64* d_index, Span out, bool accumulate, int batch, cudaStream_t st);
int automorphism_coeff(const Ctx* c, const RowMap& rm, CSpan in, u64 gen, Span out, int batch, cudaStream_t st);
int decompose_single_ntt(const Ctx* c, int levelQ, int levelP, int nbPi, int digit, CSpan c2NTT, CSpan c2Inv, Span c2Q, Span c2P,
                         bool copy_digit_rows, int batch, cudaStream_t st);
int decompose_ntt(const Ctx* c, int levelQ, int levelP, int nbPi, CSpan c2, bool c2IsNTT, u64* decomp, int batch, cudaStream_t st);
int gadget_product_lazy(const Ctx* c, int levelQ, CSpan cx, const GadgetCt& evk, const AccSpans& acc, int batch, cudaStream_t st);
int evaluator_moddown_ntt(const Ctx* c, int levelQ, int levelP, const AccSpans& acc, Span ct0, Span ct1, int batch, cudaStream_t st);
int gadget_product(const Ctx* c, int levelQ, CSpan cx, const GadgetCt& evk, Span ct0, Span ct1, int batch, cudaStream_t st);
int rgsw_external_product(const Ctx* c, const GadgetCt& rg0, const GadgetCt& rg1, CSpan ct0, CSpan ct1, Span out0, Span out1, int batch, cudaStream_t st);
// decomp_levelQ: level the DecomposeNTT buffer was laid out for (>= levelQ; -1 = levelQ) -- lintrans uses one decomposition for matrices of lower levels
int gadget_product_hoisted_lazy(const Ctx* c, int levelQ, const u64* decomp, const GadgetCt& evk, const AccSpans& acc, int batch, cudaStream_t st,
                                int decomp_levelQ = -1);
int gadget_product_hoisted(const Ctx* c, int levelQ, const u64* decomp, const GadgetCt& evk, Span ct0, Span ct1, int batch, cudaStream_t st);
int evaluator_automorphism(const Ctx* c, int level, CSpan in0, CSpan in1, u64 galEl, const GadgetCt& gk, Span out0, Span out1,
                           const u64* decomp_hoisted, int batch, cudaStream_t st);
int evaluator_relinearize(const Ctx* c, int level, CSpan c0, CSpan c1, CSpan c2, const GadgetCt& rlk, Span out0, Span out1, int batch, cudaStream_t st);
// keyswitch_fused.cu
bool ks_fused_applicable(const Ctx* c, int levelQ, const GadgetCt& evk);
int gadget_product_multiple_p_fused(const Ctx* c, int levelQ, CSpan cx, CSpan cxInv, const GadgetCt& evk, u64* acc, size_t acc_cs, size_t acc_bs,
                                    int batch, cudaStream_t st);

bool fz_applicable(const Ctx* c, int levelQ, int levelP);
int moddown_ntt_fused(const Ctx* c, int levelQ, int levelP, const u64* acc, size_t acc_cs, size_t acc_bs, const u64* D, size_t d_cs, size_t d_bs,
                      u64* out, size_t o_cs, size_t o_bs, int ncomp, int batch, cudaStream_t st, int rescale = 0);
int div_round_last_ntt_fused(const Ctx* c, int level, const u64* X, size_t x_cs, size_t x_bs, u64* out, size_t o_cs, size_t o_bs,
                             int ncomp, int batch, cudaStream_t st);

int ckks_mulrelin_rescale(const Ctx* c, int level, const u64* ctA, const u64* ctB, const GadgetCt& rlk, int nb_rescales, u64* out, int batch,
                          cudaStream_t st);

}  // namespace lgpu
