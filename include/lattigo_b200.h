/*
 * lattigo_b200.h -- C ABI of the B200-native RNS polynomial-ring engine.
 *
 * Drop-in boundary for ONE hot path of tuneinsight/lattigo v6.2.0: the `ring` package's NTT /
 * coefficient-wise / basis-extension / rescale / automorphism loops and core/rlwe.Evaluator's
 * GadgetProduct key-switch family. The reference has no FFI of its own (pure Go); each entry point
 * below names the Go method it replaces (file:line relative to the upstream tree) and is what a thin
 * cgo shim in forked `ring`, `ring/ringqp` and `core/rlwe` packages binds (see INTEGRATION.md).
 *
 * Conventions
 *   - Polynomials are `uint64_t*` DEVICE-ACCESSIBLE pointers (cudaMalloc / managed / lgpu_malloc) to a
 *     contiguous (limb, coeff) row-major block: row i = residues mod the i-th modulus, N words per row.
 *     ring.Poly{Coeffs [][]uint64} (ring/poly.go:13-15) maps onto it with Coeffs[i] = row i.
 *   - Alignment: lgpu_malloc / cudaMalloc blocks are always fine. The ring-level entry points accept any
 *     8-byte aligned pointer (odd word offsets take 64-bit kernels); the rlwe-level ones (gadget products,
 *     evaluator_*, ckks_*) and evaluation keys require 16-byte aligned blocks and even strides, and return
 *     an error otherwise (their kernels move 128 bits per access). Keys and ciphertexts that are 32-byte aligned
 *     (every cudaMalloc / lgpu_malloc block whose rows are a multiple of 4 words apart) additionally take the 256-bit
 *     accesses of the fused key-switch kernels; results are identical either way.
 *   - `ring` selects the moduli chain: LGPU_RING_Q or LGPU_RING_P (ringqp.Ring{RingQ,RingP},
 *     ring/ringqp/ring.go:15-17). `level` is the reference's level (number of limbs - 1).
 *   - All calls are asynchronous on `stream` (a cudaStream_t cast to void*; NULL = the CUDA default
 *     stream); lgpu_sync() before host access. Entry points ending in _host take HOST pointers and
 *     include the copies.
 *   - Return 0 on success, non-zero on error with lgpu_last_error() (thread-local) describing it.
 *     The shim maps ring-level errors to panic and evaluator-level errors to `error` like the
 *     reference (ring/ntt.go:212, core/rlwe/evaluator_gadget_product.go:110-112).
 *   - Outputs are bit-identical to the reference on identical inputs: canonical residues for the
 *     non-Lazy methods, the reference's exact representative for the *Lazy ones.
 */
#ifndef LATTIGO_B200_H
#define LATTIGO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lgpu_ctx lgpu_ctx;

#define LGPU_RING_Q 0
#define LGPU_RING_P 1

#define LGPU_RING_STANDARD 0           /* ring.Standard            (ring/ring.go:27-31) */
#define LGPU_RING_CONJUGATE_INVARIANT 1 /* ring.ConjugateInvariant  */

/* Opcodes of lgpu_vecop / lgpu_subring_vecop: one per kernel of ring/vec_ops.go, named after the
 * SubRing method that wraps it (ring/subring_ops.go:6-273). */
enum lgpu_vecop_code {
    LGPU_OP_ADD = 0,                             /* SubRing.Add                              vec_ops.go:7   */
    LGPU_OP_ADDLAZY,                             /* AddLazy                                  :31  */
    LGPU_OP_SUB,                                 /* Sub                                      :55  */
    LGPU_OP_SUBLAZY,                             /* SubLazy                                  :79  */
    LGPU_OP_NEG,                                 /* Neg                                      :103 */
    LGPU_OP_REDUCE,                              /* Reduce                                   :125 */
    LGPU_OP_REDUCELAZY,                          /* ReduceLazy                               :147 */
    LGPU_OP_MULCOEFFSLAZY,                       /* MulCoeffsLazy                            :169 */
    LGPU_OP_MULCOEFFSLAZYTHENADDLAZY,            /* MulCoeffsLazyThenAddLazy                 :193 */
    LGPU_OP_MULCOEFFSBARRETT,                    /* MulCoeffsBarrett                         :217 */
    LGPU_OP_MULCOEFFSBARRETTLAZY,                /* MulCoeffsBarrettLazy                     :241 */
    LGPU_OP_MULCOEFFSBARRETTTHENADD,             /* MulCoeffsBarrettThenAdd                  :265 */
    LGPU_OP_MULCOEFFSBARRETTTHENADDLAZY,         /* MulCoeffsBarrettThenAddLazy              :289 */
    LGPU_OP_MULCOEFFSMONTGOMERY,                 /* MulCoeffsMontgomery                      :313 */
    LGPU_OP_MULCOEFFSMONTGOMERYLAZY,             /* MulCoeffsMontgomeryLazy                  :336 */
    LGPU_OP_MULCOEFFSMONTGOMERYTHENADD,          /* MulCoeffsMontgomeryThenAdd               :360 */
    LGPU_OP_MULCOEFFSMONTGOMERYTHENADDLAZY,      /* MulCoeffsMontgomeryThenAddLazy           :383 */
    LGPU_OP_MULCOEFFSMONTGOMERYLAZYTHENADDLAZY,  /* MulCoeffsMontgomeryLazyThenAddLazy       :407 */
    LGPU_OP_MULCOEFFSMONTGOMERYTHENSUB,          /* MulCoeffsMontgomeryThenSub               :431 */
    LGPU_OP_MULCOEFFSMONTGOMERYTHENSUBLAZY,      /* MulCoeffsMontgomeryThenSubLazy           :455 */
    LGPU_OP_MULCOEFFSMONTGOMERYLAZYTHENSUBLAZY,  /* MulCoeffsMontgomeryLazyThenSubLazy       :479 */
    LGPU_OP_MULCOEFFSMONTGOMERYLAZYTHENNEG,      /* MulCoeffsMontgomeryLazyThenNeg           :504 */
    LGPU_OP_ADDLAZYTHENMULSCALARMONTGOMERY,      /* AddLazyThenMulScalarMontgomery (s0)      :529 */
    LGPU_OP_ADDSCALARLAZYTHENMULSCALARMONTGOMERY,/* AddScalarLazyThenMulScalarMontgomery(s0,s1) :553 */
    LGPU_OP_ADDSCALAR,                           /* AddScalar (s0)                           :575 */
    LGPU_OP_ADDSCALARLAZY,                       /* AddScalarLazy (s0)                       :597 */
    LGPU_OP_ADDSCALARLAZYTHENNEGTWOMODULUSLAZY,  /* AddScalarLazyThenNegTwoModulusLazy (s0)  :619 */
    LGPU_OP_SUBSCALAR,                           /* SubScalar (s0)                           :642 */
    LGPU_OP_MULSCALARMONTGOMERY,                 /* MulScalarMontgomery (s0)                 :664 */
    LGPU_OP_MULSCALARMONTGOMERYLAZY,             /* MulScalarMontgomeryLazy (s0)             :686 */
    LGPU_OP_MULSCALARMONTGOMERYTHENADD,          /* MulScalarMontgomeryThenAdd (s0)          :708 */
    LGPU_OP_MULSCALARMONTGOMERYTHENADDSCALAR,    /* MulScalarMontgomeryThenAddScalar (s0,s1=scalarMont) :730 */
    LGPU_OP_SUBTHENMULSCALARMONTGOMERYTWOMODULUS,/* SubThenMulScalarMontgomeryTwoModulus (s0): (p1 - p2 + 2q) * s0  :752 */
    LGPU_OP_MFORM,                               /* MForm                                    :778 */
    LGPU_OP_MFORMLAZY,                           /* MFormLazy                                :800 */
    LGPU_OP_IMFORM,                              /* IMForm                                   :822 */
    LGPU_OP_ZERO,                                /* ZeroVec                                  :847 */
    LGPU_OP_MASK,                                /* MaskVec (w = s0, mask = s1)              :870 */
    LGPU_OP_COUNT
};

/* ---- context ------------------------------------------------------------------------------------ */
/* ring.NewRing x2 + ring.NewBasisExtender + ring.NewDecomposer (ring/ring.go:258-322,
 * ring/basis_extension.go:52-87,318-377): builds every per-prime constant (BRed/MRed constants, NInv,
 * RootsForward/RootsBackward with the reference's primitive-root choice ring/subring.go:161-194,
 * RescaleConstants ring/ring.go:329-346, ModUp/ModDown/Decomposer constants) and uploads them.
 * `p` may be NULL / np = 0 (ring-only use). N = 2^logN, 16 <= N <= 2^17. */
int lgpu_create(lgpu_ctx** out, int device, int logN, int ring_type,
                const uint64_t* q, int nq, const uint64_t* p, int np);
void lgpu_destroy(lgpu_ctx* ctx);
const char* lgpu_last_error(void);
const char* lgpu_version(void);
int lgpu_sync(lgpu_ctx* ctx, void* stream);

/* Table read-back (host buffers) so the Go shim / tests can check the constants against the
 * reference's exported fields (SubRing.Modulus/MRedConstant/BRedConstant/NInv/RootsForward/
 * RootsBackward, ring/subring.go:15-35, ring/ntt.go:38-44). kind: 0 = {q, qinv, bred_hi, bred_lo, ninv,
 * primitive_root} (6 words), 1 = RootsForward (NthRoot/2 words), 2 = RootsBackward,
 * 3 = RescaleConstants row `limb-1` (limb words; Q or P ring). */
int lgpu_ring_get_table(lgpu_ctx* ctx, int ring, int limb, int kind, uint64_t* host_out, size_t nwords);
/* Replaces the generated root tables of one limb by caller-supplied ones (the Go structs' own tables),
 * so constants are identical by construction. */
int lgpu_ring_set_roots(lgpu_ctx* ctx, int ring, int limb, const uint64_t* roots_fwd, const uint64_t* roots_bwd,
                        uint64_t ninv);

/* ---- device memory (mirrors BufferPool.Get / Recycle, ring/pool.go:40-61) ---------------------------- */
int lgpu_malloc(lgpu_ctx* ctx, void** dptr, size_t bytes);
int lgpu_free(lgpu_ctx* ctx, void* dptr);
int lgpu_memcpy_h2d(lgpu_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);
int lgpu_memcpy_d2h(lgpu_ctx* ctx, void* dst, const void* src, size_t bytes, void* stream);

/* ---- NTT ----------------------------------------------------------------------------------------------
 * Ring.NTT / NTTLazy / INTT / INTTLazy (ring/ntt.go:127-152). In-place (in == out) allowed.
 * lazy != 0 returns NTTLazy's representative in [0, 6q) (exact reference schedule); INTTLazy is fully
 * reduced for N >= 16 like the reference (ring/ntt.go:197-206). `batch` polynomials, `batch_stride`
 * words apart (use batch = 1, batch_stride = 0 for a single polynomial). */
int lgpu_ntt(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, uint64_t* out, int lazy,
             int batch, size_t batch_stride, void* stream);
int lgpu_intt(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, uint64_t* out, int lazy,
              int batch, size_t batch_stride, void* stream);
/* Ring.NTT(in, out) followed by Ring.MulCoeffsMontgomery(out, other, out) (ring/ntt.go:127-131 + ring/operations.go:88-92) as
 * one pass over HBM: the product is applied in the transform's last pass (N = 2^13..2^16; two launches otherwise).
 * `other` must not alias `out`; in == out is allowed. */
int lgpu_ntt_then_mul_coeffs_montgomery(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, const uint64_t* other,
                                        uint64_t* out, int batch, size_t batch_stride, void* stream);
/* SubRing.NTT / NTTLazy / INTT / INTTLazy on one row (ring/subring_ops.go:235-253) */
int lgpu_subring_ntt(lgpu_ctx* ctx, int ring, int limb, const uint64_t* in, uint64_t* out, int lazy, void* stream);
int lgpu_subring_intt(lgpu_ctx* ctx, int ring, int limb, const uint64_t* in, uint64_t* out, int lazy, void* stream);

/* ---- coefficient-wise ops -------------------------------------------------------------------------------
 * Ring-level (ring/operations.go:11-392): loops over limbs 0..level. `scalars0/1` are HOST arrays with
 * one value per limb (NULL when the op takes none), e.g. AddScalar passes scalar mod q_i, MulScalar passes
 * MForm(scalar mod q_i). p1/p2 may be NULL for ops that do not read them. */
int lgpu_vecop(lgpu_ctx* ctx, int ring, int level, int opcode, const uint64_t* p1, const uint64_t* p2,
               uint64_t* p3, const uint64_t* scalars0, const uint64_t* scalars1,
               int batch, size_t batch_stride, void* stream);
/* SubRing-level (ring/subring_ops.go:6-273): one row of n words (n <= N) with immediate scalars. */
int lgpu_subring_vecop(lgpu_ctx* ctx, int ring, int limb, int opcode, const uint64_t* p1, const uint64_t* p2,
                       uint64_t* p3, uint64_t s0, uint64_t s1, int n, void* stream);


/* ---- automorphisms (ring/automorphism.go) --------------------------------------------------------------- */
/* AutomorphismNTTIndex (:12-34): writes the N-entry uint64 look-up table to DEVICE memory `index_out`. */
int lgpu_automorphism_ntt_index(lgpu_ctx* ctx, uint64_t gal_el, uint64_t* index_out, void* stream);
/* Ring.AutomorphismNTTWithIndex (:50-77) and ...ThenAddLazy (:82-109, accumulate != 0). Cannot be in-place. */
int lgpu_automorphism_ntt_with_index(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, const uint64_t* index,
                                     uint64_t* out, int accumulate, int batch, size_t batch_stride, void* stream);
/* Ring.AutomorphismNTT (:38-45): index computed on the fly. */
int lgpu_automorphism_ntt(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, uint64_t gal_el, uint64_t* out,
                          int batch, size_t batch_stride, void* stream);
/* Ring.Automorphism (:113-176), coefficient domain, Standard ring. Cannot be in-place. */
int lgpu_automorphism(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, uint64_t gal_el, uint64_t* out,
                      int batch, size_t batch_stride, void* stream);

/* Ring.Shift (ring/operations.go:278-282): out[i] = in[(i + k) mod N] on rows 0..level. In-place allowed. */
int lgpu_shift(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, int k, uint64_t* out,
               int batch, size_t batch_stride, void* stream);
/* Ring.MultByMonomial (ring/operations.go:306-363): out = in * X^k, k > -2N, with the reference's literal
 * `q - x` negation (a wrapped zero coefficient becomes q). In-place allowed. */
int lgpu_mult_by_monomial(lgpu_ctx* ctx, int ring, int level, const uint64_t* in, int k, uint64_t* out,
                          int batch, size_t batch_stride, void* stream);
/* MapSmallDimensionToLargerDimensionNTT (ring/operations.go:380-392): large[r][i*gap + w] = small[r][i],
 * `rows` contiguous rows of n_small resp. n_large words. */
int lgpu_map_small_dimension_to_larger_dimension_ntt(lgpu_ctx* ctx, const uint64_t* pol_small, int n_small,
                                                     uint64_t* pol_large, int n_large, int rows, void* stream);
/* ringqp.Ring.ExtendBasisSmallNormAndCenter (ring/ringqp/operations.go:325-351): reads row 0 of poly_in_q,
 * writes level_p+1 rows of poly_out_p (the copy polyOutQ = polyInQ is the caller's). */
int lgpu_extend_basis_small_norm_and_center(lgpu_ctx* ctx, const uint64_t* poly_in_q, int level_p, uint64_t* poly_out_p,
                                            int batch, size_t stride_q, size_t stride_p, void* stream);

/* bootstrapping.Evaluator.ModUp's coefficient loops (circuits/ckks/bootstrapping/evaluator.go:652-699, :729-741): the value of row 0 (mod q_0,
 * coefficient domain) centred around q_0 and written modulo q_i on rows first_q..level_q of out_q and modulo p_j on rows 0..level_p of out_p
 * (level_p = -1: none). strict = 0 uses the reference's `coeff >= q/2` test (ctIn.Value[0], and Value[1] without ephemeral key), strict = 1
 * its `coeff > q/2` (Value[1] on the sparse-key path). Literal: a negative multiple of a modulus is written as that modulus. */
int lgpu_modup_centered(lgpu_ctx* ctx, const uint64_t* row0, int first_q, int level_q, int level_p, int strict, uint64_t* out_q,
                        uint64_t* out_p, int batch, size_t stride_in, size_t stride_q, size_t stride_p, void* stream);

/* ---- RNS basis extension (ring/basis_extension.go) -------------------------------------------------------
 * polQ has levelQ+1 rows, polP has levelP+1 rows; `batch` polynomials with the given strides (words). */
/* BasisExtender.ModUpQtoP (:177-190) / ModUpPtoQ (:195-209): outputs are the reference's exact (non-canonical,
 * < 2p) representatives. */
int lgpu_modup_qtop(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* pol_q, uint64_t* pol_p,
                    int batch, size_t stride_q, size_t stride_p, void* stream);
int lgpu_modup_ptoq(lgpu_ctx* ctx, int level_p, int level_q, const uint64_t* pol_p, uint64_t* pol_q,
                    int batch, size_t stride_p, size_t stride_q, void* stream);
/* BasisExtender.ModDownQPtoQ (:215-228), ModDownQPtoQNTT (:235-256), ModDownQPtoP (:262-278) */
int lgpu_moddown_qp_to_q(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* p1q, const uint64_t* p1p, uint64_t* p2q,
                         int batch, size_t stride_q, size_t stride_p, void* stream);
int lgpu_moddown_qp_to_q_ntt(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* p1q, const uint64_t* p1p, uint64_t* p2q,
                             int batch, size_t stride_q, size_t stride_p, void* stream);
int lgpu_moddown_qp_to_p(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* p1q, const uint64_t* p1p, uint64_t* p2p,
                         int batch, size_t stride_q, size_t stride_p, void* stream);
/* Decomposer.DecomposeAndSplit (:381-502). p0q: coefficient domain. In the reconstruction branch the rows of
 * p1q that belong to the digit itself are left untouched (the reference leaves unspecified values there and its
 * only caller, DecomposeSingleNTT, overwrites them). */
int lgpu_decompose_and_split(lgpu_ctx* ctx, int level_q, int level_p, int nb_pi, int digit, const uint64_t* p0q,
                             uint64_t* p1q, uint64_t* p1p, int batch, size_t stride_q, size_t stride_p, void* stream);

/* ---- rescaling (ring/scaling.go) ---------------------------------------------------------------------------
 * Ring.DivRoundByLastModulus[NTT] (:101-144), DivFloorByLastModulus[NTT] (:6-33) and the *Many forms
 * (:37-97, :148-212). `level` = input level; the output has level - nb_rescales + 1 rows. flags: bit0 = round
 * (else floor), bit1 = NTT domain. In-place allowed. Strides in words. */
#define LGPU_DIV_ROUND 1
#define LGPU_DIV_NTT 2
int lgpu_div_by_last_modulus_many(lgpu_ctx* ctx, int ring, int level, int flags, int nb_rescales, const uint64_t* p0,
                                  uint64_t* p1, int batch, size_t stride_in, size_t stride_out, void* stream);

/* ---- rlwe.Evaluator key-switch family (core/rlwe/evaluator_gadget_product.go) --------------------------------
 * Evaluation keys are uploaded once as a device array in the layout of rlwe.GadgetCiphertext.Value
 * (core/rlwe/gadgetciphertext.go:19-45): data[digit][pw2][component][limb][coeff] with the (level_q+1) Q limbs
 * first, then the (level_p+1) P limbs; always NTT + Montgomery form (core/rlwe/keygenerator.go:309-318). */
typedef struct {
    const uint64_t* data;         /* device pointer */
    int level_q, level_p;         /* levels of the key (level_p = -1: no P) */
    int base_two_decomposition;   /* GadgetCiphertext.BaseTwoDecomposition */
    int n_digits;                 /* len(Value) */
    int n_pw2_max;                /* max_i len(Value[i]) (second array dimension) */
    const int* pw2_sizes;         /* HOST array, len(Value[i]) per digit; NULL = all 1 */
} lgpu_gadget_ct;

/* Evaluator.GadgetProduct (:16-36): ct = ModDown(<decomp(cx), evk>), cx and ct in the NTT domain.
 * cx: level_q+1 rows; ct0/ct1: level_q+1 rows each. batch with strides in words. */
int lgpu_gadget_product(lgpu_ctx* ctx, int level_q, const uint64_t* cx, const lgpu_gadget_ct* evk,
                        uint64_t* ct0, uint64_t* ct1, int batch, size_t stride_cx, size_t stride_ct, void* stream);
/* Evaluator.GadgetProductLazy (:108-127): result mod QP, not divided by P. acc{0,1}q: level_q+1 rows,
 * acc{0,1}p: level_p+1 rows (canonical residues, as the reference's trailing Reduce leaves them). */
int lgpu_gadget_product_lazy(lgpu_ctx* ctx, int level_q, const uint64_t* cx, const lgpu_gadget_ct* evk,
                             uint64_t* acc0q, uint64_t* acc0p, uint64_t* acc1q, uint64_t* acc1p,
                             int batch, size_t stride_cx, size_t stride_q, size_t stride_p, void* stream);
/* Evaluator.ModDown (:39-97), NTT -> NTT case: ct[k] = ModDownQPtoQNTT(acc[k]). */
int lgpu_evaluator_moddown(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* acc0q, const uint64_t* acc0p,
                           const uint64_t* acc1q, const uint64_t* acc1p, uint64_t* ct0, uint64_t* ct1,
                           int batch, size_t stride_q, size_t stride_p, size_t stride_ct, void* stream);
/* Evaluator.DecomposeSingleNTT (:487-510). c2ntt / c2inv: the input in and out of the NTT domain. */
int lgpu_decompose_single_ntt(lgpu_ctx* ctx, int level_q, int level_p, int nb_pi, int digit, const uint64_t* c2ntt,
                              const uint64_t* c2inv, uint64_t* c2q, uint64_t* c2p, int batch, size_t stride_in,
                              size_t stride_q, size_t stride_p, void* stream);
/* Evaluator.DecomposeNTT (:459-483). decomp: device array [digit][batch][level_q+1 + level_p+1][N]
 * (BuffDecompQP[digit].Q rows then .P rows). */
int lgpu_decompose_ntt(lgpu_ctx* ctx, int level_q, int level_p, int nb_pi, const uint64_t* c2, int c2_is_ntt,
                       uint64_t* decomp, int batch, size_t stride_in, void* stream);
/* Evaluator.GadgetProductHoisted (:348-368) / GadgetProductHoistedLazy (:381-399) on a DecomposeNTT result. */
int lgpu_gadget_product_hoisted(lgpu_ctx* ctx, int level_q, const uint64_t* decomp, const lgpu_gadget_ct* evk,
                                uint64_t* ct0, uint64_t* ct1, int batch, size_t stride_ct, void* stream);
int lgpu_gadget_product_hoisted_lazy(lgpu_ctx* ctx, int level_q, const uint64_t* decomp, const lgpu_gadget_ct* evk,
                                     uint64_t* acc0q, uint64_t* acc0p, uint64_t* acc1q, uint64_t* acc1p,
                                     int batch, size_t stride_q, size_t stride_p, void* stream);
/* Evaluator.Automorphism (core/rlwe/evaluator_automorphism.go:13-57) and AutomorphismHoisted (:63-102,
 * decomp != NULL), degree-1 NTT-domain ciphertexts stored as [batch][2][level+1][N]. */
int lgpu_evaluator_automorphism(lgpu_ctx* ctx, int level, const uint64_t* ct_in, uint64_t gal_el,
                                const lgpu_gadget_ct* gk, const uint64_t* decomp, uint64_t* ct_out, int batch, void* stream);
/* Evaluator.Relinearize (core/rlwe/evaluator_evaluationkey.go:121-148): ct_in [batch][3][level+1][N] ->
 * ct_out [batch][2][level+1][N]. */
int lgpu_evaluator_relinearize(lgpu_ctx* ctx, int level, const uint64_t* ct_in, const lgpu_gadget_ct* rlk,
                               uint64_t* ct_out, int batch, void* stream);

/* ---- hoisted linear transformations (circuits/common/lintrans/lintrans_evaluator.go) -------------------------------
 * lintrans.LinearTransformation (lintrans.go:150-160) with its diagonals resident on the device. */
typedef struct {
    int level_q, level_p;          /* LinearTransformation.LevelQ / LevelP */
    int log_slots;                 /* LogDimensions.Cols: rotations are taken modulo 2^log_slots */
    int n1;                        /* N1: 0 = naive evaluator (one key per diagonal), else the BSGS baby-step count (power of two) */
    int n_diags;                   /* len(Vec) */
    const int* diag_index;         /* HOST: the keys of Vec */
    const uint64_t* const* diag;   /* HOST array of DEVICE pointers; diag[i] = Vec[diag_index[i]] as a ringqp.Poly block:
                                      (level_q+1) Q rows then (level_p+1) P rows, NTT + Montgomery form */
} lgpu_lintrans;
/* The GaloisKeys of an rlwe.EvaluationKeySet (core/rlwe/evaluationkeyset.go): gal_els[i] -> keys[i]. HOST arrays. */
typedef struct {
    int n_keys;
    const uint64_t* gal_els;
    const lgpu_gadget_ct* keys;
} lgpu_galois_keys;
/* rlwe.Parameters.GaloisElement (core/rlwe/params.go:580-583): GaloisGen^k mod NthRoot, k may be negative. */
uint64_t lgpu_galois_element(lgpu_ctx* ctx, long long k);
/* lintrans.Evaluator.EvaluateMany (:28-79; Evaluate / EvaluateNew are the one-matrix calls): decomposes ct_in[1] once,
 * pre-rotates the baby steps once for all BSGS matrices (AutomorphismHoistedLazy, :82-114), then MultiplyByDiagMatrix
 * (:141-274) or MultiplyByDiagMatrixBSGS (:280-470) per matrix. ct_in: [batch][2][level_in+1][N], NTT domain.
 * ct_outs: HOST array of n_mats device pointers, ct_outs[i]: [batch][2][out_levels[i]+1][N]; on return out_levels[i] is the
 * level of the result = min(out_levels[i], level_in, mats[i].level_q) (the reference Resizes opOut): rows 0..that level of
 * each component are written, the block keeps its layout. ct_outs[i] == ct_in is allowed (EvaluateSequential, :117-139).
 * A missing Galois key is an error ("GaloisKey[g] is missing"), like CheckAndGetGaloisKey. */
int lgpu_lintrans_evaluate_many(lgpu_ctx* ctx, int level_in, const uint64_t* ct_in, const lgpu_lintrans* mats, int n_mats,
                                const lgpu_galois_keys* gks, uint64_t* const* ct_outs, int* out_levels, int batch, void* stream);
/* Evaluator.AutomorphismHoistedLazy (core/rlwe/evaluator_automorphism.go:107-165), NTT-domain ciphertexts: the result stays
 * modulo QP, scaled by P. ct0: ctIn.Value[0] (level_q+1 rows used); decomp: lgpu_decompose_ntt output laid out for
 * decomp_level_q >= level_q. Outputs as in lgpu_gadget_product_lazy. */
int lgpu_evaluator_automorphism_hoisted_lazy(lgpu_ctx* ctx, int level_q, const uint64_t* ct0, const uint64_t* decomp, int decomp_level_q,
                                             uint64_t gal_el, const lgpu_gadget_ct* gk, uint64_t* out0q, uint64_t* out0p, uint64_t* out1q,
                                             uint64_t* out1p, int batch, size_t stride_ct, size_t stride_q, size_t stride_p, void* stream);

/* ---- RGSW (core/rgsw) --------------------------------------------------------------------------------------------------
 * rgsw.Evaluator.ExternalProduct (core/rgsw/evaluator.go:39-88): RLWE x RGSW -> RLWE at the RGSW ciphertext's levels.
 * rgsw0 / rgsw1 = rgsw.Ciphertext.Value[0] / Value[1] (core/rgsw/elements.go:11-13). ct_in: [batch][2][level_in+1][N], NTT domain;
 * ct_out: [batch][2][level_out+1][N], rows 0..rgsw level written; ct_out == ct_in allowed (how the reference's callers use it).
 * All three reference paths (multiple P :210-283, single P / bit decomposition :130-208, 32-bit :90-128) are covered. */
int lgpu_rgsw_external_product(lgpu_ctx* ctx, const uint64_t* ct_in, int level_in, const lgpu_gadget_ct* rgsw0,
                               const lgpu_gadget_ct* rgsw1, uint64_t* ct_out, int level_out, int batch, void* stream);

/* ---- encryptor / key-generator inner loops and device samplers (core/rlwe/encryptor.go, keygenerator.go, ring/sampler_*.go) ----
 * Samplers: the reference's distributions on Philox4x32-10 counter streams keyed by (seed, stream_id) -- NOT the reference's
 * blake2b-XOF byte stream (sampling/prng.go), which is inherently sequential. Small polynomials are int64 vectors [batch][N].
 * Each (seed, stream_id, sampler kind, limb) has its own counter space: two samplers, or the Q and P rows of a uniform draw,
 * never read the same random block, and a uniform row does not depend on the level it is drawn at.
 * Philox with a 64-bit seed is a statistical generator, not a cryptographic one: it suits tests and benchmarks. Production
 * key material should come from the caller (a host CSPRNG) through the int64 / residue arguments of the functions below. */
/* ringqp.UniformSampler.Read (ring/sampler_uniform.go:48-100): rows 0..level uniform in [0, q_i). */
int lgpu_sample_uniform(lgpu_ctx* ctx, int ring, int level, uint64_t seed, uint64_t stream_id, uint64_t* out, int batch,
                        size_t batch_stride, void* stream);
/* ring.TernarySampler (ring/sampler_ternary.go): hamming_weight > 0 selects ring.Ternary{H} (exactly H non-zero coefficients),
 * otherwise ring.Ternary{P = p} (P(+1) = P(-1) = p / 2). */
int lgpu_sample_ternary(lgpu_ctx* ctx, double p, int hamming_weight, uint64_t seed, uint64_t stream_id, int64_t* out, int batch,
                        void* stream);
/* ring.GaussianSampler (ring/sampler_gaussian.go:160-182): round(|N(0,1)| sigma) with a random sign, |.| <= bound. */
int lgpu_sample_gaussian(lgpu_ctx* ctx, double sigma, double bound, uint64_t seed, uint64_t stream_id, int64_t* out, int batch,
                         void* stream);
/* What Sampler.Read + ringqp.Ring.ExtendBasisSmallNormAndCenter (ring/ringqp/operations.go:325-351) leave in a ringqp.Poly:
 * the signed value modulo every q_i (out_q, level_q+1 rows) and p_j (out_p, level_p+1 rows); either output may be NULL. */
int lgpu_small_poly_to_rns(lgpu_ctx* ctx, int level_q, int level_p, const int64_t* small, uint64_t* out_q, uint64_t* out_p,
                           int batch, size_t stride_q, size_t stride_p, void* stream);
/* Encryptor.encryptZeroPk for a plain rlwe.Ciphertext (core/rlwe/encryptor.go:204-299: one special prime, ModDownQPtoQ) or, when
 * the context has no P, encryptZeroPkNoP (:301-341). pk: rlwe.PublicKey.Value = [2][nQ + nP][N] at the maximum levels (NTT +
 * Montgomery); u (xs sample), e0, e1 (xe samples): [batch][N]; ct_out: [batch][2][level_q+1][N]. */
int lgpu_encrypt_zero_pk(lgpu_ctx* ctx, int level_q, const uint64_t* pk, const int64_t* u, const int64_t* e0, const int64_t* e1,
                         uint64_t* ct_out, int is_ntt, int is_montgomery, int batch, void* stream);
/* Encryptor.encryptZeroSkFromC1QP (:404-430; level_p = -1 for a plain ciphertext): c0 = e - c1 * sk. sk: [nQ + nP][N]; c1, c0:
 * [batch][level_q+1 + level_p+1][N] (Q rows then P rows); c1 is the uniform polynomial in the NTT domain (rewritten by INTT only
 * when !is_ntt, like the reference). */
int lgpu_encrypt_zero_sk(lgpu_ctx* ctx, int level_q, int level_p, const uint64_t* sk, uint64_t* c1, const int64_t* e, uint64_t* c0,
                         int is_ntt, int is_montgomery, int batch, void* stream);
/* KeyGenerator.genEvaluationKey (core/rlwe/keygenerator.go:287-330) + AddPolyTimesGadgetVectorToGadgetCiphertext
 * (core/rlwe/gadgetciphertext.go:171-241) at the maximum levels. On entry component 1 of every evk->data[i][j] holds the uniform
 * polynomial (e.g. from lgpu_sample_uniform; evk->data is written although the struct declares it const); e: [n_digits][n_pw2_max][N]
 * error samples; sk_in: [nQ][N], sk_out: [nQ + nP][N], NTT + Montgomery. */
int lgpu_gen_evaluation_key(lgpu_ctx* ctx, const uint64_t* sk_in, const uint64_t* sk_out, lgpu_gadget_ct* evk, const int64_t* e,
                            void* stream);
/* blindrot.Evaluator.BlindRotateCore (core/rgsw/blindrot/evaluator.go:144-229; Algorithm 3 of eprint 2022/198) on one accumulator, in place.
 * a_host: the LWE mask modulo 2N (HOST, n_lwe odd-or-zero words); acc: [2][level+1][N] NTT-domain RLWE accumulator; brk0[j] / brk1[j]:
 * Value[0] / Value[1] of RGSW(X^{s_j}) (HOST arrays of n_lwe key descriptors); gks: the automorphism keys of the window
 * (GaloisElement(1..window_size) and NthRoot - GaloisGen; a missing one is an error). window_size = 10 in the reference (keys.go:14). */
int lgpu_blind_rotate_core(lgpu_ctx* ctx, const uint64_t* a_host, int n_lwe, uint64_t* acc, int level, const lgpu_gadget_ct* brk0,
                           const lgpu_gadget_ct* brk1, const lgpu_galois_keys* gks, int window_size, void* stream);
/* ckks.SpecialFFTDouble / SpecialIFFTDouble (schemes/ckks/ckks_vector_ops.go:18-77; Encoder.FFT / IFFT, schemes/ckks/encoder.go:764-816), in
 * place on `batch` vectors of n complex128 values (device, interleaved re / im, batch_stride in complex values). rot_group (n int64 values)
 * and roots (m + 1 complex128 values) are the encoder's own tables (encoder.go:83-112), device resident. Same operations in the same order
 * as the Go code and no fused multiply-add: results are bit-identical on identical tables. */
int lgpu_ckks_special_fft(lgpu_ctx* ctx, double* values, int n, int m, const int64_t* rot_group, const double* roots, int inverse,
                          int batch, size_t batch_stride, void* stream);

/* ---- wire format -> device (the reference's WriteTo / ReadFrom byte streams, little-endian uint64 words) ------------------
 * ring.Poly (ring/poly.go:132-179): rows, then per row {len, len words}. */
int lgpu_poly_load(lgpu_ctx* ctx, const void* bytes, size_t nbytes, uint64_t* dst, int rows_cap, int* rows_out, size_t* consumed,
                   void* stream);
/* ring.Poly.WriteTo of `rows` device rows into `bytes` (8 + rows * (8 + 8 N) bytes); synchronises `stream`. */
int lgpu_poly_store(lgpu_ctx* ctx, const uint64_t* src, int rows, void* bytes, size_t cap, size_t* written, void* stream);
#define LGPU_MAX_DIGITS 128
typedef struct {
    int level_q, level_p, base_two_decomposition, n_digits, n_pw2_max;
    int pw2_sizes[LGPU_MAX_DIGITS];   /* len(Value[i]); usable as lgpu_gadget_ct.pw2_sizes */
    size_t device_bytes;              /* size of the device block in the lgpu_gadget_ct layout */
    size_t consumed;                  /* bytes of the stream that belong to this object */
} lgpu_evk_info;
/* rlwe.GadgetCiphertext.ReadFrom / UnmarshalBinary (core/rlwe/gadgetciphertext.go:101-167; also EvaluationKey and
 * RelinearizationKey, which are GadgetCiphertexts): BaseTwoDecomposition, then structs.Matrix[VectorQP]
 * (utils/structs/matrix.go:80-140). With dst == NULL only *info is filled (no device work); with a 16-byte aligned device
 * block of info->device_bytes bytes the rows are copied straight from the byte stream into the lgpu_gadget_ct layout. */
int lgpu_gadget_ct_load(lgpu_ctx* ctx, const void* bytes, size_t nbytes, uint64_t* dst, size_t dst_bytes, lgpu_evk_info* info,
                        void* stream);
/* rlwe.GaloisKey.ReadFrom (core/rlwe/keys.go:628-700): GaloisElement, NthRoot, EvaluationKey. */
int lgpu_galois_key_load(lgpu_ctx* ctx, const void* bytes, size_t nbytes, uint64_t* gal_el, uint64_t* nth_root, uint64_t* dst,
                         size_t dst_bytes, lgpu_evk_info* info, void* stream);

/* ---- fused batch entry points for the measured op sequences ---------------------------------------------------
 * ckks.Evaluator.MulRelinNew(ct_a, ct_b) followed by Rescale (schemes/ckks/evaluator.go:719-872, :477-515;
 * nb_rescales = Parameters.LevelsConsumedPerRescaling(), 0 = no rescale). ct_a, ct_b: [batch][2][level+1][N]
 * (NTT domain); ct_out: [batch][2][level+1-nb_rescales][N]. _host: pinned or pageable HOST buffers, copies
 * included and pipelined in chunks of `chunk` ciphertext pairs (0 = default). */
int lgpu_ckks_mulrelin_rescale_batch(lgpu_ctx* ctx, int level, const uint64_t* ct_a, const uint64_t* ct_b,
                                     const lgpu_gadget_ct* rlk, int nb_rescales, uint64_t* ct_out, int batch, void* stream);
int lgpu_ckks_mulrelin_rescale_batch_host(lgpu_ctx* ctx, int level, const uint64_t* ct_a_host, const uint64_t* ct_b_host,
                                          const lgpu_gadget_ct* rlk, int nb_rescales, uint64_t* ct_out_host, int batch, int chunk);


/* ---- launch accounting / profiling (used by bench.py) ------------------------------------------------------- */
enum lgpu_kclass {
    LGPU_KCLASS_NTT_FWD = 0,   /* one forward transform of rows x batch polynomials (1 or 2 kernels) */
    LGPU_KCLASS_NTT_INV,
    LGPU_KCLASS_VECOP,
    LGPU_KCLASS_MODUP,         /* basis extension / decomposition */
    LGPU_KCLASS_MAC,           /* key-switch multiply-accumulate */
    LGPU_KCLASS_TENSOR,
    LGPU_KCLASS_AUTOMORPHISM,
    LGPU_KCLASS_FUSED,         /* K2: basis extension / rescale prologue folded into the strided transform pass */
    LGPU_KCLASS_EPILOGUE,      /* chunk transform pass with the ModDown / Rescale epilogue */
    LGPU_KCLASS_COUNT
};
/* total number of CUDA kernels this library has launched in the process */
unsigned long long lgpu_launch_count(void);
/* When enabled every launch scope is bracketed by CUDA events on its stream. lgpu_profile_read sums (and clears)
 * per class: elapsed ms, algorithmic bytes (compulsory read + write of the operands), scopes and kernels. */
int lgpu_profile_enable(int on);
int lgpu_profile_read(double* ms, double* alg_bytes, unsigned long long* scopes, unsigned long long* kernels);

#ifdef __cplusplus
}
#endif
#endif /* LATTIGO_B200_H */
