/* oriana_b200.h -- C ABI of the B200-native PCMF CAVI hot path.
 *
 * Drop-in boundary for ONE path of AntoinePassemiers/Oriana: `FactorModel.step()`
 * (oriana/models/base.py:54-56) for the ZIGaP and GaP models (and, behind ORI_F_SPARSE, SparseZIGaP,
 * oriana/models/sparse_zigap.py:100-204, with the deviance metrics of base.py:58-82), i.e. the E-step
 * `update_variational_parameters` (oriana/models/zigap.py:97-141, gap.py:82-115) with its numba kernel
 * `compute_Z_q_expectations` (zigap.py:79-95, gap.py:67-80, sparse_zigap.py:100-116), the node expectations `Gamma.mean/meanlog`
 * (oriana/nodes/probabilistic/gamma.py:37-61), `Bernoulli.mean` (bernoulli.py:41-48), and the M-step
 * `update_prior_hyper_parameters` (zigap.py:143-158, gap.py:117-129) with `inverse_digamma`
 * (oriana/utils.py:39-51).
 *
 * Conventions (SURVEY.md section 8b):
 *   - plain pointers and sizes only; every DEVICE buffer is owned by the caller (PyTorch allocates);
 *     the library never allocates or frees device memory behind the caller's back, except inside the
 *     `*_host` / `*_ctx` operator entry points, which take HOST pointers and keep their staging buffers in a
 *     context (ori_ctx_t) between calls;
 *   - device entry points are stream-ordered on the `stream` argument (a cudaStream_t passed as void*),
 *     never synchronise the device and never touch the host copy of any result;
 *   - return 0 on success, a negative ORI_E* code otherwise; `ori_last_error` gives the message;
 *   - accumulators are zero-filled by the callee, like the reference kernels (zigap.py:81-83).
 * There is NO CPU fallback anywhere in this library.
 */
#ifndef ORIANA_B200_H
#define ORIANA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORI_OK 0
#define ORI_EINVAL (-1)   /* bad argument (shape, alignment, null pointer)   */
#define ORI_ECUDA (-2)    /* a CUDA runtime call or kernel launch failed      */
#define ORI_ENODEV (-3)   /* no sm_100 device                                 */
#define ORI_EUNSUPPORTED (-4)

/* flags of ori_problem_t::flags */
#define ORI_F_DROPOUT 1u      /* ZIGaP (zero-inflation layer D); clear = GaP                              */
#define ORI_F_QUIRK 2u        /* reproduce zigap.py:94: Zj weighted by D_hat[i, k] instead of D_hat[i, j] */
#define ORI_F_ELBO 4u         /* accumulate the ELBO terms inside the row pass                            */
#define ORI_F_NO_TENSOR 8u    /* force the CUDA-core kernels (tests); default picks tcgen05 when it can   */
#define ORI_F_SPARSE 16u      /* SparseZIGaP: spike-and-slab layer S on V (sparse_zigap.py:100-204); needs
                                 ORI_F_DROPOUT, the `sparse` block below, K <= 64 (tensor kernels: K <= 32), no ELBO */
#define ORI_F_DEVICE_ITER 32u /* the iteration count (index into elbo_trace) is read from scal[ORI_SC_ITER] on the
                                 device instead of ori_problem_t::iter, so that one captured CUDA graph of a whole
                                 step can be replayed for every iteration                                   */

#define ORI_F_PRECISE 64u     /* tensor path only (K <= 32): the accumulating contractions R.eV, D.V_hat and their transposes
                                 take R, D_hat and the factor operands split hi/lo (tf32 + one bf16 chain for the cross terms)
                                 like den and U.V^T: every sum fp32-grade (~2^-21) instead of TF32-grade; about half the rate.
                                 K > 32 with this flag runs the CUDA-core kernels                                           */
#define ORI_F_FIXED_CHAIN 128u /* this problem is a row slab of a larger matrix (host-streamed steps): keep the tensor kernels'
                                 accumulation chunks at their nominal length even when the slab is too small to fill the
                                 machine, so that its sums are chained -- and rounded -- like the resident matrix's          */

#define ORI_F_DETERMINISTIC 256u /* every sum that the plain kernels form with floating-point atomics is formed in a fixed order
                                 instead, so two runs of the same problem on the same device agree bit for bit.  Tensor kernels:
                                 the chunk items of a row block / gene block add their partial sums one after the other (a
                                 ticket per block); per-item ELBO terms and per-block factor sums go through scratch arrays
                                 that are summed in index order.  CUDA-core kernels (up to 2^26 matrix entries): one CTA per
                                 row block, per-CTA / per-row-chunk slots summed in index order.  Needs det_ws.             */
#define ORI_F_X_U16 512u      /* X holds the counts as uint16_t (the caller casts the pointer): half the bytes of float32 in HBM.
                                 ldx (elements) must be a multiple of 8, so that a row starts on 16 bytes for TMA.  Every kernel
                                 widens a count to float32 exactly (u < 2^23) as it reads it, so the results are those of the
                                 float32 matrix of the same counts                                                          */

/* modes of ori_mstep */
#define ORI_M_STEP 0          /* regular end of iteration t+1: finalise ELBO(t), pi(t); M-step; next lp   */
#define ORI_M_INIT 1          /* after ori_init_expectations: M-step on the initial expectations          */
#define ORI_M_INIT_KEEP 2     /* same but keep the caller's alpha/beta (state copied from a model)        */
#define ORI_M_FINALIZE 3      /* flush: pi(t) and ELBO(t) of the CURRENT state, nothing else changes      */
#define ORI_M_REFRESH 4       /* after ori_init_expectations on edited (a,b): only the pending ELBO terms  */

/* Layout of the reduction buffers of ori_problem_t (the caller allocates them at these sizes):
 *   red32 = [Zj | b2s | Zl]               float32, blocks of p x KP; the block Zl only with eUl (ORI_F_SPARSE)
 *   red64 = [colsum D_hat (p) | sum_i log U_hat (KP) | sum_i U_hat (KP) | ELBO partials (ORI_R64_NSLOTS)]
 *   gsum  = [sum_j log V_hat (KP) | sum_j V_hat (KP) | gene partials (ORI_GSUM_NSLOTS)]
 *   scal  = ORI_SC_NSLOTS per-model scalars                                                                 */
#define ORI_RED32_FLOATS(p, KP, third) (((third) ? 3 : 2) * (int64_t)(p) * (KP))
#define ORI_RED64_DOUBLES(p, KP) ((int64_t)(p) + 2 * (KP) + ORI_R64_NSLOTS)
#define ORI_GSUM_DOUBLES(KP) (2 * (KP) + ORI_GSUM_NSLOTS)

/* slots of the ELBO partials of red64 (summed over ranks with it) */
#define ORI_R64_XLOGDEN 0     /* sum_{X>0} X log den                                                      */
#define ORI_R64_ENT 1         /* sum_{X==0} entropy of q(D_ij)                                            */
#define ORI_R64_PUV 2         /* sum_ij D_hat_ij (U_hat V_hat^T)_ij                                       */
#define ORI_R64_HROW 3        /* sum_ik entropy of q(U_ik)                                                */
#define ORI_R64_LGAMX 4       /* sum_{X>0} lgamma(X+1)   (ori_count_stats)                                */
#define ORI_R64_NNZ 5         /* number of non-zero entries   (ori_count_stats)                           */
#define ORI_R64_NSLOTS 8

/* slots of the gene partials of gsum */
#define ORI_GSUM_HGENE 0      /* sum_jk entropy of q(V_jk)                                                */
#define ORI_GSUM_NSLOTS 8

/* slots of scal (float64 scalars that persist between calls); slot 3 and slots 7.. are unused */
#define ORI_SC_LGAMX 0        /* sum_{X>0} lgamma(X+1)         (constant, all ranks)                      */
#define ORI_SC_NNZ 1          /* number of non-zero entries    (constant, all ranks)                      */
#define ORI_SC_PENDING 2      /* K-, p- and nK-sized ELBO terms of the current state, entropies included  */
#define ORI_SC_ELBO_LAST 4    /* last finalised ELBO                                                      */
#define ORI_SC_ITER 5         /* completed iterations (read by ORI_F_DEVICE_ITER)                         */
#define ORI_SC_UVSUM 6        /* sum_k (sum_i U_hat_ik)(sum_j V_hat_jk) of the current state (GaP's ELBO)  */
#define ORI_SC_NSLOTS 16

/* One rank's view of the problem.  Factor arrays are row-major with row stride KP (K padded to a
 * multiple of 8, pad columns hold zeros).  "gen" arrays are ping-pong generations of the row factors:
 * the gene pass needs U_hat(t) (to rebuild D_hat(t)) and U_hat(t+1) at the same time (zigap.py:124).   */
typedef struct ori_problem {
    int64_t n_rows;        /* cells owned by this rank                                   */
    int64_t n_total;       /* cells over all ranks (denominator of the M-step means)     */
    int64_t ldx;           /* row stride of X in elements (multiple of 4; of 8 with ORI_F_X_U16) */
    int32_t p;             /* genes                                                      */
    int32_t K;             /* latent dimension                                           */
    int32_t KP;            /* padded latent dimension: 8, 16, 32 or 64, >= K             */
    uint32_t flags;        /* ORI_F_*                                                    */
    int32_t iter;          /* completed iterations (index into elbo_trace)               */
    int32_t trace_cap;     /* capacity of elbo_trace                                     */

    const float* X;        /* [n_rows x ldx] counts as float32 (zigap.py:112), or uint16_t with ORI_F_X_U16 */

    /* row side, [n_rows x KP] float32 */
    float* a1;             /* Gamma shape of q(U)   zigap.py:115                         */
    float* a2;             /* Gamma rate  of q(U)   zigap.py:116                         */
    float* U_hat[2];       /* E[U]      = a1/a2             gamma.py:37-46               */
    float* eU[2];          /* exp(E[log U]) = exp(psi(a1))/a2   gamma.py:48-61           */
    float* eUw;            /* eU * D_hat[:, :K] (quirk operand, zigap.py:94) or NULL     */
    float* Zi;             /* accumulator  sum_j R_ij eV_jk                              */
    float* a2s;            /* accumulator  sum_j D_hat_ij V_hat_jk                       */

    /* gene side, [p x KP] float32 (replicated on every rank) */
    float* b1;             /* zigap.py:123 */
    float* b2;             /* zigap.py:124 */
    float* V_hat;
    float* eV;
    float* red32;          /* [ORI_RED32_FLOATS(p, KP, eUl != NULL)] Zj | b2s (| Zl) -- allreduce(sum) buffer #1 */

    float* lp;             /* [p] logit(pi) generating the CURRENT D_hat; -inf: D_hat=(X>0) (zigap.py:77) */
    float* pfloor;         /* [p] 1e-10 where pi<=0 (zigap.py:133), else 0               */

    /* float64 small state */
    double* hyper;         /* [4 x K] alpha1 | alpha2 | beta1 | beta2                    */
    double* red64;         /* [ORI_RED64_DOUBLES(p, KP)] colsum D_hat | sum_i log U_hat | sum_i U_hat |
                              ORI_R64_* partials -- allreduce(sum) buffer #2              */
    double* gsum;          /* [ORI_GSUM_DOUBLES(KP)] sum_j log V_hat | sum_j V_hat | ORI_GSUM_* partials */
    double* pi_d;          /* [p] Bernoulli prior pi(t)  zigap.py:158                    */
    double* scal;          /* [ORI_SC_NSLOTS] the ORI_SC_* scalars                       */
    double* elbo_trace;    /* [trace_cap]                                                */

    /* tensor path (tcgen05/TMA kernels, csrc/kernels_tc.cu): caller-owned scratch of at least
     * ori_tc_workspace_floats(n_rows, p, KP) floats, 128-byte aligned; NULL selects the CUDA-core kernels.
     * Needs KP == 32 (K <= 32) or KP == 64 (K <= 64), zero padded. */
    float* tc_ws;
    int64_t tc_ws_floats;

    /* SparseZIGaP (ORI_F_SPARSE).  With this flag b1, b2 parametrise V' (sparse_zigap.py:24-28), eV holds
     * exp(E[log V']) without the mask, V_hat holds the EFFECTIVE factor S_hat * V'_hat (:140) and red32
     * has its third block, Zl = sum_i R_ij eU_ik E[log U_ik] (:116).
     * Gene-side arrays are [p x KP] float32. */
    float* p_s;            /* Bernoulli parameter of q(S) = S_hat (float32(p_s), bernoulli.py:45)          */
    float* logV;           /* E[log V'] (read by :116 and :157)                                            */
    float* eVd;            /* eV * (p_s > tau): denominator operand (:103-104, :134)                       */
    float* eVz;            /* eVd * S_hat: operand of the row sums (:114)                                  */
    float* Vh_old;         /* S_hat * V'_hat of the PREVIOUS iteration: generates the current D_hat
                              (:166 multiplies the new U_hat with the V_hat local of :140)                 */
    float* eUl[2];         /* row side, per generation: eU * E[log U] (operand of :116).  Set, it asks the gene
                              pass for the third sum in red32 block 2; only with ORI_F_SPARSE (ori_problem_check) */
    double* pi_s;          /* [p] prior of S, row means of p_s (:196), float64                             */
    double tau;            /* threshold of S_tilde (:134)                                                  */

    /* eU / eV hold exp(E[log .]) of each cell / gene rescaled by 2^58 / max_k exp(E[log .]) (the multinomial step only
     * uses ratios, zigap.py:86-92; see csrc/special.cuh).  The ELBO term sum_ij X_ij log den_ij takes the scales back
     * through the row sums of this rank's X and the column sums of the WHOLE X (ori_row_sums_f32,
     * ori_column_sums_f64 + all-reduce, as float32); required with ORI_F_ELBO, NULL otherwise. */
    const float* xrow;     /* [n_rows] */
    const float* xcol;     /* [p]      */

    /* Float32-underflow emulation of the reference's multinomial step (zigap.py:86-90, gap.py:73-76), optional: both
     * NULL = off (exact ratios everywhere).  thr = 2^-17 exp(-max_k E[log .]) per cell / gene, written next to eU / eV by
     * ori_init_expectations, ori_row_update and ori_gene_update; the passes drop every term with
     * eU_ik eV_jk <= thrU_i thrV_j -- the terms whose float32 exp(log_U_hat + log_V_hat) is 0 in the reference -- so an
     * entry whose terms all underflow assigns its count to no component (den = 0 -> 1, :90).  CUDA-core kernels: per
     * term; tcgen05 kernels: per entry (den < thrU_i thrV_j).  The sparse model's terms carry the mask S_tilde
     * (sparse_zigap.py:109): same rule. */
    float* thrU;           /* [2 x n_rows], per generation like eU */
    float* thrV;           /* [p]                                  */

    /* ORI_F_DETERMINISTIC: scratch of ori_det_workspace_doubles(n_rows, p, KP) doubles (NULL otherwise) */
    double* det_ws;
    int64_t det_ws_doubles;
} ori_problem_t;

/* ---- library ---------------------------------------------------------------------------------- */
int ori_version(void);
/* Number of CUDA kernels this library has launched in this process (memsets and copies not counted). */
unsigned long long ori_kernel_launches(void);
/* Copies the last error message of the calling thread into buf; returns its length. */
int ori_last_error(char* buf, size_t len);
/* 0 when device `dev` is an sm_100 part, ORI_ENODEV otherwise. */
int ori_device_check(int dev);

/* ---- special functions on device arrays (oriana/utils.py:9-51; KATs test/test.py:13-32) -------- */
/* op: 0 digamma, 1 trigamma (digamma_prime), 2 inverse_digamma, 3 sigmoid, 4 logit */
int ori_special_f64(int op, const double* in, double* out, int64_t count, void* stream);

/* ---- node expectations (gamma.py:37-61): E = a1/a2, Elog = psi(a1) - log(a2), eE = exp(Elog) ---- */
/* any of E, Elog, eE may be NULL */
int ori_gamma_expect_f32(const float* a1, const float* a2, float* E, float* Elog, float* eE,
                         int64_t count, void* stream);

/* ---- the CAVI iteration, device-resident state -------------------------------------------------- */
/* Scratch floats the tensor path needs for a rank owning n_rows cells of p genes at padded latent dimension KP. */
int64_t ori_tc_workspace_floats(int64_t n_rows, int32_t p, int32_t KP);
/* Size of ori_problem_t::det_ws in doubles (ORI_F_DETERMINISTIC). */
int64_t ori_det_workspace_doubles(int64_t n_rows, int32_t p, int32_t KP);
/* 1 when the calls below will take the tensor path for this problem, 0 for the CUDA-core kernels. */
int ori_uses_tensor_path(const ori_problem_t* P);
/* Validate a problem description (shapes, alignment, null pointers). */
int ori_problem_check(const ori_problem_t* P);
/* Constant data statistics: sum lgamma(X+1), nnz -> red64 slots ORI_R64_LGAMX, ORI_R64_NNZ (ori_mstep ORI_M_INIT and
 * ORI_M_INIT_KEEP copy them to scal); column sums of (X>0) -> red64[0..p). */
int ori_count_stats(const ori_problem_t* P, void* stream);
/* Expectations of generation `gen` from (a1,a2,b1,b2) (zigap.py:160-165) + their column sums. */
int ori_init_expectations(const ori_problem_t* P, int gen, void* stream);
/* Zero-fill the accumulators of one iteration: Zi, a2s, red64 and (genes != 0) red32 (zigap.py:81-83). */
int ori_zero_accumulators(const ori_problem_t* P, int genes, void* stream);
/* Row pass ("KA"): Zi, a2s, colsum D_hat, ELBO partials from X and the state of generation gen_old. */
int ori_pass_rows(const ori_problem_t* P, int gen_old, void* stream);
/* U update (zigap.py:115-120) into generation 1-gen_old, plus sum_i log U_hat, sum_i U_hat.
 * write_state: 1 regular; 0 only the ELBO term of the swept state; 2 expectations of generation gen_old
 * from (a1, a2) with their column sums; 3 the same without touching any sum (host-streamed slabs). */
int ori_row_update(const ori_problem_t* P, int gen_old, int write_state, void* stream);
/* Gene pass ("KA'"): Zj and b2s = D_hat^T U_hat_new (zigap.py:94,124) into red32. */
int ori_pass_genes(const ori_problem_t* P, int gen_old, void* stream);
/* V update (zigap.py:123-128) from red32 (already summed over ranks). */
int ori_gene_update(const ori_problem_t* P, int write_state, void* stream);
/* M-step / finalisation (zigap.py:143-158), see ORI_M_*; reads red64 (already summed over ranks). */
int ori_mstep(const ori_problem_t* P, int mode, void* stream);
/* Convenience for world size 1: one full `step()` (base.py:54-56) = zero accumulators, row pass,
 * U update, gene pass, V update, M-step.  Flips the generation: new state is in 1-gen_old. */
int ori_cavi_step(const ori_problem_t* P, int gen_old, void* stream);
/* First half / second half of the above around the caller's allreduce of red32 and red64. */
int ori_cavi_step_local(const ori_problem_t* P, int gen_old, void* stream);
int ori_cavi_step_global(const ori_problem_t* P, int gen_old, void* stream);
/* Flush of the one-pass lag: pi(t), ELBO(t) of the current state (generation gen). Local part,
 * then (after the caller's allreduce of red64) ori_mstep(P, ORI_M_FINALIZE). */
int ori_finalize_local(const ori_problem_t* P, int gen, void* stream);

/* Materialise D_hat = float32(p_d) (zigap.py:131-136) for rows [row0, row0+nrows) of generation gen. */
int ori_dropout_posterior_f32(const ori_problem_t* P, int gen, float* out, int64_t ldo,
                              int64_t row0, int64_t nrows, void* stream);

/* ---- convergence metrics of the reference's drivers (base.py:58-82, sparse_zigap.py:44-51) ------- */
/* out[r] = sum_j X[r, j], float32 (device pointers). */
int ori_row_sums_f32(const float* X, int64_t ldx, int64_t n_rows, int32_t p, float* out, void* stream);
/* out[c] = sum_i X[i, c] over this rank's rows, float64 (device pointers). */
int ori_column_sums_f64(const float* X, int64_t ldx, int64_t n_rows, int32_t p, double* out, void* stream);
/* The same two sums of a uint16 count matrix (ORI_F_X_U16 storage; ldx in elements). */
int ori_row_sums_u16_f32(const uint16_t* X, int64_t ldx, int64_t n_rows, int32_t p, float* out, void* stream);
int ori_column_sums_u16_f64(const uint16_t* X, int64_t ldx, int64_t n_rows, int32_t p, double* out, void* stream);
/* The three zero-inflated Poisson log-likelihood sums behind reconstruction_deviance / explained_deviance for
 * this rank's rows: rate = U_hat V_hat^T masked where round(D_hat) == 0 (base.py:64-67), rate = X (saturated,
 * :68), rate = column means of X (:76; col_mean [p] float64, all ranks).  pi [p] float64 = the finalised pi_d.
 * out_int[3]: every entry's term truncated toward zero to int64 before a wrapping sum, exactly what the
 * reference's integer output buffer does (sparse_zigap.py:45; -inf / NaN become INT64_MIN); out_f64[3]: the
 * plain float64 sums, or NULL (then zero entries of genes with 1 - pi >= 1/e, whose terms all truncate to 0, are
 * skipped).  Both are ACCUMULATED into (caller zero-fills). */
int ori_deviance_sums(const ori_problem_t* P, int gen, const double* pi, const double* col_mean,
                      long long* out_int, double* out_f64, void* stream);

/* ---- operator-level drop-ins with HOST buffers (the reference's plugin seam) --------------------
 * A context keeps the device side of these calls between invocations: two streams, the events, the slab staging
 * buffers and the tensor-path workspaces (grow-only: sized by the largest call so far).  After the first call of a
 * given shape a call creates no stream or event and allocates no device memory.  Row slabs of >= 2^21 entries run the
 * tcgen05 / TMA passes (D_hat is an explicit input of this seam, so it is folded into X and the GaP-shaped kernels are
 * used), smaller problems the CUDA-core kernels.  One call at a time per context (internally serialised).
 * slab_rows: cells per slab (rounded to a multiple of 128), 0 = ~256 MB of X per slab. */
typedef struct ori_ctx ori_ctx_t;
int ori_ctx_create(ori_ctx_t** out, int64_t slab_rows);
int ori_ctx_destroy(ori_ctx_t* ctx);
/* Counters of a context (NULL: the default context used by the *_host entry points): calls served, cudaMalloc calls
 * made, slabs processed by the tensor / the CUDA-core kernels.  Any output pointer may be NULL. */
int ori_ctx_stats(ori_ctx_t* ctx, unsigned long long* calls, unsigned long long* device_allocations,
                  unsigned long long* tensor_slabs, unsigned long long* simt_slabs);

/* Same argument list and semantics as `ZIGaP.compute_Z_q_expectations` (zigap.py:79-95): every array
 * is a C-contiguous float32 HOST array; DZ_hat_i [n x K], DZ_hat_j [p x K] are overwritten.
 * DZ_exp_logsum_hat may be NULL (never read by the reference, zigap.py:95); when given it is filled.
 * `quirk` != 0 weights DZ_hat_j by D_hat[i, k] exactly like zigap.py:94.  Synchronous. */
int ori_zigap_compute_Z_q_expectations_host(float* DZ_hat_i, float* DZ_hat_j, float* DZ_exp_logsum_hat,
                                            const float* log_U_hat, const float* log_V_hat,
                                            const float* D_hat, const float* X,
                                            int64_t n, int64_t p, int64_t K, int quirk);
/* `GaP.compute_Z_q_expectations` (gap.py:67-80). */
int ori_gap_compute_Z_q_expectations_host(float* Z_hat_i, float* Z_hat_j,
                                          const float* log_U_hat, const float* log_V_hat,
                                          const float* X, int64_t n, int64_t p, int64_t K);
/* The same two operators on an explicit context (the *_host forms use a process-wide default context). */
int ori_zigap_compute_Z_q_expectations_ctx(ori_ctx_t* ctx, float* DZ_hat_i, float* DZ_hat_j, float* DZ_exp_logsum_hat,
                                           const float* log_U_hat, const float* log_V_hat,
                                           const float* D_hat, const float* X,
                                           int64_t n, int64_t p, int64_t K, int quirk);
int ori_gap_compute_Z_q_expectations_ctx(ori_ctx_t* ctx, float* Z_hat_i, float* Z_hat_j,
                                         const float* log_U_hat, const float* log_V_hat,
                                         const float* X, int64_t n, int64_t p, int64_t K);
/* `SparseZIGaP.compute_Z_q_expectations` (sparse_zigap.py:100-116), same argument order: C-contiguous float32 HOST
 * arrays, log_U_hat [n x K], log_V_hat = E[log V'] [p x K], S_tilde = the mask (p_s > tau) and S_hat [p x K], D_hat and
 * X [n x p].  DSZ_hat [n x K], DZ_hat [p x K] and DZ_exp_logsum_hat [p x K] are overwritten; all three outputs and
 * D_hat are required (the reference's S-step reads the third, sparse_zigap.py:155).  K <= 64 (ORI_EUNSUPPORTED above).
 * Row slabs of >= 2^21 entries with K <= 32 run the tcgen05 passes with fp32-grade contractions (ORI_F_PRECISE), all
 * other slabs the CUDA-core kernels.  Synchronous. */
int ori_sparse_zigap_compute_Z_q_expectations_host(float* DSZ_hat, float* DZ_hat, float* DZ_exp_logsum_hat,
                                                   const float* log_U_hat, const float* log_V_hat,
                                                   const float* S_tilde, const float* S_hat,
                                                   const float* D_hat, const float* X,
                                                   int64_t n, int64_t p, int64_t K);
int ori_sparse_zigap_compute_Z_q_expectations_ctx(ori_ctx_t* ctx, float* DSZ_hat, float* DZ_hat, float* DZ_exp_logsum_hat,
                                                  const float* log_U_hat, const float* log_V_hat,
                                                  const float* S_tilde, const float* S_hat,
                                                  const float* D_hat, const float* X,
                                                  int64_t n, int64_t p, int64_t K);

/* ---- synthetic counts on device (SURVEY.md section 8d; bench only) ------------------------------- */
/* X[i, j] = Poisson(g_ij * sum_k U*[i,k] V*[j,k]) * Bernoulli(pi_j) with U*, V* ~ Gamma(2, 1/2),
 * g ~ Gamma(2, 1/2) (negative-binomial over-dispersion; nb = 0 gives plain Poisson) and keep
 * probability pi_j ~ Beta(1, 1/z - 1); counter-based RNG (Philox-4x32-10) keyed by (seed, GLOBAL row,
 * gene), so any row sharding produces the same matrix.  Rows [row0, row0+n_rows) are written.
 * Scratch (caller-owned, device): Ustar [n_rows x K], Vstar [p x K], pi [p]. */
int ori_synth_counts_f32(float* X, int64_t ldx, int64_t row0, int64_t n_rows, int32_t p, int32_t K,
                         uint64_t seed, float zero_level, int nb, float* Ustar, float* Vstar, float* pi,
                         void* stream);

/* ---- compact count storage (count-matrix ingest, oriana/singlecell/cmatrix.py:56-61) -------------- */
/* dst[r, c] = (float)src[r, c] for unsigned integer counts of elem_bytes = 1 or 2 (device pointers; lds, ldd in
 * elements, ldd a multiple of 4, dst 16-byte aligned).  Lets a host keep X as uint8 / uint16 and stream a
 * quarter / half of the bytes per step; the kernels always see the float32 matrix of zigap.py:112. */
int ori_widen_counts_f32(const void* src, int elem_bytes, int64_t lds, float* dst, int64_t ldd,
                         int64_t rows, int32_t p, void* stream);

/* Sparse ingest: dst[r, 32 w + l] = bit l of bitmap[r, w] ? (float)nz[rowoff[r] - base + rank of that bit in row r] : 0
 * (device pointers; bitmap rows of words_per_row >= ceil(p / 32) uint32 words, pad bits zero; nz = the non-zero counts
 * of the rows in gene order as saturating bytes, 255 = see ori_scatter_counts_f32; rowoff[r] = position of row r's
 * first byte in the caller's whole stream, base = position of nz[0]).  p / 8 + nnz bytes per cell cross PCIe instead
 * of p: the sparse form of cmatrix.py:100-104 (as_sparse_matrix) as the streaming format of the host-facing step. */
int ori_expand_bitmap_counts_f32(const uint32_t* bitmap, int64_t words_per_row, const uint8_t* nz,
                                 const int64_t* rowoff, int64_t base, float* dst, int64_t ldd, int64_t rows,
                                 int32_t p, void* stream);

/* CSR ingest, the device side of cmatrix.py:39-54 (as_sparse_matrix): rows [0, rows) of a CSR slab into a dense
 * [rows x ldd] matrix.  Row r's non-zeros are [indptr[r] - base, indptr[r + 1] - base) of indices / values (device
 * pointers; base = indptr of the slab's first row, so a slab cut from the middle of a matrix needs no rebasing).  The
 * indices of a row are distinct (canonical CSR): idx_bytes = 2 (uint16, p <= 65536) or 4 (int32).  values: ORI_CSR_U8,
 * ORI_CSR_U16 or ORI_CSR_F32 (the value type's size in bytes).  dst: dst_bytes = 4 (float32 X) or 2 (uint16 X, the
 * ORI_F_X_U16 storage; ORI_CSR_F32 values are rejected there), 16-byte aligned, ldd a multiple of 16 / dst_bytes.
 * EVERY element of the destination is written -- counts, zeros and the pad columns p..ldd-1 -- so it needs no memset.
 * indices / values may be null when the rows hold no non-zero. */
#define ORI_CSR_U8 1
#define ORI_CSR_U16 2
#define ORI_CSR_F32 4
int ori_expand_csr_counts(const int64_t* indptr, int64_t base, const void* indices, int32_t idx_bytes,
                          const void* values, int32_t val_type, void* dst, int32_t dst_bytes, int64_t ldd,
                          int64_t rows, int32_t p, void* stream);

/* Escapes of the saturating uint8 encoding: X[row[e] - row0, col[e]] = val[e] (device pointers; row = global
 * cell index, row0 = first cell of the slab held in X).  Entries outside the slab are ignored. */
int ori_scatter_counts_f32(float* X, int64_t ldx, int64_t row0, int64_t rows, int32_t p, const int32_t* row,
                           const int32_t* col, const float* val, int64_t count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ORIANA_B200_H */
