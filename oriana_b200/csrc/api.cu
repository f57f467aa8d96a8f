// api.cu -- extern "C" entry points of liboriana_b200.so (declared in include/oriana_b200.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>
#include "common.cuh"
#include "special.cuh"

namespace ori {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static std::atomic<unsigned long long> g_launches{0};

int check_launch(const char* what, int n_kernels) {
    g_launches.fetch_add((unsigned long long)n_kernels, std::memory_order_relaxed);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(ORI_ECUDA, "%s: %s", what, cudaGetErrorString(e));
    return ORI_OK;
}

#define ORI_CUDA(call)                                                                             \
    do {                                                                                           \
        const cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess) return ori::set_error(ORI_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)
#define ORI_TRY(call)              \
    do {                           \
        const int r_ = (call);     \
        if (r_ != ORI_OK) return r_; \
    } while (0)

// ---- small elementwise kernels --------------------------------------------------------------------
__global__ void k_special_f64(int op, const double* __restrict__ in, double* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double x = in[i];
    double y;
    switch (op) {
        case 0: y = digamma_f64(x); break;
        case 1: y = trigamma_f64(x); break;
        case 2: y = inverse_digamma_f64(x); break;
        case 3: y = sigmoid_f64(x); break;
        default: y = logit_f64(x); break;
    }
    out[i] = y;
}

// gamma.py:37-61
__global__ void k_gamma_expect(const float* __restrict__ a1, const float* __restrict__ a2,
                               float* __restrict__ E, float* __restrict__ Elog, float* __restrict__ eE,
                               long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float h1 = a1[i], h2 = a2[i];
    const float l = (float)digamma_f64((double)h1) - logf(h2);
    if (E) E[i] = (float)((double)h1 / (double)h2);
    if (Elog) Elog[i] = l;
    if (eE) eE[i] = expf(l);
}

// operator-level helpers: padded exp of a [rows x K] log-expectation array, optional extra weight
__global__ void k_exp_pad(const float* __restrict__ logE, const float* __restrict__ W, long long ldw,
                          int mul_log, float* __restrict__ out, long long rows, int K, int KP,
                          float* __restrict__ thr_out = nullptr) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * KP) return;
    const long long i = idx / KP; const int k = (int)(idx % KP);
    float v = 0.f;
    if (k < K) {
        float m = -INFINITY;                       // centred exponent of the row (special.cuh): outputs are ratios
        for (int q = 0; q < K; ++q) m = fmaxf(m, logE[i * K + q]);
        if (thr_out && k == 0) thr_out[i] = underflow_thr_f32(m);   // the reference's float32 exp underflow (zigap.py:86-90)
        const float l = logE[i * K + k];
        v = centred_exp_f32(l, m);
        if (W) v *= W[i * ldw + k];
        if (mul_log && v != 0.f) v *= l;
    }
    out[idx] = v;
}
// sparse model's gene-side operands (sparse_zigap.py:109, :114): eVd = centred exp(lV) * S_tilde (denominator), eVz =
// eVd * S_hat (row sums); thr from the UNMASKED lV -- the reference's mask multiplies after its float32 exp
__global__ void k_exp_pad_sparse(const float* __restrict__ logE, const float* __restrict__ St, const float* __restrict__ Sh,
                                 float* __restrict__ eVd, float* __restrict__ eVz, float* __restrict__ thr_out,
                                 long long rows, int K, int KP) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * KP) return;
    const long long i = idx / KP; const int k = (int)(idx % KP);
    float vd = 0.f, vz = 0.f;
    if (k < K) {
        float m = -INFINITY;
        for (int q = 0; q < K; ++q) m = fmaxf(m, logE[i * K + q]);
        if (k == 0) thr_out[i] = underflow_thr_f32(m);
        vd = centred_exp_f32(logE[i * K + k], m) * St[i * K + k];
        vz = vd * Sh[i * K + k];
    }
    eVd[idx] = vd;
    eVz[idx] = vz;
}
__global__ void k_mul(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] * b[i];
}
// out[i,k] (stride K) = acc[i,k] * e[i,k] (stride KP)  [+ acc2[i,k] * e[i,k] * l[i,k]]
__global__ void k_scale_unpad(const float* __restrict__ acc, const float* __restrict__ e,
                              const float* __restrict__ acc2, const float* __restrict__ l,
                              float* __restrict__ out, long long rows, int K, int KP) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * K) return;
    const long long i = idx / K; const int k = (int)(idx % K);
    float v = acc[i * KP + k] * e[i * KP + k];
    if (acc2) v += acc2[i * KP + k] * e[i * KP + k] * l[i * K + k];
    out[idx] = v;
}

static int pad_k(long long K) { return K <= 8 ? 8 : K <= 16 ? 16 : K <= 32 ? 32 : K <= 64 ? 64 : -1; }

}  // namespace ori

using namespace ori;

extern "C" {

int ori_version(void) { return 101; }

unsigned long long ori_kernel_launches(void) { return ori::g_launches.load(std::memory_order_relaxed); }

int ori_last_error(char* buf, size_t len) {
    if (buf && len) { strncpy(buf, g_err, len - 1); buf[len - 1] = 0; }
    return (int)strlen(g_err);
}

int ori_device_check(int dev) {
    cudaDeviceProp prop;
    ORI_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) return set_error(ORI_ENODEV, "device %d is sm_%d%d, this library is sm_100a only", dev, prop.major, prop.minor);
    return ORI_OK;
}

int ori_special_f64(int op, const double* in, double* out, int64_t count, void* stream) {
    if (op < 0 || op > 4) return set_error(ORI_EINVAL, "ori_special_f64: bad op %d", op);
    if (count < 0 || (count && (!in || !out))) return set_error(ORI_EINVAL, "ori_special_f64: null buffer");
    if (count == 0) return ORI_OK;
    k_special_f64<<<cdiv(count, 256), 256, 0, (cudaStream_t)stream>>>(op, in, out, count);
    return check_launch("k_special_f64");
}

int ori_gamma_expect_f32(const float* a1, const float* a2, float* E, float* Elog, float* eE,
                         int64_t count, void* stream) {
    if (count < 0 || (count && (!a1 || !a2))) return set_error(ORI_EINVAL, "ori_gamma_expect_f32: null buffer");
    if (count == 0) return ORI_OK;
    k_gamma_expect<<<cdiv(count, 256), 256, 0, (cudaStream_t)stream>>>(a1, a2, E, Elog, eE, count);
    return check_launch("k_gamma_expect");
}

int ori_problem_check(const ori_problem_t* P) {
    if (!P) return set_error(ORI_EINVAL, "null problem");
    if (P->n_rows < 0 || P->p <= 0 || P->K <= 0) return set_error(ORI_EINVAL, "bad shape n_rows=%lld p=%d K=%d", (long long)P->n_rows, P->p, P->K);
    if (P->K > 64) return set_error(ORI_EUNSUPPORTED, "K=%d > 64 is not supported", P->K);
    if (P->KP < P->K || (P->KP != 8 && P->KP != 16 && P->KP != 32 && P->KP != 64))
        return set_error(ORI_EINVAL, "KP=%d must be 8, 16, 32 or 64 and >= K=%d", P->KP, P->K);
    if (P->tc_ws && (((uintptr_t)P->tc_ws & 127) || P->tc_ws_floats < tc_workspace_floats(P->n_rows, P->p, P->KP)))
        return set_error(ORI_EINVAL, "tc_ws must be 128-byte aligned and hold ori_tc_workspace_floats() floats");
    if (P->flags & ORI_F_DETERMINISTIC) {
        if (!P->tc_ws && !det_simt_ok(P->n_rows, P->p))
            return set_error(ORI_EUNSUPPORTED, "ORI_F_DETERMINISTIC on the CUDA-core kernels is limited to 2^26 matrix entries");
        if (!P->det_ws || P->det_ws_doubles < det_carve(nullptr, P->n_rows, P->p).doubles)
            return set_error(ORI_EINVAL, "ORI_F_DETERMINISTIC needs det_ws of ori_det_workspace_doubles() doubles");
    }
    if (P->ldx < P->p || (P->ldx & 3)) return set_error(ORI_EINVAL, "ldx=%lld must be >= p and a multiple of 4", (long long)P->ldx);
    if ((P->flags & ORI_F_X_U16) && (P->ldx & 7))     // uint16 rows start on 16 bytes (TMA)
        return set_error(ORI_EINVAL, "ORI_F_X_U16: ldx=%lld must be a multiple of 8", (long long)P->ldx);
    if (P->n_total < P->n_rows || P->n_total <= 0) return set_error(ORI_EINVAL, "n_total=%lld < n_rows", (long long)P->n_total);
    if ((P->flags & ORI_F_QUIRK) && P->p < P->K) return set_error(ORI_EINVAL, "quirk mode needs p >= K (zigap.py:94 reads D_hat[i, k])");
    const void* need[] = {P->a1, P->a2, P->U_hat[0], P->U_hat[1], P->eU[0], P->eU[1], P->Zi, P->b1, P->b2,
                          P->V_hat, P->eV, P->red32, P->hyper, P->red64, P->gsum, P->scal, P->elbo_trace};
    for (size_t i = 0; i < sizeof(need) / sizeof(need[0]); ++i)
        if (!need[i]) return set_error(ORI_EINVAL, "null buffer #%zu in ori_problem_t", i);
    if (P->n_rows > 0 && !P->X) return set_error(ORI_EINVAL, "null X");
    if (P->flags & ORI_F_DROPOUT)
        if (!P->a2s || !P->lp || !P->pfloor || !P->pi_d) return set_error(ORI_EINVAL, "dropout buffers missing");
    if ((P->flags & ORI_F_QUIRK) && !P->eUw) return set_error(ORI_EINVAL, "quirk mode needs eUw");
    if ((P->flags & ORI_F_ELBO) && (!P->xcol || (P->n_rows > 0 && !P->xrow)))
        return set_error(ORI_EINVAL, "ORI_F_ELBO needs xrow / xcol (row and column sums of X)");
    if (P->flags & ORI_F_SPARSE) {
        if (!(P->flags & ORI_F_DROPOUT) || (P->flags & (ORI_F_QUIRK | ORI_F_ELBO)))
            return set_error(ORI_EINVAL, "ORI_F_SPARSE needs ORI_F_DROPOUT and excludes ORI_F_QUIRK / ORI_F_ELBO");
        if (!P->p_s || !P->logV || !P->eVd || !P->eVz || !P->Vh_old || !P->eUl[0] || !P->eUl[1] || !P->pi_s)
            return set_error(ORI_EINVAL, "sparse buffers missing");
        if (((uintptr_t)P->eVd & 15) || ((uintptr_t)P->eVz & 15) || ((uintptr_t)P->Vh_old & 15))
            return set_error(ORI_EINVAL, "eVd, eVz, Vh_old must be 16-byte aligned");
    } else if (P->eUl[0] || P->eUl[1]) {
        return set_error(ORI_EINVAL, "eUl (the third gene sum) needs ORI_F_SPARSE");
    }
    if (((uintptr_t)P->X & 15) || ((uintptr_t)P->eV & 15) || ((uintptr_t)P->V_hat & 15))
        return set_error(ORI_EINVAL, "X, eV, V_hat must be 16-byte aligned");
    return ORI_OK;
}

static size_t red64_bytes(const ori_problem_t* P) { return sizeof(double) * (size_t)ORI_RED64_DOUBLES(P->p, P->KP); }
static size_t gsum_bytes(const ori_problem_t* P) { return sizeof(double) * (size_t)ORI_GSUM_DOUBLES(P->KP); }
static size_t rowf_bytes(const ori_problem_t* P) { return sizeof(float) * (size_t)P->n_rows * P->KP; }

int ori_count_stats(const ori_problem_t* P, void* stream) {
    ORI_TRY(ori_problem_check(P));
    cudaStream_t st = (cudaStream_t)stream;
    ORI_CUDA(cudaMemsetAsync(P->red64, 0, red64_bytes(P), st));
    if (P->n_rows == 0) return ORI_OK;
    return launch_count_stats(P, st);
}

int ori_init_expectations(const ori_problem_t* P, int gen, void* stream) {
    ORI_TRY(ori_problem_check(P));
    cudaStream_t st = (cudaStream_t)stream;
    ORI_CUDA(cudaMemsetAsync(P->gsum, 0, gsum_bytes(P), st));
    if (P->n_rows > 0) ORI_TRY(launch_row_update(P, gen, 2, st));
    return launch_gene_update(P, 2, st);
}

// row pass: tensor path = operand preparation + tcgen05 kernel (statistics come from the gene pass there)
static int pass_rows_any(const ori_problem_t* P, int gen_old, cudaStream_t st) {
    if (!tc_eligible(P)) return launch_pass_rows_simt(P, gen_old, st);
    ORI_TRY(launch_tc_prep_genes(P, st));
    return launch_pass_rows_tc(P, gen_old, st);
}
// gene sums: Zj | b2s, and with eUl[gen_old] the third sum sum_i R_ij eU_ik E[log U_ik] into red32 block 2 (zigap.py:95,
// sparse_zigap.py:116) -- in the same sweep on the CUDA-core kernels, in a second, dropout-free one on the tensor path
static int gene_sums(const ori_problem_t* P, int gen_old, cudaStream_t st) {
    if (!tc_eligible(P)) return launch_pass_genes_simt(P, gen_old, st);
    ORI_TRY(launch_tc_prep_rows(P, gen_old, st));
    ORI_TRY(launch_pass_genes_tc(P, gen_old, st));
    if (!P->eUl[gen_old]) return ORI_OK;
    ORI_TRY(launch_tc_prep_rows_logsum(P, gen_old, st));
    return launch_pass_genes_logsum_tc(P, gen_old, st);
}
// the models' gene pass: under the quirk the Zj weight eU * D_hat[:, :K] (zigap.py:94) comes from their own state first
static int pass_genes_any(const ori_problem_t* P, int gen_old, cudaStream_t st) {
    if (P->flags & ORI_F_QUIRK) ORI_TRY(launch_quirk_weights(P, gen_old, st));
    return gene_sums(P, gen_old, st);
}

int64_t ori_tc_workspace_floats(int64_t n_rows, int32_t p, int32_t KP) { return tc_workspace_floats(n_rows, p, KP); }
int64_t ori_det_workspace_doubles(int64_t n_rows, int32_t p, int32_t KP) { (void)KP; return det_carve(nullptr, n_rows, p).doubles; }

int ori_uses_tensor_path(const ori_problem_t* P) { return (P && tc_eligible(P)) ? 1 : 0; }

int ori_pass_rows(const ori_problem_t* P, int gen_old, void* stream) {
    ORI_TRY(ori_problem_check(P));
    if (P->n_rows == 0) return ORI_OK;
    return pass_rows_any(P, gen_old, (cudaStream_t)stream);
}

int ori_row_update(const ori_problem_t* P, int gen_old, int write_state, void* stream) {
    ORI_TRY(ori_problem_check(P));
    if (P->n_rows == 0) return ORI_OK;
    return launch_row_update(P, gen_old, write_state, (cudaStream_t)stream);
}

int ori_pass_genes(const ori_problem_t* P, int gen_old, void* stream) {
    ORI_TRY(ori_problem_check(P));
    if (P->n_rows == 0) return ORI_OK;
    return pass_genes_any(P, gen_old, (cudaStream_t)stream);
}

int ori_gene_update(const ori_problem_t* P, int write_state, void* stream) {
    ORI_TRY(ori_problem_check(P));
    cudaStream_t st = (cudaStream_t)stream;
    ORI_CUDA(cudaMemsetAsync(P->gsum, 0, gsum_bytes(P), st));
    return launch_gene_update(P, write_state, st);
}

int ori_mstep(const ori_problem_t* P, int mode, void* stream) {
    ORI_TRY(ori_problem_check(P));
    if (mode < 0 || mode > 4) return set_error(ORI_EINVAL, "ori_mstep: bad mode %d", mode);
    return launch_mstep(P, mode, (cudaStream_t)stream);
}

static int zero_accumulators(const ori_problem_t* P, cudaStream_t st, bool genes) {
    if (P->n_rows > 0) {
        ORI_CUDA(cudaMemsetAsync(P->Zi, 0, rowf_bytes(P), st));
        if (P->flags & ORI_F_DROPOUT) ORI_CUDA(cudaMemsetAsync(P->a2s, 0, rowf_bytes(P), st));
    }
    if (genes) ORI_CUDA(cudaMemsetAsync(P->red32, 0, sizeof(float) * (size_t)ORI_RED32_FLOATS(P->p, P->KP, P->eUl[0] != nullptr), st));
    ORI_CUDA(cudaMemsetAsync(P->red64, 0, red64_bytes(P), st));
    return ORI_OK;
}

int ori_zero_accumulators(const ori_problem_t* P, int genes, void* stream) {
    ORI_TRY(ori_problem_check(P));
    return zero_accumulators(P, (cudaStream_t)stream, genes != 0);
}

int ori_cavi_step_local(const ori_problem_t* P, int gen_old, void* stream) {
    ORI_TRY(ori_problem_check(P));
    cudaStream_t st = (cudaStream_t)stream;
    ORI_TRY(zero_accumulators(P, st, true));
    if (P->n_rows == 0) return ORI_OK;
    ORI_TRY(pass_rows_any(P, gen_old, st));
    ORI_TRY(launch_row_update(P, gen_old, 1, st));
    return pass_genes_any(P, gen_old, st);
}

int ori_cavi_step_global(const ori_problem_t* P, int gen_old, void* stream) {
    (void)gen_old;
    ORI_TRY(ori_problem_check(P));
    cudaStream_t st = (cudaStream_t)stream;
    ORI_CUDA(cudaMemsetAsync(P->gsum, 0, gsum_bytes(P), st));
    ORI_TRY(launch_gene_update(P, 1, st));
    return launch_mstep(P, ORI_M_STEP, st);
}

int ori_cavi_step(const ori_problem_t* P, int gen_old, void* stream) {
    ORI_TRY(ori_cavi_step_local(P, gen_old, stream));
    return ori_cavi_step_global(P, gen_old, stream);
}

int ori_finalize_local(const ori_problem_t* P, int gen, void* stream) {
    ORI_TRY(ori_problem_check(P));
    cudaStream_t st = (cudaStream_t)stream;
    const bool tc = tc_eligible(P);
    ORI_TRY(zero_accumulators(P, st, tc));
    if (P->n_rows == 0) return ORI_OK;
    ORI_TRY(pass_rows_any(P, gen, st));
    ORI_TRY(launch_row_update(P, gen, 0, st));
    // tensor path: colsum D_hat and the ELBO partials come out of the gene pass (red32 is scratch here)
    return tc ? pass_genes_any(P, gen, st) : ORI_OK;
}

int ori_dropout_posterior_f32(const ori_problem_t* P, int gen, float* out, int64_t ldo,
                              int64_t row0, int64_t nrows, void* stream) {
    ORI_TRY(ori_problem_check(P));
    if (!(P->flags & ORI_F_DROPOUT)) return set_error(ORI_EINVAL, "model has no dropout layer");
    if (!out || ldo < P->p || row0 < 0 || row0 + nrows > P->n_rows) return set_error(ORI_EINVAL, "bad slab");
    return launch_dropout_posterior(P, gen, out, ldo, row0, nrows, (cudaStream_t)stream);
}

int ori_row_sums_f32(const float* X, int64_t ldx, int64_t n_rows, int32_t p, float* out, void* stream) {
    if (n_rows < 0 || p <= 0 || ldx < p || (n_rows > 0 && (!X || !out))) return set_error(ORI_EINVAL, "ori_row_sums_f32: bad argument");
    return launch_row_sums(X, ldx, n_rows, p, out, (cudaStream_t)stream);
}

int ori_column_sums_f64(const float* X, int64_t ldx, int64_t n_rows, int32_t p, double* out, void* stream) {
    if (n_rows < 0 || p <= 0 || ldx < p || !out || (n_rows > 0 && !X)) return set_error(ORI_EINVAL, "ori_column_sums_f64: bad argument");
    ORI_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)p, (cudaStream_t)stream));
    return launch_col_sums(X, ldx, n_rows, p, out, (cudaStream_t)stream);
}

int ori_row_sums_u16_f32(const uint16_t* X, int64_t ldx, int64_t n_rows, int32_t p, float* out, void* stream) {
    if (n_rows < 0 || p <= 0 || ldx < p || (n_rows > 0 && (!X || !out))) return set_error(ORI_EINVAL, "ori_row_sums_u16_f32: bad argument");
    return launch_row_sums(X, ldx, n_rows, p, out, (cudaStream_t)stream);
}

int ori_column_sums_u16_f64(const uint16_t* X, int64_t ldx, int64_t n_rows, int32_t p, double* out, void* stream) {
    if (n_rows < 0 || p <= 0 || ldx < p || !out || (n_rows > 0 && !X)) return set_error(ORI_EINVAL, "ori_column_sums_u16_f64: bad argument");
    ORI_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * (size_t)p, (cudaStream_t)stream));
    return launch_col_sums(X, ldx, n_rows, p, out, (cudaStream_t)stream);
}

int ori_deviance_sums(const ori_problem_t* P, int gen, const double* pi, const double* col_mean,
                      long long* out_int, double* out_f64, void* stream) {
    ORI_TRY(ori_problem_check(P));
    if (!(P->flags & ORI_F_DROPOUT)) return set_error(ORI_EINVAL, "the deviance metrics need the dropout layer (sparse_zigap.py:44-51)");
    if (!pi || !col_mean || !out_int || gen < 0 || gen > 1) return set_error(ORI_EINVAL, "ori_deviance_sums: bad argument");
    if (P->n_rows == 0) return ORI_OK;
    // integer sums of a problem on the tensor path: the tcgen05 pass; the float64 sums (int_quirk=False) and small
    // problems: the CUDA-core kernel
    if (!out_f64 && tc_eligible(P) && !(P->flags & ORI_F_QUIRK))
        return launch_deviance_tc(P, gen, pi, col_mean, out_int, (cudaStream_t)stream);
    return launch_deviance(P, gen, pi, col_mean, out_int, out_f64, (cudaStream_t)stream);
}

}  // extern "C"

// ---- operator-level drop-in with HOST buffers ------------------------------------------------------
// A context owns everything a call needs on the device -- two streams, the events, the slab staging buffers, the
// tensor-path workspaces -- and keeps it between calls: after the first call of a given shape no cudaMalloc, no stream
// or event is created (ori_ctx_stats counts them).  The *_host entry points without a context argument use one
// process-wide default context behind a mutex.
#include <condition_variable>
#include <mutex>
#include <thread>

// Host arrays of the reference are pageable numpy memory: a plain cudaMemcpy from them runs at ~11 GB/s (one driver thread
// staging through its own small pinned buffer).  CopyPool + the context's ring of pinned staging chunks do the same
// staging with several threads, so that the DMA of chunk i overlaps the memcpy of chunk i+1 (operator seam, bench.py
// `operator_seam`).
struct CopyPool {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    const char* src = nullptr; char* dst = nullptr; size_t bytes = 0;
    unsigned long long gen = 0;
    int pending = 0;
    bool stop = false;
    void start(int n) {
        for (int i = 0; i < n; ++i) th.emplace_back([this, i, n] { run(i, n); });
    }
    void run(int i, int n) {
        unsigned long long seen = 0;
        for (;;) {
            const char* s_; char* d_; size_t b_;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_go.wait(lk, [&] { return stop || gen != seen; });
                if (stop) return;
                seen = gen; s_ = src; d_ = dst; b_ = bytes;
            }
            const size_t per = ((b_ + n - 1) / n + 63) & ~(size_t)63;
            const size_t lo = per * i < b_ ? per * i : b_, hi = lo + per < b_ ? lo + per : b_;
            if (hi > lo) memcpy(d_ + lo, s_ + lo, hi - lo);
            {
                std::lock_guard<std::mutex> lk(mu);
                if (--pending == 0) cv_done.notify_one();
            }
        }
    }
    void copy(void* d, const void* s, size_t b) {
        if (th.empty() || b < (1u << 20)) { memcpy(d, s, b); return; }
        std::unique_lock<std::mutex> lk(mu);
        src = (const char*)s; dst = (char*)d; bytes = b; pending = (int)th.size(); ++gen;
        cv_go.notify_all();
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    void shutdown() {
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv_go.notify_all();
        for (auto& t : th) t.join();
        th.clear();
    }
};

struct ori_ctx {
    cudaStream_t st[2] = {nullptr, nullptr};
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    // pinned staging ring for pageable host inputs
    static constexpr int NSTG = 4;
    static constexpr size_t STG_BYTES = 32u << 20;
    void* stg[NSTG] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t stg_ev[NSTG] = {nullptr, nullptr, nullptr, nullptr};
    bool stg_busy[NSTG] = {false, false, false, false};
    int stg_next = 0;
    CopyPool pool;
    unsigned long long staged_bytes = 0;
    struct Buf { void* p = nullptr; size_t cap = 0; };
    enum { X0, X1, D0, D1, LUS0, LUS1, EU0, EU1, EUW0, EUW1, EUL0, EUL1, ZI0, ZI1, OI0, OI1, WS0, WS1, THRU0, THRU1,
           LVRAW, EV, ZJ, ZJ3, OUTJ, D64, THRV, EVZ, SRAW, NBUF };     // EVZ, SRAW: sparse calls only
    Buf buf[NBUF];
    unsigned long long allocs = 0, calls = 0, tensor_slabs = 0, simt_slabs = 0;
    int64_t slab_rows = 0;     // 0: ~256 MB of X per slab
    std::mutex mu;

    int init() {
        for (int i = 0; i < 2; ++i) {
            const cudaError_t e = cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking);
            if (e != cudaSuccess) return set_error(ORI_ECUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        }
        for (int i = 0; i < 3; ++i) {
            const cudaError_t e = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming);
            if (e != cudaSuccess) return set_error(ORI_ECUDA, "cudaEventCreate: %s", cudaGetErrorString(e));
        }
        return ORI_OK;
    }
    // rows of `width` bytes, contiguous on the host, to a pitched device buffer on stream s.  Pinned (or registered) host
    // memory is copied directly; pageable memory goes through the staging ring.
    int h2d_rows(void* dst, size_t dpitch, const void* src, size_t width, int64_t rows, cudaStream_t s) {
        if (rows <= 0 || width == 0) return ORI_OK;
        cudaPointerAttributes at;
        const bool pinned = cudaPointerGetAttributes(&at, src) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (pinned || (size_t)rows * width < (4u << 20)) {
            const cudaError_t e = cudaMemcpy2DAsync(dst, dpitch, src, width, width, rows, cudaMemcpyHostToDevice, s);
            return e == cudaSuccess ? ORI_OK : set_error(ORI_ECUDA, "cudaMemcpy2DAsync: %s", cudaGetErrorString(e));
        }
        if (!stg[NSTG - 1] || !stg_ev[NSTG - 1]) {
            for (int i = 0; i < NSTG; ++i) {
                cudaError_t e = stg[i] ? cudaSuccess : cudaHostAlloc(&stg[i], STG_BYTES, cudaHostAllocDefault);
                if (e == cudaSuccess && !stg_ev[i]) e = cudaEventCreateWithFlags(&stg_ev[i], cudaEventDisableTiming);
                if (e != cudaSuccess) return set_error(ORI_ECUDA, "pinned staging: %s", cudaGetErrorString(e));   // retried by the next call
            }
            if (pool.th.empty()) {
                unsigned hc = std::thread::hardware_concurrency();
                pool.start((int)(hc >= 16 ? 8 : (hc >= 4 ? hc / 2 : 1)));
            }
            ++allocs;
        }
        int64_t per = (int64_t)(STG_BYTES / width);
        if (per < 1) {     // a single row longer than a staging chunk: let the driver stage it
            const cudaError_t e = cudaMemcpy2DAsync(dst, dpitch, src, width, width, rows, cudaMemcpyHostToDevice, s);
            return e == cudaSuccess ? ORI_OK : set_error(ORI_ECUDA, "cudaMemcpy2DAsync: %s", cudaGetErrorString(e));
        }
        for (int64_t r = 0; r < rows; r += per) {
            const int64_t nr = rows - r < per ? rows - r : per;
            const int i = stg_next; stg_next = (stg_next + 1) % NSTG;
            if (stg_busy[i]) { cudaEventSynchronize(stg_ev[i]); stg_busy[i] = false; }
            pool.copy(stg[i], (const char*)src + (size_t)r * width, (size_t)nr * width);
            cudaError_t e = cudaMemcpy2DAsync((char*)dst + (size_t)r * dpitch, dpitch, stg[i], width, width, nr, cudaMemcpyHostToDevice, s);
            if (e == cudaSuccess) e = cudaEventRecord(stg_ev[i], s);
            if (e != cudaSuccess) return set_error(ORI_ECUDA, "staged copy: %s", cudaGetErrorString(e));
            stg_busy[i] = true;
            staged_bytes += (size_t)nr * width;
        }
        return ORI_OK;
    }
    void release() {
        pool.shutdown();
        for (int i = 0; i < NSTG; ++i) {
            if (stg_ev[i]) { cudaEventDestroy(stg_ev[i]); stg_ev[i] = nullptr; }
            if (stg[i]) { cudaFreeHost(stg[i]); stg[i] = nullptr; }
            stg_busy[i] = false;
        }
        for (auto& b : buf) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }
        for (auto& e : ev) { if (e) cudaEventDestroy(e); e = nullptr; }
        for (auto& s : st) { if (s) cudaStreamDestroy(s); s = nullptr; }
    }
    // grow-only: a buffer is reallocated only when a call needs more than any call before it
    int need(int id, size_t bytes) {
        Buf& b = buf[id];
        if (bytes <= b.cap && b.p) return ORI_OK;
        if (b.p) { cudaStreamSynchronize(st[0]); cudaStreamSynchronize(st[1]); cudaFree(b.p); b.p = nullptr; b.cap = 0; }
        const size_t cap = bytes < 256 ? 256 : bytes;
        const cudaError_t e = cudaMalloc(&b.p, cap);
        if (e != cudaSuccess) return set_error(ORI_ECUDA, "cudaMalloc(%zu): %s", cap, cudaGetErrorString(e));
        b.cap = cap; ++allocs;
        return ORI_OK;
    }
    template <class T> T* as(int id) { return (T*)buf[id].p; }
};

static int z_operator_args(const float* Zi_out, const float* Zj_out, const float* logU, const float* logV, const float* D,
                           const float* X, int64_t n, int64_t p, int64_t K, int quirk)
{
    if (n < 0 || p <= 0 || K <= 0) return set_error(ORI_EINVAL, "bad shape n=%lld p=%lld K=%lld", (long long)n, (long long)p, (long long)K);
    if (p > 0x7fffffff) return set_error(ORI_EINVAL, "p too large");
    if (!Zi_out || !Zj_out || !logU || !logV || !X) return set_error(ORI_EINVAL, "null array (the reference raises TypeError, zigap.py:79)");
    if (pad_k(K) < 0) return set_error(ORI_EUNSUPPORTED, "K=%lld > 64 is not supported", (long long)K);
    if (quirk && D && p < K) return set_error(ORI_EINVAL, "quirk mode needs p >= K");
    return ORI_OK;
}

// St, Sh non-NULL: the sparse model's operator (sparse_zigap.py:100-116), with D and Z3_out required.  Its denominator
// operand carries the mask S_tilde, the row sums contract with eVd * S_hat, and the kernel family follows the sparse
// model's plan (tensor path for K <= 32 only, in the fp32-grade mode).  The arguments are checked by the entry points.
static int z_operator_ctx(ori_ctx* C, float* Zi_out, float* Zj_out, float* Z3_out, const float* logU, const float* logV,
                          const float* St, const float* Sh, const float* D, const float* X, int64_t n, int64_t p, int64_t K,
                          int quirk)
{
    if (!C) return set_error(ORI_EINVAL, "null context");
    const bool sparse = St != nullptr;
    if (n == 0) { memset(Zj_out, 0, sizeof(float) * p * K); if (Z3_out) memset(Z3_out, 0, sizeof(float) * p * K); return ORI_OK; }
    std::lock_guard<std::mutex> lock(C->mu);
    ++C->calls;
    cudaStream_t st = C->st[0], st2 = C->st[1];

    const int64_t ldx = (p + 3) & ~3ll;
    // slab of cells sized to ~256 MB of X (or the context's setting), a multiple of 128
    int64_t slab = C->slab_rows > 0 ? C->slab_rows : (256ll << 20) / (ldx * 4);
    slab = slab < 128 ? 128 : (slab / 128) * 128;
    if (slab > n) slab = n;
    const int nbuf = n > slab ? 2 : 1;
    // kernel family: slabs that fill the machine take the tcgen05 / TMA passes (GaP-shaped: D_hat is an explicit input
    // here, folded into X), smaller ones the CUDA-core kernels -- the same rule as the device models.  The sparse model:
    // K <= 32 only, with fp32-grade contractions (its S-step is a sigmoid of the difference of two large gene sums,
    // sparse_zigap.py:155-157, which amplifies their absolute error exponentially: no TF32 operands)
    const bool tensor = slab * p >= (1ll << 21) && !(sparse && K > 32);
    const int KP = tensor ? (K <= 32 ? 32 : 64) : pad_k(K);
    const size_t ws_floats = tensor ? (size_t)tc_workspace_floats(slab, (int)p, KP) + 32 : 0;
    // the third output takes the third gene sum, weighted by D_hat[i, j] (zigap.py:95, sparse_zigap.py:116).  Under the
    // quirk Zj is weighted by D_hat[i, k] instead (zigap.py:94): the third sum then takes a sweep over X*D_hat of its own,
    // into ZJ3 = [plain gene sums | (unused) | Zl]; otherwise it comes out of the Zj sweep, into ZJ's third block
    const bool qw = D && quirk;
    const bool sweep3 = Z3_out && qw;
    const size_t zj_bytes = sizeof(float) * ORI_RED32_FLOATS(p, KP, Z3_out && !sweep3);
    const size_t zj3_bytes = sizeof(float) * ORI_RED32_FLOATS(p, KP, 1);

    typedef ori_ctx B;
    for (int b = 0; b < nbuf; ++b) {
        ORI_TRY(C->need(B::X0 + b, sizeof(float) * slab * ldx));
        if (D) ORI_TRY(C->need(B::D0 + b, sizeof(float) * slab * ldx));
        ORI_TRY(C->need(B::LUS0 + b, sizeof(float) * slab * K));
        ORI_TRY(C->need(B::EU0 + b, sizeof(float) * slab * KP));
        if (qw) ORI_TRY(C->need(B::EUW0 + b, sizeof(float) * slab * KP));
        if (Z3_out) ORI_TRY(C->need(B::EUL0 + b, sizeof(float) * slab * KP));
        ORI_TRY(C->need(B::ZI0 + b, sizeof(float) * slab * KP));
        ORI_TRY(C->need(B::OI0 + b, sizeof(float) * slab * K));
        ORI_TRY(C->need(B::THRU0 + b, sizeof(float) * slab));
        if (tensor) ORI_TRY(C->need(B::WS0 + b, sizeof(float) * ws_floats));
    }
    ORI_TRY(C->need(B::LVRAW, sizeof(float) * p * K));
    ORI_TRY(C->need(B::EV, sizeof(float) * p * KP));
    ORI_TRY(C->need(B::ZJ, zj_bytes));
    if (sweep3) ORI_TRY(C->need(B::ZJ3, zj3_bytes));
    if (sparse) {
        ORI_TRY(C->need(B::EVZ, sizeof(float) * p * KP));
        ORI_TRY(C->need(B::SRAW, sizeof(float) * 2 * p * K));
    }
    ORI_TRY(C->need(B::OUTJ, sizeof(float) * p * K));
    ORI_TRY(C->need(B::D64, sizeof(double) * ORI_RED64_DOUBLES(p, KP)));
    ORI_TRY(C->need(B::THRV, sizeof(float) * p));

    float* dlogVraw = C->as<float>(B::LVRAW);
    float* deV = C->as<float>(B::EV);
    float* dZj = C->as<float>(B::ZJ);
    float* dZ3 = sweep3 ? C->as<float>(B::ZJ3) : dZj;     // the buffer of the third sum
    float* dOutJ = C->as<float>(B::OUTJ);

    ORI_CUDA(cudaMemcpyAsync(dlogVraw, logV, sizeof(float) * p * K, cudaMemcpyHostToDevice, st));
    // the operator IS the reference's numba loop: its float32 exp underflow (den = 0 -> 1, zigap.py:86-90) is part of
    // the contract here, so the thresholds are always on
    float* deVz = sparse ? C->as<float>(B::EVZ) : nullptr;
    if (sparse) {    // deV = eVd (denominator, masked by S_tilde), deVz = eVd * S_hat (row sums)
        float* dS = C->as<float>(B::SRAW);
        ORI_CUDA(cudaMemcpyAsync(dS, St, sizeof(float) * p * K, cudaMemcpyHostToDevice, st));
        ORI_CUDA(cudaMemcpyAsync(dS + p * K, Sh, sizeof(float) * p * K, cudaMemcpyHostToDevice, st));
        k_exp_pad_sparse<<<cdiv(p * KP, 256), 256, 0, st>>>(dlogVraw, dS, dS + p * K, deV, deVz, C->as<float>(B::THRV),
                                                            p, (int)K, KP);
    } else {
        k_exp_pad<<<cdiv(p * KP, 256), 256, 0, st>>>(dlogVraw, nullptr, 0, 0, deV, p, (int)K, KP, C->as<float>(B::THRV));
    }
    ORI_TRY(check_launch("k_exp_pad"));
    ORI_CUDA(cudaMemsetAsync(dZj, 0, zj_bytes, st));
    if (sweep3) ORI_CUDA(cudaMemsetAsync(dZ3, 0, zj3_bytes, st));
    // [0],[1]: last work on each stream; [2]: gene-side operands ready
    ORI_CUDA(cudaEventRecord(C->ev[2], st));
    ORI_CUDA(cudaStreamWaitEvent(st2, C->ev[2], 0));

    ori_problem_t P;
    memset(&P, 0, sizeof(P));
    P.p = (int)p; P.K = (int)K; P.KP = KP; P.ldx = ldx;
    P.eV = deV; P.V_hat = deV;
    P.eVd = deV; P.eVz = deVz;
    P.thrV = C->as<float>(B::THRV);
    P.red64 = C->as<double>(B::D64);
    // the sparse problem has no dropout layer (D_hat is folded into X): ori_problem_check refuses it from outside callers
    const uint32_t flags = sparse ? ORI_F_SPARSE | (tensor ? ORI_F_PRECISE : 0u) : 0u;

    int b = 0;
    for (int64_t r0 = 0; r0 < n; r0 += slab, b ^= (nbuf - 1)) {
        const int64_t nr = (n - r0 < slab) ? n - r0 : slab;
        cudaStream_t s = b ? st2 : st;
        float* x = C->as<float>(B::X0 + b);
        float* dD = D ? C->as<float>(B::D0 + b) : nullptr;
        float* dlUs = C->as<float>(B::LUS0 + b);
        float* deU = C->as<float>(B::EU0 + b); float* deUw = C->as<float>(B::EUW0 + b); float* deUl = C->as<float>(B::EUL0 + b);
        float* dZi = C->as<float>(B::ZI0 + b); float* dOutI = C->as<float>(B::OI0 + b);
        ORI_TRY(C->h2d_rows(x, sizeof(float) * ldx, X + r0 * p, sizeof(float) * p, nr, s));
        if (D) ORI_TRY(C->h2d_rows(dD, sizeof(float) * ldx, D + r0 * p, sizeof(float) * p, nr, s));
        ORI_CUDA(cudaMemcpyAsync(dlUs, logU + r0 * K, sizeof(float) * nr * K, cudaMemcpyHostToDevice, s));
        k_exp_pad<<<cdiv(nr * KP, 256), 256, 0, s>>>(dlUs, nullptr, 0, 0, deU, nr, (int)K, KP, C->as<float>(B::THRU0 + b));
        if (qw)   // zigap.py:94: weight of cell i for latent k is D_hat[i, k]
            k_exp_pad<<<cdiv(nr * KP, 256), 256, 0, s>>>(dlUs, dD, ldx, 0, deUw, nr, (int)K, KP);
        if (Z3_out)
            k_exp_pad<<<cdiv(nr * KP, 256), 256, 0, s>>>(dlUs, nullptr, 0, 1, deUl, nr, (int)K, KP);
        const float* xq = x;  // X for the quirk gene sums (unweighted)
        if (D) {              // X*D in place of X for everything weighted by D_hat[i, j]
            if (quirk) {      // keep X: write X*D into the D buffer
                k_mul<<<cdiv(nr * ldx, 256), 256, 0, s>>>(x, dD, dD, nr * ldx);
                x = dD;
            } else {
                k_mul<<<cdiv(nr * ldx, 256), 256, 0, s>>>(x, dD, x, nr * ldx);
                xq = x;
            }
        }
        ORI_TRY(check_launch("operator prologue"));
        ORI_CUDA(cudaMemsetAsync(dZi, 0, sizeof(float) * nr * KP, s));
        P.n_rows = nr; P.n_total = n; P.flags = flags;
        P.eU[0] = deU; P.U_hat[0] = deU; P.U_hat[1] = deU;
        P.Zi = dZi;
        P.thrU = C->as<float>(B::THRU0 + b);
        P.tc_ws = tensor ? C->as<float>(B::WS0 + b) : nullptr;
        P.tc_ws_floats = tensor ? (int64_t)ws_floats : 0;
        // row sums (zigap.py:93)
        P.X = x;
        (tc_eligible(&P) ? C->tensor_slabs : C->simt_slabs) += 1;
        ORI_TRY(pass_rows_any(&P, 0, s));
        k_scale_unpad<<<cdiv(nr * K, 256), 256, 0, s>>>(dZi, deU, nullptr, nullptr, dOutI, nr, (int)K, KP);
        ORI_CUDA(cudaMemcpyAsync(Zi_out + r0 * K, dOutI, sizeof(float) * nr * K, cudaMemcpyDeviceToHost, s));
        // gene sums (zigap.py:94): both streams add into the same accumulators with atomics
        P.red32 = dZj;
        P.eUl[0] = Z3_out && !sweep3 ? deUl : nullptr;
        if (qw) { P.X = xq; P.flags = ORI_F_QUIRK; P.eUw = deUw; }
        ORI_TRY(gene_sums(&P, 0, s));
        if (sweep3) {
            P.X = x; P.flags = flags; P.eUl[0] = deUl; P.red32 = dZ3;
            ORI_TRY(gene_sums(&P, 0, s));
        }
        ORI_CUDA(cudaEventRecord(C->ev[b], s));
    }
    ORI_CUDA(cudaStreamWaitEvent(st, C->ev[0], 0));
    ORI_CUDA(cudaStreamWaitEvent(st, C->ev[1 % nbuf], 0));
    k_scale_unpad<<<cdiv(p * K, 256), 256, 0, st>>>(dZj, deV, nullptr, nullptr, dOutJ, p, (int)K, KP);
    ORI_CUDA(cudaMemcpyAsync(Zj_out, dOutJ, sizeof(float) * p * K, cudaMemcpyDeviceToHost, st));
    if (Z3_out) {   // eV * Zl + logV * (eV * plain gene sums)
        P.red32 = dZ3;
        const RedBufs z3 = red_carve(P);
        k_scale_unpad<<<cdiv(p * K, 256), 256, 0, st>>>(z3.Zl, deV, z3.Zj, dlogVraw, dOutJ, p, (int)K, KP);
        ORI_CUDA(cudaMemcpyAsync(Z3_out, dOutJ, sizeof(float) * p * K, cudaMemcpyDeviceToHost, st));
    }
    ORI_TRY(check_launch("operator epilogue"));
    ORI_CUDA(cudaStreamSynchronize(st2));
    ORI_CUDA(cudaStreamSynchronize(st));
    return ORI_OK;
}

static ori_ctx* default_ctx(int* rc) {
    static std::mutex mu;
    static ori_ctx* ctx = nullptr;
    std::lock_guard<std::mutex> lock(mu);
    *rc = ORI_OK;
    if (!ctx) {
        ctx = new ori_ctx();
        *rc = ctx->init();
        if (*rc != ORI_OK) { ctx->release(); delete ctx; ctx = nullptr; }
    }
    return ctx;
}

extern "C" {

int ori_ctx_create(ori_ctx_t** out, int64_t slab_rows) {
    if (!out || slab_rows < 0) return set_error(ORI_EINVAL, "ori_ctx_create: bad argument");
    ori_ctx* c = new ori_ctx();
    const int rc = c->init();
    if (rc != ORI_OK) { c->release(); delete c; *out = nullptr; return rc; }
    c->slab_rows = slab_rows;
    *out = c;
    return ORI_OK;
}

int ori_ctx_destroy(ori_ctx_t* ctx) {
    if (!ctx) return ORI_OK;
    ctx->release();
    delete ctx;
    return ORI_OK;
}

int ori_ctx_stats(ori_ctx_t* ctx, unsigned long long* calls, unsigned long long* device_allocations,
                  unsigned long long* tensor_slabs, unsigned long long* simt_slabs) {
    int rc = ORI_OK;
    ori_ctx* c = ctx ? ctx : default_ctx(&rc);
    if (!c) return rc;
    std::lock_guard<std::mutex> lock(c->mu);
    if (calls) *calls = c->calls;
    if (device_allocations) *device_allocations = c->allocs;
    if (tensor_slabs) *tensor_slabs = c->tensor_slabs;
    if (simt_slabs) *simt_slabs = c->simt_slabs;
    return ORI_OK;
}

// The operator entry points check their arguments before any device work, so a bad *_host call creates no default
// context; the *_host forms are the *_ctx ones on the process-wide default context.
static int zigap_args(const float* DZ_hat_i, const float* DZ_hat_j, const float* log_U_hat, const float* log_V_hat,
                      const float* D_hat, const float* X, int64_t n, int64_t p, int64_t K, int quirk) {
    if (!D_hat) return set_error(ORI_EINVAL, "D_hat is NULL");
    return z_operator_args(DZ_hat_i, DZ_hat_j, log_U_hat, log_V_hat, D_hat, X, n, p, K, quirk);
}

int ori_zigap_compute_Z_q_expectations_ctx(ori_ctx_t* ctx, float* DZ_hat_i, float* DZ_hat_j, float* DZ_exp_logsum_hat,
                                           const float* log_U_hat, const float* log_V_hat,
                                           const float* D_hat, const float* X,
                                           int64_t n, int64_t p, int64_t K, int quirk) {
    ORI_TRY(zigap_args(DZ_hat_i, DZ_hat_j, log_U_hat, log_V_hat, D_hat, X, n, p, K, quirk));
    return z_operator_ctx(ctx, DZ_hat_i, DZ_hat_j, DZ_exp_logsum_hat, log_U_hat, log_V_hat, nullptr, nullptr, D_hat, X, n, p, K, quirk);
}

int ori_gap_compute_Z_q_expectations_ctx(ori_ctx_t* ctx, float* Z_hat_i, float* Z_hat_j, const float* log_U_hat,
                                         const float* log_V_hat, const float* X, int64_t n, int64_t p, int64_t K) {
    ORI_TRY(z_operator_args(Z_hat_i, Z_hat_j, log_U_hat, log_V_hat, nullptr, X, n, p, K, 0));
    return z_operator_ctx(ctx, Z_hat_i, Z_hat_j, nullptr, log_U_hat, log_V_hat, nullptr, nullptr, nullptr, X, n, p, K, 0);
}

int ori_zigap_compute_Z_q_expectations_host(float* DZ_hat_i, float* DZ_hat_j, float* DZ_exp_logsum_hat,
                                            const float* log_U_hat, const float* log_V_hat,
                                            const float* D_hat, const float* X,
                                            int64_t n, int64_t p, int64_t K, int quirk) {
    ORI_TRY(zigap_args(DZ_hat_i, DZ_hat_j, log_U_hat, log_V_hat, D_hat, X, n, p, K, quirk));
    int rc;
    ori_ctx* c = default_ctx(&rc);
    return c ? ori_zigap_compute_Z_q_expectations_ctx(c, DZ_hat_i, DZ_hat_j, DZ_exp_logsum_hat, log_U_hat, log_V_hat, D_hat,
                                                      X, n, p, K, quirk) : rc;
}

int ori_gap_compute_Z_q_expectations_host(float* Z_hat_i, float* Z_hat_j, const float* log_U_hat,
                                          const float* log_V_hat, const float* X, int64_t n, int64_t p, int64_t K) {
    ORI_TRY(z_operator_args(Z_hat_i, Z_hat_j, log_U_hat, log_V_hat, nullptr, X, n, p, K, 0));
    int rc;
    ori_ctx* c = default_ctx(&rc);
    return c ? ori_gap_compute_Z_q_expectations_ctx(c, Z_hat_i, Z_hat_j, log_U_hat, log_V_hat, X, n, p, K) : rc;
}

// sparse_zigap.py:100-116: D_hat, S_tilde, S_hat and the third output (read by the S-step, :155) are required
static int sparse_args(const float* DSZ_hat, const float* DZ_hat, const float* DZ_exp_logsum_hat, const float* log_U_hat,
                       const float* log_V_hat, const float* S_tilde, const float* S_hat, const float* D_hat, const float* X,
                       int64_t n, int64_t p, int64_t K) {
    if (!D_hat) return set_error(ORI_EINVAL, "D_hat is NULL");
    if (!DZ_exp_logsum_hat) return set_error(ORI_EINVAL, "DZ_exp_logsum_hat is NULL (sparse_zigap.py:155 reads it)");
    if (!S_tilde || !S_hat) return set_error(ORI_EINVAL, "S_tilde / S_hat is NULL");
    return z_operator_args(DSZ_hat, DZ_hat, log_U_hat, log_V_hat, D_hat, X, n, p, K, 0);
}

int ori_sparse_zigap_compute_Z_q_expectations_ctx(ori_ctx_t* ctx, float* DSZ_hat, float* DZ_hat, float* DZ_exp_logsum_hat,
                                                  const float* log_U_hat, const float* log_V_hat, const float* S_tilde,
                                                  const float* S_hat, const float* D_hat, const float* X,
                                                  int64_t n, int64_t p, int64_t K) {
    ORI_TRY(sparse_args(DSZ_hat, DZ_hat, DZ_exp_logsum_hat, log_U_hat, log_V_hat, S_tilde, S_hat, D_hat, X, n, p, K));
    return z_operator_ctx(ctx, DSZ_hat, DZ_hat, DZ_exp_logsum_hat, log_U_hat, log_V_hat, S_tilde, S_hat, D_hat, X, n, p, K, 0);
}

int ori_sparse_zigap_compute_Z_q_expectations_host(float* DSZ_hat, float* DZ_hat, float* DZ_exp_logsum_hat,
                                                   const float* log_U_hat, const float* log_V_hat, const float* S_tilde,
                                                   const float* S_hat, const float* D_hat, const float* X,
                                                   int64_t n, int64_t p, int64_t K) {
    ORI_TRY(sparse_args(DSZ_hat, DZ_hat, DZ_exp_logsum_hat, log_U_hat, log_V_hat, S_tilde, S_hat, D_hat, X, n, p, K));
    int rc;
    ori_ctx* c = default_ctx(&rc);
    return c ? ori_sparse_zigap_compute_Z_q_expectations_ctx(c, DSZ_hat, DZ_hat, DZ_exp_logsum_hat, log_U_hat, log_V_hat,
                                                             S_tilde, S_hat, D_hat, X, n, p, K) : rc;
}

}  // extern "C"
