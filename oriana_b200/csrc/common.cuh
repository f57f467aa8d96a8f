// common.cuh -- shared declarations of the oriana_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "../../include/oriana_b200.h"

namespace ori {

// error plumbing (api.cu)
int set_error(int code, const char* fmt, ...);
int check_launch(const char* what, int n_kernels = 1);   // also counts the kernels launched (ori_kernel_launches)

// The regions of the reduction buffers red32, red64 and gsum (layout: include/oriana_b200.h).  Zl exists only with eUl.
struct RedBufs {
    float *Zj, *b2s, *Zl;                   // red32
    double *colsum, *SlogU, *SU, *part;     // red64; part: the ORI_R64_* slots
    double *SlogV, *SV, *gpart;             // gsum; gpart: the ORI_GSUM_* slots
};
__host__ __device__ inline RedBufs red_carve(const ori_problem_t& P) {
    RedBufs r;
    r.Zj = P.red32;
    r.b2s = P.red32 + (long long)P.p * P.KP;
    r.Zl = P.red32 + 2ll * P.p * P.KP;
    r.colsum = P.red64;
    r.SlogU = P.red64 + P.p;
    r.SU = P.red64 + P.p + P.KP;
    r.part = P.red64 + P.p + 2 * P.KP;
    r.SlogV = P.gsum;
    r.SV = P.gsum + P.KP;
    r.gpart = P.gsum + 2 * P.KP;
    return r;
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// Counts stored as uint16 (ORI_F_X_U16) are widened to float32 as they are read, exactly (u < 2^23): the bits
// 0x4B000000 | u are the float 2^23 + u, and one FADD takes 2^23 off.  Integer / FMA pipes only -- no I2F, which would
// add to the XU / MIO path that bounds the tensor passes (DESIGN.md 4.1).  float32 counts pass through unchanged.
__device__ __forceinline__ float u16_to_f32(uint32_t u) { return __uint_as_float(0x4B000000u | u) - 8388608.f; }
__device__ __forceinline__ float count_f32(float x) { return x; }
__device__ __forceinline__ float count_f32(uint16_t x) { return u16_to_f32(x); }
// the count at p through the read-only cache
template <class XT> __device__ __forceinline__ float ldg_count(const XT* p) { return count_f32(__ldg(p)); }
// f(X) with the problem's X pointer in its storage type (const float* or const uint16_t*)
template <class F> static inline int with_counts(const ori_problem_t* P, F&& f) {
    return (P->flags & ORI_F_X_U16) ? f(reinterpret_cast<const uint16_t*>(P->X)) : f(P->X);
}
template <class Ptr> using count_t = std::remove_const_t<std::remove_pointer_t<Ptr>>;

// kernels_simt.cu
int launch_pass_rows_simt(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_pass_genes_simt(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_row_update(const ori_problem_t* P, int gen_old, int write_state, cudaStream_t st);
int launch_gene_update(const ori_problem_t* P, int write_state, cudaStream_t st);
int launch_mstep(const ori_problem_t* P, int mode, cudaStream_t st);
int launch_count_stats(const ori_problem_t* P, cudaStream_t st);
int launch_quirk_weights(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_dropout_posterior(const ori_problem_t* P, int gen, float* out, long long ldo,
                             long long row0, long long nrows, cudaStream_t st);
template <class XT> int launch_row_sums(const XT* X, long long ldx, long long n_rows, int p, float* out, cudaStream_t st);
template <class XT> int launch_col_sums(const XT* X, long long ldx, long long n_rows, int p, double* out, cudaStream_t st);
int launch_deviance(const ori_problem_t* P, int gen, const double* pi, const double* col_mean, long long* out_int,
                    double* out_f64, cudaStream_t st);

// kernels_tc.cu
long long tc_workspace_floats(long long n_rows, int p, int KP);

// ORI_F_DETERMINISTIC scratch (ori_problem_t::det_ws): the regions det_carve places
constexpr int DET_FU_BLOCKS = 148 * 8;             // the most blocks of k_factor_update / k_sparse_gene_update
constexpr int DET_FU_SLOTS = 2 * 64 + 2;
constexpr int DET_ITEM_SLOTS = 2 * 8 * 2;          // CTAs of a pair x element-wise warps x (x log den, entropy)
// CUDA-core kernels (problems up to DET_SIMT_MAX entries): row blocks of k_pass_rows, row chunks of k_pass_genes
constexpr long long DET_SIMT_MAX = 1ll << 26;
constexpr int DET_SIMT_BLOCK_ROWS = 128;
constexpr int DET_SIMT_CHUNK_ROWS = 8192;
struct DetWs {
    double* fu_part;      // [DET_FU_BLOCKS x DET_FU_SLOTS] per-block sums of the factor updates (sum log E | sum E | entropy | D.uv)
    double* colsum2;      // [p, padded to 128] column sums of D_hat of the second column slice of the tensor gene pass
    double* item_part;    // [items x DET_ITEM_SLOTS] per-item, per-CTA, per-warp ELBO terms of the tensor gene pass
    int* tickets;         // one per own tile of the running tensor pass (chunk order of the accumulator adds)
    double* simt_colsum;  // [row blocks x p] column sums of D_hat per row block     } CUDA-core kernels,
    double* simt_elbo;    // [row blocks x 2] ELBO terms per row block               } NULL above
    float* simt_gene;     // [row chunks x red32] gene sums per row chunk             } DET_SIMT_MAX entries
    long long doubles;    // size of the whole scratch: ori_det_workspace_doubles
};
// ws == NULL: every pointer NULL, the size all the same
DetWs det_carve(double* ws, long long n_rows, int p);
inline bool det_simt_ok(long long n_rows, int p) { return n_rows * (long long)p <= DET_SIMT_MAX; }
// src[n][2] added in index order by one block: *dst0 += sum src[.][0], *dst1 += sum src[.][1]
int launch_det_sum_pairs(const double* src, long long n, double* dst0, double* dst1, cudaStream_t st);
bool tc_eligible(const ori_problem_t* P);
int launch_tc_prep_genes(const ori_problem_t* P, cudaStream_t st);
int launch_tc_prep_rows(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_pass_rows_tc(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_pass_genes_tc(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_tc_prep_rows_logsum(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_pass_genes_logsum_tc(const ori_problem_t* P, int gen_old, cudaStream_t st);
int launch_deviance_tc(const ori_problem_t* P, int gen, const double* pi, const double* col_mean, long long* out_int, cudaStream_t st);

}  // namespace ori
