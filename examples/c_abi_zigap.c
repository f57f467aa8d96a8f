/* c_abi_zigap.c -- the drop-in boundary used from plain C: no Python, no torch.
 *
 * Builds a ZIGaP problem (zigap.py:15-165) on device memory it allocates itself, fills X with the library's
 * synthetic-count generator, runs the construction sequence of base.py:43-52 and a few `step()`s (base.py:54-56)
 * through the entry points of include/oriana_b200.h, and prints the ELBO trace.
 *
 *   gcc -std=c99 -Iinclude -I/usr/local/cuda/include examples/c_abi_zigap.c \
 *       -Loriana_b200/lib -loriana_b200 -L/usr/local/cuda/lib64 -lcudart -lm -o c_abi_zigap
 *   LD_LIBRARY_PATH=oriana_b200/lib ./c_abi_zigap [n p K steps]
 */
#include <cuda_runtime_api.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "oriana_b200.h"

#define CHECK_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    fprintf(stderr, "%s: %s\n", #call, cudaGetErrorString(e_)); return 2; } } while (0)
#define CHECK_ORI(call) do { int rc_ = (call); if (rc_ != ORI_OK) { char msg_[512]; ori_last_error(msg_, sizeof msg_); \
    fprintf(stderr, "%s -> %d: %s\n", #call, rc_, msg_); return 3; } } while (0)

static void* dalloc(size_t bytes) {
    void* p = NULL;
    if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) { fprintf(stderr, "cudaMalloc(%zu) failed\n", bytes); exit(2); }
    cudaMemset(p, 0, bytes ? bytes : 16);
    return p;
}

/* a1 / b1 ~ Gamma(1) (zigap.py:61,71), drawn on the host with a fixed LCG: Exp(1) = -log(u) */
static void fill_exp1(float* dst, long long rows, int K, int KP, unsigned long long* state) {
    for (long long i = 0; i < rows; ++i)
        for (int k = 0; k < KP; ++k) {
            *state = *state * 6364136223846793005ULL + 1442695040888963407ULL;
            const double u = ((double)((*state >> 11) + 1)) / 9007199254740993.0;
            dst[i * KP + k] = k < K ? (float)fmax(-log(u), 1e-15) : 0.f;
        }
}

int main(int argc, char** argv) {
    const long long n = argc > 1 ? atoll(argv[1]) : 4096;
    const int p = argc > 2 ? atoi(argv[2]) : 1024, K = argc > 3 ? atoi(argv[3]) : 10, steps = argc > 4 ? atoi(argv[4]) : 5;
    const int KP = K <= 32 ? 32 : 64;                       /* the tensor path wants 32 or 64 */
    const long long ldx = (p + 3) / 4 * 4;
    if (K < 1 || K > 64 || steps < 1 || steps > 60) { fprintf(stderr, "need 1 <= K <= 64, 1 <= steps <= 60\n"); return 1; }
    CHECK_ORI(ori_device_check(0));

    ori_problem_t P;
    memset(&P, 0, sizeof P);
    P.n_rows = P.n_total = n; P.ldx = ldx; P.p = p; P.K = K; P.KP = KP;
    P.flags = ORI_F_DROPOUT | ORI_F_ELBO;
    P.trace_cap = 64;
    const size_t rowf = sizeof(float) * (size_t)n * KP, genef = sizeof(float) * (size_t)p * KP;
    float* X = (float*)dalloc(sizeof(float) * (size_t)n * ldx);
    P.X = X;
    P.a1 = (float*)dalloc(rowf); P.a2 = (float*)dalloc(rowf);
    for (int g = 0; g < 2; ++g) { P.U_hat[g] = (float*)dalloc(rowf); P.eU[g] = (float*)dalloc(rowf); }
    P.Zi = (float*)dalloc(rowf); P.a2s = (float*)dalloc(rowf);
    P.b1 = (float*)dalloc(genef); P.b2 = (float*)dalloc(genef); P.V_hat = (float*)dalloc(genef); P.eV = (float*)dalloc(genef);
    P.red32 = (float*)dalloc(sizeof(float) * (size_t)ORI_RED32_FLOATS(p, KP, 0));
    P.lp = (float*)dalloc(sizeof(float) * p); P.pfloor = (float*)dalloc(sizeof(float) * p);
    P.hyper = (double*)dalloc(sizeof(double) * 4 * K);
    P.red64 = (double*)dalloc(sizeof(double) * (size_t)ORI_RED64_DOUBLES(p, KP));
    P.gsum = (double*)dalloc(sizeof(double) * ORI_GSUM_DOUBLES(KP));
    P.pi_d = (double*)dalloc(sizeof(double) * p);
    P.scal = (double*)dalloc(sizeof(double) * ORI_SC_NSLOTS);
    P.elbo_trace = (double*)dalloc(sizeof(double) * P.trace_cap);
    P.tc_ws_floats = ori_tc_workspace_floats(n, p, KP) + 32;
    P.tc_ws = (float*)dalloc(sizeof(float) * (size_t)P.tc_ws_floats);

    /* synthetic zero-inflated counts, generated in HBM (SURVEY.md 8d) */
    float* Us = (float*)dalloc(sizeof(float) * (size_t)n * K);
    float* Vs = (float*)dalloc(sizeof(float) * (size_t)p * K);
    float* pis = (float*)dalloc(sizeof(float) * p);
    CHECK_ORI(ori_synth_counts_f32(X, ldx, 0, n, p, K, 7, 0.5f, 1, Us, Vs, pis, NULL));

    /* row / column sums of X: the ELBO's bookkeeping for the per-row scaling of exp(E log .) */
    float* xrow = (float*)dalloc(sizeof(float) * (size_t)n);
    double* xcol64 = (double*)dalloc(sizeof(double) * p);
    float* xcol = (float*)dalloc(sizeof(float) * p);
    CHECK_ORI(ori_row_sums_f32(X, ldx, n, p, xrow, NULL));
    CHECK_ORI(ori_column_sums_f64(X, ldx, n, p, xcol64, NULL));
    {
        double* h = (double*)malloc(sizeof(double) * p); float* hf = (float*)malloc(sizeof(float) * p);
        CHECK_CUDA(cudaMemcpy(h, xcol64, sizeof(double) * p, cudaMemcpyDeviceToHost));
        for (int j = 0; j < p; ++j) hf[j] = (float)h[j];
        CHECK_CUDA(cudaMemcpy(xcol, hf, sizeof(float) * p, cudaMemcpyHostToDevice));
        free(h); free(hf);
    }
    P.xrow = xrow; P.xcol = xcol;

    /* initial variational parameters (zigap.py:55-77): a1, b1 ~ Gamma(1), a2 = b2 = 1, p_d = (X > 0); priors Gamma(2), 1 */
    {
        unsigned long long st = 12345;
        float* h = (float*)malloc(rowf > genef ? rowf : genef);
        fill_exp1(h, n, K, KP, &st); CHECK_CUDA(cudaMemcpy(P.a1, h, rowf, cudaMemcpyHostToDevice));
        for (long long i = 0; i < n * KP; ++i) h[i] = (i % KP) < K ? 1.f : 0.f;
        CHECK_CUDA(cudaMemcpy(P.a2, h, rowf, cudaMemcpyHostToDevice));
        fill_exp1(h, p, K, KP, &st); CHECK_CUDA(cudaMemcpy(P.b1, h, genef, cudaMemcpyHostToDevice));
        for (long long i = 0; i < (long long)p * KP; ++i) h[i] = (i % KP) < K ? 1.f : 0.f;
        CHECK_CUDA(cudaMemcpy(P.b2, h, genef, cudaMemcpyHostToDevice));
        double* hy = (double*)malloc(sizeof(double) * 4 * K);
        for (int k = 0; k < K; ++k) { hy[k] = 2.0; hy[K + k] = 1.0; hy[2 * K + k] = 2.0; hy[3 * K + k] = 1.0; }
        CHECK_CUDA(cudaMemcpy(P.hyper, hy, sizeof(double) * 4 * K, cudaMemcpyHostToDevice));
        float* ninf = (float*)malloc(sizeof(float) * p);
        for (int j = 0; j < p; ++j) ninf[j] = -INFINITY;          /* D_hat(0) is the indicator (zigap.py:77) */
        CHECK_CUDA(cudaMemcpy(P.lp, ninf, sizeof(float) * p, cudaMemcpyHostToDevice));
        free(h); free(hy); free(ninf);
    }

    /* construction (base.py:43-52): expectations of the initial state, then one M-step */
    CHECK_ORI(ori_problem_check(&P));
    printf("tensor path: %s\n", ori_uses_tensor_path(&P) ? "yes" : "no");
    CHECK_ORI(ori_count_stats(&P, NULL));
    CHECK_ORI(ori_init_expectations(&P, 0, NULL));
    CHECK_ORI(ori_mstep(&P, ORI_M_INIT, NULL));

    /* step() x steps (base.py:54-56); the generation of the row factors ping-pongs */
    int gen = 0;
    for (int it = 0; it < steps; ++it) {
        P.iter = it;
        CHECK_ORI(ori_cavi_step(&P, gen, NULL));
        gen ^= 1;
    }
    /* flush of the one-pass lag: ELBO of the final state */
    P.iter = steps;
    CHECK_ORI(ori_finalize_local(&P, gen, NULL));
    CHECK_ORI(ori_mstep(&P, ORI_M_FINALIZE, NULL));
    CHECK_CUDA(cudaDeviceSynchronize());

    double trace[64];
    CHECK_CUDA(cudaMemcpy(trace, P.elbo_trace, sizeof(double) * (steps + 1), cudaMemcpyDeviceToHost));
    int monotone = 1;
    for (int it = 0; it <= steps; ++it) {
        printf("ELBO[%d] = %.9e\n", it, trace[it]);
        if (it > 0 && !(trace[it] >= trace[it - 1] - 1e-6 * fabs(trace[it - 1]))) monotone = 0;
    }
    printf("kernels launched: %llu, ELBO monotone: %s\n", ori_kernel_launches(), monotone ? "yes" : "no");
    return monotone ? 0 : 4;
}
