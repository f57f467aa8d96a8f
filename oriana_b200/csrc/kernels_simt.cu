// kernels_simt.cu -- CUDA-core (fp32 FMA) implementation of every kernel of the CAVI iteration.
//
// This is the reference-exact device path: it is what the tensor-core kernels (kernels_tc.cu) are
// validated against, and it serves the small / odd shapes they do not take.  Reference lines replaced:
//   k_pass_rows   zigap.py:79-95 (row sums DZ_hat_i), :116 (np.dot(D_hat, V_hat)), :131-136 (D_hat,
//                 recomputed on the fly instead of stored), :158 (column sums of p_d)
//   k_pass_genes  zigap.py:79-95 (gene sums DZ_hat_j, incl. the D_hat[i,k] quirk of :94), :124
//   k_factor_update  zigap.py:115-120 / :123-128, gamma.py:37-61
//   k_mstep       zigap.py:143-158, utils.py:39-51
#include "common.cuh"
#include "special.cuh"

namespace ori {

// ------------------------------------------------------------------------------------------------
// D_hat for an entry with X == 0 (zigap.py:131-134):  sigma(logit(pi_j) - uv), floor 1e-10 where pi_j<=0.
// lp = -inf encodes the initial indicator state p_d = (X>0) (zigap.py:77): the result is exactly 0.
// e (clamped to +-87) and ex = exp(e) are returned for the entropy term of the ELBO.
__device__ __forceinline__ float dropout_p(float uv, float lp, float fl, float& e, float& ex) {
    e = fminf(fmaxf(uv - lp, -87.f), 87.5f);
    ex = __expf(e);
    const float pz = (e > 87.f) ? 0.f : __fdividef(1.f, 1.f + ex);
    return fmaxf(pz, fl);
}

__device__ __forceinline__ double block_reduce_sum(double v, double* sbuf) {
    // all threads of the block call this; result valid in thread 0
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (l == 0) sbuf[w] = v;
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x == 0) for (int i = 0; i < nw; ++i) r += sbuf[i];
    return r;
}

// ------------------------------------------------------------------------------------------------
// Row pass.  CTA = 128 threads = 128 consecutive cells; thread r keeps its cell's eU, U_hat and the 2*KP
// accumulators in registers and sweeps gene tiles of 32; the X tile is staged (coalesced) through smem.
constexpr int PR_TR = 128;
constexpr int PR_TG = 32;
static_assert(PR_TR == DET_SIMT_BLOCK_ROWS, "det_carve sizes the per-row-block scratch by DET_SIMT_BLOCK_ROWS");

// SPARSE (sparse_zigap.py:100-116, :140-142, :166): the denominator operand eV carries the mask S_tilde, the row
// sums contract with eVz = eV * S_hat, D_hat is rebuilt from Vh = the PREVIOUS effective V_hat and the rate sums
// contract with Vc = the current one.  Otherwise eVz == eV and Vc == Vh (not read).  SPARSE without DROPOUT (the
// operator seam, D_hat folded into X): Vh and Vc are not read.
// TG: genes per tile (32; 16 for the sparse model at KP = 64, whose four gene-side operand tiles would not fit 48 KB)
// XT: element type of X (float, or uint16_t under ORI_F_X_U16)
template <int KP, bool DROPOUT, bool ELBO, bool SPARSE, int TG, class XT>
__global__ void __launch_bounds__(PR_TR)
k_pass_rows(const XT* __restrict__ X, long long ldx, long long n_rows, int p,
            const float* __restrict__ eU, const float* __restrict__ Uh,
            const float* __restrict__ eV, const float* __restrict__ Vh,
            const float* __restrict__ eVz, const float* __restrict__ Vc,
            const float* __restrict__ lp, const float* __restrict__ pfloor,
            float* __restrict__ Zi, float* __restrict__ a2s,
            double* __restrict__ colsum, double* __restrict__ part64,
            const float* __restrict__ thrU, const float* __restrict__ thrV,
            double* __restrict__ det_cs, double* __restrict__ det_part)
{
    // det_cs / det_part (ORI_F_DETERMINISTIC, launched with gridDim.y == 1): this CTA's column sums and ELBO terms go to
    // its own slots [blockIdx.x][p] / [blockIdx.x][2] instead of atomic targets; launch_det_sum_* add them in index order
    __shared__ float sX[PR_TR][TG + 1];
    __shared__ float sthr[TG];
    __shared__ __align__(16) float sV[TG][KP];
    __shared__ __align__(16) float sVh[DROPOUT ? TG : 1][KP];
    __shared__ __align__(16) float sVz[SPARSE ? TG : 1][KP];
    __shared__ __align__(16) float sVc[SPARSE && DROPOUT ? TG : 1][KP];
    __shared__ float slp[TG], sfl[TG];
    __shared__ float scs[PR_TR / 32][TG];
    __shared__ double sred[PR_TR / 32];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long row0 = (long long)blockIdx.x * PR_TR;
    const long long row = row0 + tid;
    const bool row_ok = row < n_rows;

    float eu[KP], uh[DROPOUT ? KP : 1], zi[KP], as[DROPOUT ? KP : 1];
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        eu[k] = row_ok ? eU[row * KP + k] : 0.f;
        zi[k] = 0.f;
        if (DROPOUT) { uh[k] = row_ok ? Uh[row * KP + k] : 0.f; as[k] = 0.f; }
    }
    double acc_xl = 0.0, acc_ent = 0.0;
    const float tu = (thrU && row_ok) ? thrU[row] : 0.f;         // underflow emulation (special.cuh); 0: never triggers

    const int ntiles = (p + TG - 1) / TG;
    for (int t = blockIdx.y; t < ntiles; t += gridDim.y) {
        const int j0 = t * TG;
        const int gcount = min(TG, p - j0);
        __syncthreads();  // previous tile fully consumed
        // X tile: warp w loads rows w, w+4, ...; a row segment is 32 consecutive floats
        for (int rr = warp; rr < PR_TR; rr += PR_TR / 32) {
            const long long r = row0 + rr;
            float v = 0.f;
            if (r < n_rows && lane < gcount) v = ldg_count(X + r * ldx + j0 + lane);
            if (lane < TG) sX[rr][lane] = v;
        }
        float* sVf = &sV[0][0];
        float* sVhf = &sVh[0][0];
        float* sVzf = &sVz[0][0];
        float* sVcf = &sVc[0][0];
        for (int idx = tid; idx < TG * KP; idx += PR_TR) {
            const int g = idx / KP;
            const bool ok = g < gcount;
            sVf[idx] = ok ? eV[(long long)j0 * KP + idx] : 0.f;
            if (DROPOUT) sVhf[idx] = ok ? Vh[(long long)j0 * KP + idx] : 0.f;
            if (SPARSE) {
                sVzf[idx] = ok ? eVz[(long long)j0 * KP + idx] : 0.f;
                if (DROPOUT) sVcf[idx] = ok ? Vc[(long long)j0 * KP + idx] : 0.f;
            }
        }
        if (DROPOUT && tid < TG) {
            slp[tid] = tid < gcount ? lp[j0 + tid] : 0.f;
            sfl[tid] = tid < gcount ? pfloor[j0 + tid] : 0.f;
        }
        if (tid < TG) sthr[tid] = (thrV && tid < gcount) ? thrV[j0 + tid] : 0.f;
        __syncthreads();

        float t_xl = 0.f, t_ent = 0.f;
        for (int g = 0; g < gcount; ++g) {
            const float x = sX[tid][g];
            float den = 0.f, uv = 0.f;
            const float4* v4 = reinterpret_cast<const float4*>(&sV[g][0]);
            const float4* h4 = reinterpret_cast<const float4*>(&sVh[DROPOUT ? g : 0][0]);
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                const float4 v = v4[q];
                den = fmaf(eu[4 * q + 0], v.x, den); den = fmaf(eu[4 * q + 1], v.y, den);
                den = fmaf(eu[4 * q + 2], v.z, den); den = fmaf(eu[4 * q + 3], v.w, den);
                if (DROPOUT) {
                    const float4 h = h4[q];
                    uv = fmaf(uh[4 * q + 0], h.x, uv); uv = fmaf(uh[4 * q + 1], h.y, uv);
                    uv = fmaf(uh[4 * q + 2], h.z, uv); uv = fmaf(uh[4 * q + 3], h.w, uv);
                }
            }
            const bool nz = x != 0.f;
            den = den > 0.f ? den : 1.f;                 // zigap.py:90
            float R = x / den;
            const float T = tu * sthr[g];
            if (nz && T > 0.f && den < T * UFL_NEAR) {
                // some term of this entry is (or is close to) one the reference's float32 exp flushes to 0 (zigap.py:86,
                // sparse_zigap.py:109): redo the entry from its terms, dropping those; nothing survives -> den = 1, no
                // count assigned (:90).  SPARSE: sV carries the mask S_tilde, the sums contract with sVz = sV * S_hat.
                float d2 = 0.f;
#pragma unroll
                for (int k = 0; k < KP; ++k) { const float tk = eu[k] * sV[g][k]; d2 += tk > T ? tk : 0.f; }
                const float r2 = d2 > 0.f ? x / d2 : 0.f;
#pragma unroll
                for (int k = 0; k < KP; ++k)
                    if (eu[k] * sV[g][k] > T) zi[k] = fmaf(r2, SPARSE ? sVz[SPARSE ? g : 0][k] : sV[g][k], zi[k]);
                R = 0.f;
            }
            float D = 1.f;
            if (DROPOUT) {
                float e, ex;
                const float pz = dropout_p(uv, slp[g], sfl[g], e, ex);
                D = nz ? 1.f : pz;                       // zigap.py:135-136: float32(1 - 1e-10) == 1
                if (ELBO && !nz) t_ent += __logf(1.f + ex) - (1.f - pz) * e;
                sX[tid][g] = row_ok ? D : 0.f;           // for the column sums below
            }
            if (ELBO && nz) t_xl = fmaf(x, logf(den), t_xl);
            const float4* z4 = SPARSE ? reinterpret_cast<const float4*>(&sVz[SPARSE ? g : 0][0]) : v4;
            const float4* c4 = SPARSE ? reinterpret_cast<const float4*>(&sVc[SPARSE && DROPOUT ? g : 0][0]) : h4;
#pragma unroll
            for (int q = 0; q < KP / 4; ++q) {
                const float4 v = z4[q];
                zi[4 * q + 0] = fmaf(R, v.x, zi[4 * q + 0]); zi[4 * q + 1] = fmaf(R, v.y, zi[4 * q + 1]);
                zi[4 * q + 2] = fmaf(R, v.z, zi[4 * q + 2]); zi[4 * q + 3] = fmaf(R, v.w, zi[4 * q + 3]);
                if (DROPOUT) {
                    const float4 h = c4[q];
                    as[4 * q + 0] = fmaf(D, h.x, as[4 * q + 0]); as[4 * q + 1] = fmaf(D, h.y, as[4 * q + 1]);
                    as[4 * q + 2] = fmaf(D, h.z, as[4 * q + 2]); as[4 * q + 3] = fmaf(D, h.w, as[4 * q + 3]);
                }
            }
        }
        if (ELBO) { acc_xl += (double)t_xl; acc_ent += (double)t_ent; }

        if (DROPOUT) {  // column sums of D_hat over this CTA's 128 cells -> pi (zigap.py:158)
            __syncthreads();
            float cs = 0.f;
            if (lane < gcount) {
#pragma unroll 8
                for (int rr = 0; rr < 32; ++rr) cs += sX[warp * 32 + rr][lane];
            }
            if (lane < TG) scs[warp][lane] = cs;
            __syncthreads();
            if (tid < gcount) {
                float tot = 0.f;
#pragma unroll
                for (int w = 0; w < PR_TR / 32; ++w) tot += scs[w][tid];
                if (det_cs) det_cs[(long long)blockIdx.x * p + j0 + tid] = (double)tot;
                else atomicAdd(colsum + j0 + tid, (double)tot);
            }
        }
    }

    if (row_ok) {
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            atomicAdd(Zi + row * KP + k, zi[k]);
            if (DROPOUT) atomicAdd(a2s + row * KP + k, as[k]);
        }
    }
    if (ELBO) {
        if (!row_ok) { acc_xl = 0.0; acc_ent = 0.0; }
        const double s1 = block_reduce_sum(acc_xl, sred);
        const double s2 = block_reduce_sum(acc_ent, sred);
        if (tid == 0) {
            if (det_part) { det_part[2 * blockIdx.x] = s1; det_part[2 * blockIdx.x + 1] = s2; }
            else { atomicAdd(&part64[ORI_R64_XLOGDEN], s1); atomicAdd(&part64[ORI_R64_ENT], s2); }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Gene pass.  CTA = 128 threads = 128 consecutive genes; thread keeps its gene's eV, V_hat and 2*KP
// accumulators in registers and sweeps a chunk of cells; X is read straight from global (coalesced),
// the row operands of 32 cells at a time are broadcast from smem.
constexpr int PG_TG = 128;
constexpr int PG_TR = 32;

// THIRD: a third sum Zl[j,k] = sum_i R_ij eU_ik E[log U_ik] (zigap.py:95, sparse_zigap.py:116) with the sweep operand
// eUl = eU * E[log U].  The sparse model passes eV = its masked denominator operand and Vh = the previous effective
// V_hat (see k_pass_rows).
template <int KP, bool DROPOUT, bool QUIRK, bool THIRD, class XT>
__global__ void __launch_bounds__(PG_TG)
k_pass_genes(const XT* __restrict__ X, long long ldx, long long n_rows, int p, int rows_per_chunk,
             const float* __restrict__ eU, const float* __restrict__ eUw, const float* __restrict__ Uh,
             const float* __restrict__ Un, const float* __restrict__ eUl,
             const float* __restrict__ eV, const float* __restrict__ Vh,
             const float* __restrict__ lp, const float* __restrict__ pfloor,
             float* __restrict__ Zj, float* __restrict__ b2s, float* __restrict__ Zl,
             const float* __restrict__ thrU, const float* __restrict__ thrV,
             float* __restrict__ det_z, long long det_stride)
{
    // det_z (ORI_F_DETERMINISTIC): the sums of row chunk blockIdx.y are stored to det_z[blockIdx.y][Zj | b2s | Zl][p x KP]
    // instead of added atomically; k_det_sum_chunks adds the chunks in index order
    __shared__ float sthr[PG_TR];
    __shared__ __align__(16) float sUl[THIRD ? PG_TR : 1][KP];
    __shared__ __align__(16) float sU[PG_TR][KP];
    __shared__ __align__(16) float sUw[QUIRK ? PG_TR : 1][KP];
    __shared__ __align__(16) float sUh[DROPOUT ? PG_TR : 1][KP];
    __shared__ __align__(16) float sUn[DROPOUT ? PG_TR : 1][KP];

    const int tid = threadIdx.x;
    const int j = blockIdx.x * PG_TG + tid;
    const bool j_ok = j < p;
    const long long r_begin = (long long)blockIdx.y * rows_per_chunk;
    const long long r_end = min(n_rows, r_begin + rows_per_chunk);

    float ev[KP], vh[DROPOUT ? KP : 1], zj[KP], bs[DROPOUT ? KP : 1], zl[THIRD ? KP : 1];
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        ev[k] = j_ok ? eV[(long long)j * KP + k] : 0.f;
        zj[k] = 0.f;
        if (THIRD) zl[k] = 0.f;
        if (DROPOUT) { vh[k] = j_ok ? Vh[(long long)j * KP + k] : 0.f; bs[k] = 0.f; }
    }
    const float lpj = (DROPOUT && j_ok) ? lp[j] : 0.f;
    const float flj = (DROPOUT && j_ok) ? pfloor[j] : 0.f;
    const float tv = (thrV && j_ok) ? thrV[j] : 0.f;            // underflow emulation (special.cuh); 0: never triggers

    float* sUf = &sU[0][0]; float* sUwf = &sUw[0][0]; float* sUhf = &sUh[0][0]; float* sUnf = &sUn[0][0];
    float* sUlf = &sUl[0][0];
    for (long long r0 = r_begin; r0 < r_end; r0 += PG_TR) {
        const int rcount = (int)min((long long)PG_TR, r_end - r0);
        __syncthreads();
        // rows past rcount are zero-filled: they contribute nothing (R = 0 and U_hat_new = 0)
        for (int idx = tid; idx < PG_TR * KP; idx += PG_TG) {
            const bool ok = idx / KP < rcount;
            sUf[idx] = ok ? eU[r0 * KP + idx] : 0.f;
            if (QUIRK) sUwf[idx] = ok ? eUw[r0 * KP + idx] : 0.f;
            if (THIRD) sUlf[idx] = ok ? eUl[r0 * KP + idx] : 0.f;
            if (DROPOUT) {
                sUhf[idx] = ok ? Uh[r0 * KP + idx] : 0.f;
                sUnf[idx] = ok ? Un[r0 * KP + idx] : 0.f;
            }
        }
        if (tid < PG_TR) sthr[tid] = (thrU && tid < rcount) ? thrU[r0 + tid] : 0.f;
        __syncthreads();
        for (int rb = 0; rb < PG_TR; rb += 8) {
            float xs[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                xs[u] = (j_ok && rb + u < rcount) ? ldg_count(X + (r0 + rb + u) * ldx + j) : 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int rr = rb + u;
                const float x = xs[u];
                float den = 0.f, uv = 0.f;
                const float4* u4 = reinterpret_cast<const float4*>(&sU[rr][0]);
                const float4* w4 = reinterpret_cast<const float4*>(&sUw[QUIRK ? rr : 0][0]);
                const float4* h4 = reinterpret_cast<const float4*>(&sUh[DROPOUT ? rr : 0][0]);
                const float4* n4 = reinterpret_cast<const float4*>(&sUn[DROPOUT ? rr : 0][0]);
                const float4* l4 = reinterpret_cast<const float4*>(&sUl[THIRD ? rr : 0][0]);
#pragma unroll
                for (int q = 0; q < KP / 4; ++q) {
                    const float4 uu = u4[q];
                    den = fmaf(uu.x, ev[4 * q + 0], den); den = fmaf(uu.y, ev[4 * q + 1], den);
                    den = fmaf(uu.z, ev[4 * q + 2], den); den = fmaf(uu.w, ev[4 * q + 3], den);
                    if (DROPOUT) {
                        const float4 h = h4[q];
                        uv = fmaf(h.x, vh[4 * q + 0], uv); uv = fmaf(h.y, vh[4 * q + 1], uv);
                        uv = fmaf(h.z, vh[4 * q + 2], uv); uv = fmaf(h.w, vh[4 * q + 3], uv);
                    }
                }
                den = den > 0.f ? den : 1.f;
                float R = x / den;
                const float T = tv * sthr[rr];
                if (x != 0.f && T > 0.f && den < T * UFL_NEAR) {     // see k_pass_rows
                    float d2 = 0.f;
#pragma unroll
                    for (int k = 0; k < KP; ++k) { const float tk = sU[rr][k] * ev[k]; d2 += tk > T ? tk : 0.f; }
                    const float r2 = d2 > 0.f ? x / d2 : 0.f;
#pragma unroll
                    for (int k = 0; k < KP; ++k)
                        if (sU[rr][k] * ev[k] > T) {
                            zj[k] = fmaf(r2, QUIRK ? sUw[QUIRK ? rr : 0][k] : sU[rr][k], zj[k]);
                            if (THIRD) zl[k] = fmaf(r2, sUl[THIRD ? rr : 0][k], zl[k]);
                        }
                    R = 0.f;
                }
                float D = 1.f;
                if (DROPOUT) {
                    float e, ex;
                    const float pz = dropout_p(uv, lpj, flj, e, ex);
                    D = (x != 0.f) ? 1.f : pz;
                }
#pragma unroll
                for (int q = 0; q < KP / 4; ++q) {
                    const float4 uu = QUIRK ? w4[q] : u4[q];
                    zj[4 * q + 0] = fmaf(R, uu.x, zj[4 * q + 0]); zj[4 * q + 1] = fmaf(R, uu.y, zj[4 * q + 1]);
                    zj[4 * q + 2] = fmaf(R, uu.z, zj[4 * q + 2]); zj[4 * q + 3] = fmaf(R, uu.w, zj[4 * q + 3]);
                    if (DROPOUT) {
                        const float4 nn = n4[q];
                        bs[4 * q + 0] = fmaf(D, nn.x, bs[4 * q + 0]); bs[4 * q + 1] = fmaf(D, nn.y, bs[4 * q + 1]);
                        bs[4 * q + 2] = fmaf(D, nn.z, bs[4 * q + 2]); bs[4 * q + 3] = fmaf(D, nn.w, bs[4 * q + 3]);
                    }
                    if (THIRD) {
                        const float4 ll = l4[q];
                        zl[4 * q + 0] = fmaf(R, ll.x, zl[4 * q + 0]); zl[4 * q + 1] = fmaf(R, ll.y, zl[4 * q + 1]);
                        zl[4 * q + 2] = fmaf(R, ll.z, zl[4 * q + 2]); zl[4 * q + 3] = fmaf(R, ll.w, zl[4 * q + 3]);
                    }
                }
            }
        }
    }
    if (j_ok && det_z) {
        float* base = det_z + (long long)blockIdx.y * det_stride + (long long)j * KP;
        const long long pk = (long long)p * KP;
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            base[k] = zj[k];
            if (DROPOUT) base[pk + k] = bs[k];
            if (THIRD) base[2 * pk + k] = zl[k];
        }
    } else if (j_ok) {
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            atomicAdd(Zj + (long long)j * KP + k, zj[k]);
            if (DROPOUT) atomicAdd(b2s + (long long)j * KP + k, bs[k]);
            if (THIRD) atomicAdd(Zl + (long long)j * KP + k, zl[k]);
        }
    }
}

// ORI_F_DETERMINISTIC helpers of the CUDA-core passes: ordered sums over CTAs / row chunks
__global__ void k_det_sum_cols(double* __restrict__ colsum, const double* __restrict__ det_cs, int nb, int p)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    double s = 0.0;
    for (int b = 0; b < nb; ++b) s += det_cs[(long long)b * p + j];
    colsum[j] += s;
}
__global__ void k_det_sum_chunks_strided(float* __restrict__ dst, const float* __restrict__ det_z, int ny, long long total,
                                         long long stride)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    float s = 0.f;
    for (int y = 0; y < ny; ++y) s += det_z[(long long)y * stride + i];
    dst[i] += s;
}

// ------------------------------------------------------------------------------------------------
// Factor update (both sides).  One thread per (row, k):
//   h1 = clamp(c1_k + acc1 * e_old)            zigap.py:115,117 / :123,125
//   h2 = clamp(c2_k + acc2  [or rate_const_k]) zigap.py:116,118 / :124,126  (gap.py:98,106: column sums)
//   E = h1/h2, Elog = psi(float32(h1)) - log(float32(h2)), eE = exp(Elog)      gamma.py:37-61
// and the column sums the M-step needs (zigap.py:146-155) plus the ELBO terms of this factor.
// FROM_PARAMS: h1,h2 are read instead of computed (update_expectations, zigap.py:160-165).
template <bool FROM_PARAMS>
__global__ void __launch_bounds__(256)
k_factor_update(long long rows, int K, int KP,
                const float* __restrict__ acc1, const float* __restrict__ e_old,
                const float* __restrict__ acc2, const double* __restrict__ rate_const,
                const double* __restrict__ c1, const double* __restrict__ c2,
                const float* __restrict__ E_old,
                float* __restrict__ h1_io, float* __restrict__ h2_io,
                float* __restrict__ E_new, float* __restrict__ eE_new, float* __restrict__ eEl_new,
                const float* __restrict__ xsum,
                double* __restrict__ Slog, double* __restrict__ Shat,
                double* __restrict__ Hsum, double* __restrict__ PUVsum, int write_state,
                float* __restrict__ thr_out, double* __restrict__ blk_part)
{
    // blk_part (ORI_F_DETERMINISTIC): no floating-point atomics -- every thread keeps the sums of its own component (a
    // thread's k is fixed: the grid stride is a multiple of KP), the block adds them in thread order and writes its
    // partials to blk_part[block][DET_FU_SLOTS]; k_det_sum_blocks adds the blocks in index order.
    __shared__ double sSlog[64], sShat[64], sH, sP;
    __shared__ double sA[256], sB[256];
    double dSlog = 0.0, dShat = 0.0;
    __shared__ float smax[8];
    if (threadIdx.x < 64) { sSlog[threadIdx.x] = 0.0; sShat[threadIdx.x] = 0.0; }
    if (threadIdx.x == 0) { sH = 0.0; sP = 0.0; }
    __syncthreads();
    const long long total = rows * KP;
    const int warp = threadIdx.x >> 5;
    double tH = 0.0, tP = 0.0;
    // a row occupies KP consecutive threads (KP divides 256); the trip count is uniform over the block
    for (long long base = (long long)blockIdx.x * blockDim.x; base < total; base += (long long)gridDim.x * blockDim.x) {
        const long long idx = base + threadIdx.x;
        const bool in = idx < total;
        const int k = in ? (int)(idx % KP) : KP;
        const bool live = in && k < K;
        float h1 = 0.f, h2 = 0.f, E = 0.f, Elog = -INFINITY;
        if (live) {
            double h1d, h2d;
            if (FROM_PARAMS) {
                h1d = (double)h1_io[idx]; h2d = (double)h2_io[idx];
            } else {
                const double z = (double)(acc1[idx] * e_old[idx]);
                const double rate = acc2 ? (double)acc2[idx] : rate_const[k];
                h1d = clamp_param_f64(c1[k] + z);
                h2d = clamp_param_f64(c2[k] + rate);
                if (PUVsum && acc2) tP += (double)E_old[idx] * (double)acc2[idx];
            }
            h1 = (float)h1d; h2 = (float)h2d;
            E = (float)(h1d / h2d);
            Elog = (float)digamma_f64((double)h1) - logf(h2);
        }
        // largest log-expectation of the row -> centred exponent (special.cuh)
        float m = Elog;
        for (int o = (KP < 32 ? KP : 32) >> 1; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (KP == 64) {
            smax[warp] = m;
            __syncthreads();
            m = fmaxf(smax[warp], smax[warp ^ 1]);
            __syncthreads();
        }
        const bool dead = !(m > EXP_DEAD);
        const double shift = dead ? 0.0 : EXP_CENTER - (double)m;
        if (thr_out && write_state && in && k == 0) thr_out[idx / KP] = underflow_thr_f32(m);
        if (!live) {
            if (in && write_state) {
                E_new[idx] = 0.f; eE_new[idx] = 0.f;
                if (eEl_new) eEl_new[idx] = 0.f;
                if (!FROM_PARAMS) { h1_io[idx] = 0.f; h2_io[idx] = 0.f; }
            }
            continue;
        }
        if (write_state) {
            if (!FROM_PARAMS) { h1_io[idx] = h1; h2_io[idx] = h2; }
            E_new[idx] = E;
            const float eE = centred_exp_f32(Elog, m);
            eE_new[idx] = eE;
            if (eEl_new) eEl_new[idx] = eE != 0.f ? eE * Elog : 0.f;     // sparse_zigap.py:116 operand
        }
        if (!Slog) continue;
        if (blk_part) { dSlog += (double)Elog; dShat += (double)E; }
        else { atomicAdd(&sSlog[k], (double)Elog); atomicAdd(&sShat[k], (double)E); }
        // entropy of q: a - log b + lgamma(a) + (1 - a) psi(a), with psi(a) taken as Elog + log b from the float32
        // Elog that also enters the prior term (alpha1 - 1) sum Elog: when a ~ 1e-15 (zero NMF factors, base.py:38-40)
        // psi ~ -1e15 and the two terms only cancel if they carry the same rounding
        const double lb = log((double)h2);
        tH += (double)h1 - lb + lgamma((double)h1) + (1.0 - (double)h1) * ((double)Elog + lb);
        // the passes will see den * exp(shift_i + shift_j): sum_ij X_ij log den_ij gets back  - shift_i * sum_j X_ij
        if (k == 0 && xsum) tH -= shift * (double)xsum[idx / KP];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tH += __shfl_xor_sync(0xffffffffu, tH, o);
        tP += __shfl_xor_sync(0xffffffffu, tP, o);
    }
    if (blk_part) {
        double* out = blk_part + (long long)blockIdx.x * DET_FU_SLOTS;
        sA[threadIdx.x] = dSlog; sB[threadIdx.x] = dShat;
        __shared__ double sW[2][8];
        if ((threadIdx.x & 31) == 0) { sW[0][warp] = tH; sW[1][warp] = tP; }
        __syncthreads();
        if (threadIdx.x < KP) {
            double a = 0.0, b = 0.0;
            for (int r = 0; r < 256 / KP; ++r) { a += sA[r * KP + threadIdx.x]; b += sB[r * KP + threadIdx.x]; }
            out[threadIdx.x] = a; out[64 + threadIdx.x] = b;
        }
        if (threadIdx.x == 0) {
            double h = 0.0, q = 0.0;
            for (int w = 0; w < 8; ++w) { h += sW[0][w]; q += sW[1][w]; }
            out[128] = h; out[129] = q;
        }
        return;
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sH, tH); atomicAdd(&sP, tP); }
    __syncthreads();
    if (Slog && threadIdx.x < K) {
        atomicAdd(Slog + threadIdx.x, sSlog[threadIdx.x]);
        atomicAdd(Shat + threadIdx.x, sShat[threadIdx.x]);
    }
    if (threadIdx.x == 0) {
        if (Slog) atomicAdd(Hsum, sH);
        if (PUVsum) atomicAdd(PUVsum, sP);
    }
}

// ------------------------------------------------------------------------------------------------
// M-step and ELBO assembly: one CTA.
__global__ void __launch_bounds__(1024)
k_mstep(ori_problem_t P, int mode)
{
    __shared__ double sbuf[32];
    const int tid = threadIdx.x;
    const int p = P.p, K = P.K;
    const double n = (double)P.n_total;
    const bool dropout = (P.flags & ORI_F_DROPOUT) != 0;
    const RedBufs red = red_carve(P);
    double* colsum = red.colsum, *SlogU = red.SlogU, *SU = red.SU, *part = red.part;
    double* SlogV = red.SlogV, *SV = red.SV, *gpart = red.gpart;

    // ---- phase 1: pi(t) and ELBO(t) of the state the row pass has just swept
    if (mode == ORI_M_STEP || mode == ORI_M_FINALIZE) {
        double bern = 0.0;
        if (dropout) {
            for (int j = tid; j < p; j += blockDim.x) {
                const double cs = colsum[j];
                const double pi = cs / n;                                  // zigap.py:158
                P.pi_d[j] = pi;
                const double pc = fmin(fmax(pi, 1e-15), 1.0 - 1e-15);
                bern += cs * log(pc) + (n - cs) * log1p(-pc);
                if (mode == ORI_M_STEP) {                                  // generates the next D_hat
                    P.lp[j] = pi <= 0.0 ? -INFINITY : (pi >= 1.0 ? INFINITY : (float)log(pc / (1.0 - pc)));
                    P.pfloor[j] = pi <= 0.0 ? 1e-10f : 0.f;                // zigap.py:133
                }
            }
        }
        const double b = block_reduce_sum(bern, sbuf);
        if (tid == 0) {
            double e = part[ORI_R64_XLOGDEN] - P.scal[ORI_SC_LGAMX] + P.scal[ORI_SC_PENDING];
            if (dropout) {
                const double q = 1e-10;  // p_d of a non-zero entry is 1 - 1e-10 (zigap.py:135)
                const double h_nz = -(1.0 - q) * log1p(-q) - q * log(q);
                e += -part[ORI_R64_PUV] + part[ORI_R64_ENT] + P.scal[ORI_SC_NNZ] * h_nz + b;
            } else {
                e -= P.scal[ORI_SC_UVSUM];  // sum_k (sum_i U_hat_ik)(sum_j V_hat_jk) of the swept state
            }
            P.scal[ORI_SC_ELBO_LAST] = e;
            const int it = (P.flags & ORI_F_DEVICE_ITER) ? (int)P.scal[ORI_SC_ITER] : P.iter;
            if (it >= 0 && it < P.trace_cap) P.elbo_trace[it] = e;
        }
        __syncthreads();
        if (mode == ORI_M_FINALIZE) return;
    }

    // ---- phase 2: M-step on the new expectations (zigap.py:143-155); alpha1 uses the OLD alpha2
    if (mode == ORI_M_INIT || mode == ORI_M_INIT_KEEP) {
        if (tid == 0) { P.scal[ORI_SC_LGAMX] = part[ORI_R64_LGAMX]; P.scal[ORI_SC_NNZ] = part[ORI_R64_NNZ]; }
        if (dropout)
            for (int j = tid; j < p; j += blockDim.x) {
                P.pi_d[j] = colsum[j] / n;        // column means of p_d = (X>0)  (base.py:52 -> zigap.py:158)
                P.lp[j] = -INFINITY;              // D_hat(0) is the indicator (zigap.py:77)
                P.pfloor[j] = 0.f;
            }
    }
    if (mode != ORI_M_INIT_KEEP && mode != ORI_M_REFRESH && tid < K) {
        double* a1 = P.hyper, *a2 = P.hyper + K, *b1 = P.hyper + 2 * K, *b2 = P.hyper + 3 * K;
        const int k = tid;
        double v = clamp_param_f64(inverse_digamma_f64(log(a2[k]) + SlogU[k] / n));
        a1[k] = v;
        a2[k] = clamp_param_f64(v / (SU[k] / n));
        v = clamp_param_f64(inverse_digamma_f64(log(b2[k]) + SlogV[k] / (double)p));
        b1[k] = v;
        b2[k] = clamp_param_f64(v / (SV[k] / (double)p));
    }
    __syncthreads();
    double pend = 0.0, uvs = 0.0;
    if (tid < K) {
        const double* a1 = P.hyper, *a2 = P.hyper + K, *b1 = P.hyper + 2 * K, *b2 = P.hyper + 3 * K;
        const int k = tid;
        pend = n * (a1[k] * log(a2[k]) - lgamma(a1[k])) + (a1[k] - 1.0) * SlogU[k] - a2[k] * SU[k]
             + (double)p * (b1[k] * log(b2[k]) - lgamma(b1[k])) + (b1[k] - 1.0) * SlogV[k] - b2[k] * SV[k];
        uvs = SU[k] * SV[k];
    }
    const double ps = block_reduce_sum(pend, sbuf);
    const double us = block_reduce_sum(uvs, sbuf);
    if (tid == 0) {
        P.scal[ORI_SC_PENDING] = ps + part[ORI_R64_HROW] + gpart[ORI_GSUM_HGENE];
        P.scal[ORI_SC_UVSUM] = us;
        const int it = (P.flags & ORI_F_DEVICE_ITER) ? (int)P.scal[ORI_SC_ITER] : P.iter;
        P.scal[ORI_SC_ITER] = (double)(mode == ORI_M_STEP ? it + 1 : it);
    }
}

// ------------------------------------------------------------------------------------------------
// Constant statistics of X: sum lgamma(X+1), nnz, column sums of (X>0).
template <class XT>
__global__ void __launch_bounds__(128)
k_count_stats(const XT* __restrict__ X, long long ldx, long long n_rows, int p, int rows_per_chunk,
              double* __restrict__ colsum, double* __restrict__ part64)
{
    __shared__ double sred[4];
    const int j = blockIdx.x * 128 + threadIdx.x;
    const long long r0 = (long long)blockIdx.y * rows_per_chunk;
    const long long r1 = min(n_rows, r0 + rows_per_chunk);
    double lg = 0.0; float cnt = 0.f;
    if (j < p)
        for (long long r = r0; r < r1; ++r) {
            const float x = ldg_count(X + r * ldx + j);
            if (x > 0.f) { cnt += 1.f; lg += (double)lgammaf(x + 1.f); }
        }
    if (j < p && cnt != 0.f) atomicAdd(colsum + j, (double)cnt);
    const double s1 = block_reduce_sum(lg, sred);
    const double s2 = block_reduce_sum((double)cnt, sred);
    if (threadIdx.x == 0) { atomicAdd(&part64[ORI_R64_LGAMX], s1); atomicAdd(&part64[ORI_R64_NNZ], s2); }
}

// eUw[i,k] = eU[i,k] * D_hat[i, gene k]   (the operand that reproduces zigap.py:94)
template <class XT>
__global__ void __launch_bounds__(256)
k_quirk_weights(const XT* __restrict__ X, long long ldx, long long n_rows, int K, int KP,
                const float* __restrict__ eU, const float* __restrict__ Uh, const float* __restrict__ Vh,
                const float* __restrict__ lp, const float* __restrict__ pfloor, float* __restrict__ eUw)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows * KP) return;
    const long long i = idx / KP; const int k = (int)(idx % KP);
    if (k >= K) { eUw[idx] = 0.f; return; }
    const float x = count_f32(X[i * ldx + k]);
    float D = 1.f;
    if (x == 0.f) {
        float uv = 0.f;
        for (int q = 0; q < K; ++q) uv = fmaf(Uh[i * KP + q], Vh[(long long)k * KP + q], uv);
        float e, ex;
        D = dropout_p(uv, lp[k], pfloor[k], e, ex);
    }
    eUw[idx] = eU[idx] * D;
}

// D_hat slab (tests / API access to model.D_hat): zigap.py:131-136
template <class XT>
__global__ void __launch_bounds__(256)
k_dropout_posterior(const XT* __restrict__ X, long long ldx, int p, int K, int KP,
                    const float* __restrict__ Uh, const float* __restrict__ Vh,
                    const float* __restrict__ lp, const float* __restrict__ pfloor,
                    float* __restrict__ out, long long ldo, long long row0, long long nrows)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nrows * p) return;
    const long long i = row0 + idx / p; const int j = (int)(idx % p);
    const float x = count_f32(X[i * ldx + j]);
    float D = 1.f;
    if (x == 0.f) {
        float uv = 0.f;
        for (int q = 0; q < K; ++q) uv = fmaf(Uh[i * KP + q], Vh[(long long)j * KP + q], uv);
        float e, ex;
        D = dropout_p(uv, lp[j], pfloor[j], e, ex);
    }
    out[(idx / p) * ldo + j] = D;
}

// ------------------------------------------------------------------------------------------------
// SparseZIGaP gene side (sparse_zigap.py:144-163, :198-204, :196): V' update, S update, expectations and the masked
// operands of the next iteration.  One thread per gene (the K components of a gene share logit(pi_s_j) and feed
// pi_s_j).  FROM_PARAMS: expectations from (b1, b2, p_s) as they are (update_expectations); pi_s is left alone.
__device__ __forceinline__ double nan_to_num_f64(double x) {
    if (x != x) return 0.0;
    if (x > 1.7976931348623157e308) return 1.7976931348623157e308;
    if (x < -1.7976931348623157e308) return -1.7976931348623157e308;
    return x;
}

template <bool FROM_PARAMS>
__global__ void __launch_bounds__(128)
k_sparse_gene_update(ori_problem_t P, double* __restrict__ blk_part)
{
    // blk_part (ORI_F_DETERMINISTIC): the column sums of E[log V'] and E[V'] are formed without atomics -- a fixed
    // shuffle tree per warp and component, the block's four warps in order, the blocks in order (k_det_sum_blocks)
    __shared__ double sSlog[64], sShat[64];
    __shared__ double sW[4][64][2];
    if (threadIdx.x < 64) { sSlog[threadIdx.x] = 0.0; sShat[threadIdx.x] = 0.0; }
    __syncthreads();
    const int p = P.p, K = P.K, KP = P.KP;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    double dL[32], dE[32];               // this gene's contributions (K <= 32), kept for the ordered sums
#pragma unroll
    for (int k = 0; k < 32; ++k) { dL[k] = 0.0; dE[k] = 0.0; }
    const RedBufs red = red_carve(P);
    if (j < p) {
        const float* Zj = red.Zj, *b2s = red.b2s, *Zl = red.Zl;
        const double* beta1 = P.hyper + 2 * K, *beta2 = P.hyper + 3 * K;
        const double pis = P.pi_s[j];
        const double lps = logit_f64(pis);
        double ssum = 0.0;
        float m = -INFINITY;
        for (int k = 0; k < KP; ++k) {
            const long long idx = (long long)j * KP + k;
            if (k >= K) {
                P.b1[idx] = 0.f; P.b2[idx] = 0.f; P.p_s[idx] = 0.f; P.logV[idx] = 0.f; P.eV[idx] = 0.f;
                P.eVd[idx] = 0.f; P.eVz[idx] = 0.f; P.Vh_old[idx] = 0.f; P.V_hat[idx] = 0.f;
                continue;
            }
            double h1d, h2d, ps;
            if (FROM_PARAMS) {
                h1d = (double)P.b1[idx]; h2d = (double)P.b2[idx]; ps = (double)P.p_s[idx];
            } else {
                const float S = P.p_s[idx];                       // S_hat of the iteration's start (:139)
                const float ed = P.eVd[idx], lV = P.logV[idx];
                const float RtU = Zj[idx], DtU = b2s[idx];
                const float DZ = RtU * ed;                        // :115
                const float DZl = fmaf(lV, RtU, Zl[idx]) * ed;    // :116
                h1d = clamp_param_f64(beta1[k] + (double)(S * DZ));            // :149, :151
                h2d = clamp_param_f64(beta2[k] + (double)S * (double)DtU);     // :150, :152
                const double Vp = h1d / h2d;
                const double tmp = -(double)DZl + nan_to_num_f64((double)DtU * Vp);   // :157-158
                ps = nan_to_num_f64(sigmoid_f64(lps - tmp));                           // :159-160
                if (pis <= 0.0) ps = 1e-10;                                            // :161
                if (pis >= 1.0) ps = 1.0 - 1e-10;                                      // :162
                P.b1[idx] = (float)h1d; P.b2[idx] = (float)h2d;
            }
            const float h1 = (float)h1d, h2 = (float)h2d;
            const float E = (float)(h1d / h2d);
            const float Elog = (float)digamma_f64((double)h1) - logf(h2);     // gamma.py:48-61
            const float Sn = (float)ps;                                       // bernoulli.py:45
            const float veff = Sn * E;                                        // :140
            P.Vh_old[idx] = FROM_PARAMS ? veff : P.V_hat[idx];
            P.p_s[idx] = Sn; P.logV[idx] = Elog; P.V_hat[idx] = veff;
            P.eVd[idx] = ps > P.tau ? 1.f : 0.f;                              // S_tilde (:134), scaled below
            m = fmaxf(m, Elog);
            if (blk_part) {
#pragma unroll
                for (int q = 0; q < 32; ++q) if (q == k) { dL[q] = (double)Elog; dE[q] = (double)E; }
            } else {
                atomicAdd(&sSlog[k], (double)Elog);
                atomicAdd(&sShat[k], (double)E);
            }
            ssum += ps;
        }
        // centred exponentials of this gene (special.cuh) and the masked operands of the next iteration
        for (int k = 0; k < K; ++k) {
            const long long idx = (long long)j * KP + k;
            const float eE = centred_exp_f32(P.logV[idx], m);
            const float ed_new = P.eVd[idx] * eE;                             // :103-104
            P.eV[idx] = eE; P.eVd[idx] = ed_new; P.eVz[idx] = ed_new * P.p_s[idx];
        }
        if (P.thrV) P.thrV[j] = underflow_thr_f32(m);
        if (!FROM_PARAMS) P.pi_s[j] = ssum / (double)K;                       // :196
    }
    if (blk_part) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            double a = dL[k], b = dE[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
            if (lane == 0) { sW[warp][k][0] = a; sW[warp][k][1] = b; }
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            double a = 0.0, b = 0.0;
            for (int w = 0; w < 4; ++w) { a += sW[w][threadIdx.x][0]; b += sW[w][threadIdx.x][1]; }
            double* out = blk_part + (long long)blockIdx.x * DET_FU_SLOTS;
            out[threadIdx.x] = a; out[64 + threadIdx.x] = b;
        }
        return;
    }
    __syncthreads();
    if (threadIdx.x < K) {
        atomicAdd(&red.SlogV[threadIdx.x], sSlog[threadIdx.x]);
        atomicAdd(&red.SV[threadIdx.x], sShat[threadIdx.x]);
    }
}

// ------------------------------------------------------------------------------------------------
// Column sums of X in float64 (column means for explained_deviance, base.py:76).
template <class XT>
__global__ void __launch_bounds__(128)
k_col_sums(const XT* __restrict__ X, long long ldx, long long n_rows, int p, int rows_per_chunk,
           double* __restrict__ out)
{
    const int j = blockIdx.x * 128 + threadIdx.x;
    if (j >= p) return;
    const long long r0 = (long long)blockIdx.y * rows_per_chunk;
    const long long r1 = min(n_rows, r0 + rows_per_chunk);
    double s = 0.0;
    for (long long r = r0; r < r1; ++r) s += (double)ldg_count(X + r * ldx + j);
    if (s != 0.0) atomicAdd(out + j, s);
}

// Row sums of X (float32): one warp per cell.
template <class XT>
__global__ void __launch_bounds__(256)
k_row_sums(const XT* __restrict__ X, long long ldx, long long n_rows, int p, float* __restrict__ out)
{
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int lane = threadIdx.x & 31;
    float s = 0.f;
    for (int j = lane; j < p; j += 32) s += ldg_count(X + row * ldx + j);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[row] = s;
}

// ------------------------------------------------------------------------------------------------
// Zero-inflated Poisson log-likelihood sums behind reconstruction_deviance / explained_deviance (base.py:58-82,
// sparse_zigap.py:44-51).  Same tiling as the row pass.  A float64 value assigned into the reference's int64
// buffer (sparse_zigap.py:45) is truncated toward zero; NaN / inf / out of range become INT64_MIN (x86 cvttsd2si).
__device__ __forceinline__ long long trunc_like_numpy(double v) {
    if (!(fabs(v) < 9.2233720368547758e18)) return (long long)0x8000000000000000ull;
    return (long long)v;
}

// EXACT: float64 throughout (the float64 sums are wanted).  Otherwise (integer sums only) the rate is a float32 dot
// product with a float64 fallback where it could underflow, the logarithms are float32 (an error of 1e-7 moves a term
// across an integer boundary with probability ~1e-7: invisible in sums of ~1e9), log(x) of small counts comes from a
// table, and zero entries whose terms all truncate to 0 are skipped.
constexpr int DEV_LOGX = 1024;

template <int KP, bool EXACT, class XT>
__global__ void __launch_bounds__(PR_TR)
k_deviance(const XT* __restrict__ X, long long ldx, long long n_rows, int p,
           const float* __restrict__ Uh, const float* __restrict__ b1, const float* __restrict__ b2,
           const float* __restrict__ Sh, const float* __restrict__ Vo,
           const float* __restrict__ lp, const float* __restrict__ pfloor,
           const double* __restrict__ pi, const double* __restrict__ cmean,
           unsigned long long* __restrict__ out_int, double* __restrict__ out_f64)
{
    __shared__ float sX[PR_TR][PR_TG + 1];
    // EXACT: the rate is accumulated in float64 from V' = b1 / b2 and S_hat -- the reference's float64 product
    // (base.py:63-66) stays positive where a float32 S_hat * V'_hat underflows, and log(0) would turn the metric into
    // INT64_MIN; the fast path keeps a float32 copy and falls back to float64 (from global memory) below 1e-30
    __shared__ __align__(16) double sVc[EXACT ? PR_TG : 1][KP];
    __shared__ __align__(16) float sVf[EXACT ? 1 : PR_TG][KP];
    __shared__ __align__(16) float sVo[PR_TG][KP];
    __shared__ float slp[PR_TG], sfl[PR_TG];
    __shared__ double spi[PR_TG], scm[PR_TG], slpi[PR_TG], slcm[PR_TG];
    __shared__ float slogx[EXACT ? 1 : DEV_LOGX];
    __shared__ float sgf[EXACT ? 1 : PR_TG][6];               // fast path: pi, 1 - pi, log pi, mean, log mean, exp(-mean)
    __shared__ double sred[PR_TR / 32];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long row0 = (long long)blockIdx.x * PR_TR;
    const long long row = row0 + tid;
    const bool row_ok = row < n_rows;
    float uh[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) uh[k] = row_ok ? Uh[row * KP + k] : 0.f;
    if (!EXACT)
        for (int i = tid; i < DEV_LOGX; i += PR_TR) slogx[i] = i ? (float)log((double)i) : 0.f;

    unsigned long long ti[3] = {0ull, 0ull, 0ull};
    double tf[3] = {0.0, 0.0, 0.0};
    const int ntiles = (p + PR_TG - 1) / PR_TG;
    for (int t = blockIdx.y; t < ntiles; t += gridDim.y) {
        const int j0 = t * PR_TG;
        const int gcount = min(PR_TG, p - j0);
        __syncthreads();
        for (int rr = warp; rr < PR_TR; rr += PR_TR / 32) {
            const long long r = row0 + rr;
            float v = 0.f;
            if (r < n_rows && lane < gcount) v = ldg_count(X + r * ldx + j0 + lane);
            sX[rr][lane] = v;
        }
        float* sVof = &sVo[0][0];
        for (int idx = tid; idx < PR_TG * KP; idx += PR_TR) {
            const bool ok = idx / KP < gcount;
            const long long gi = (long long)j0 * KP + idx;
            double v = 0.0;
            if (ok && b2[gi] != 0.f) v = (double)b1[gi] / (double)b2[gi] * (Sh ? (double)Sh[gi] : 1.0);   // pad columns: 0
            if (EXACT) (&sVc[0][0])[idx] = v; else (&sVf[0][0])[idx] = (float)v;
            sVof[idx] = ok ? Vo[gi] : 0.f;
        }
        if (tid < PR_TG) {
            const bool ok = tid < gcount;
            slp[tid] = ok ? lp[j0 + tid] : 0.f;
            sfl[tid] = ok ? pfloor[j0 + tid] : 0.f;
            spi[tid] = ok ? pi[j0 + tid] : 0.5;
            scm[tid] = ok ? cmean[j0 + tid] : 0.0;
            slpi[tid] = log(spi[tid]);                            // per-gene logarithms of the non-zero branch
            slcm[tid] = log(scm[tid]);
            if (!EXACT) {
                float* gf = &sgf[EXACT ? 0 : tid][0];
                gf[0] = (float)spi[tid]; gf[1] = (float)(1.0 - spi[tid]); gf[2] = (float)slpi[tid];
                gf[3] = (float)scm[tid]; gf[4] = (float)slcm[tid]; gf[5] = (float)exp(-scm[tid]);
            }
        }
        __syncthreads();
        if (!row_ok) continue;
        for (int g = 0; g < gcount; ++g) {
            const float x = sX[tid][g];
            const bool nz = x != 0.f;
            const double pj = spi[g], cm = scm[g], xd = (double)x;
            // integer-only mode: a zero entry's terms lie in (log(1 - pi_j), 0], so they all truncate to 0 when
            // 1 - pi_j >= 1/e -- no work at all for those genes' zeros
            if (!nz && !EXACT && (1.0 - pj) >= 0.36787944117144233) continue;
            // both contractions for every lane, four partial sums each: one serial chain of 32 dependent FMAs per
            // branch made this kernel latency-bound (3 warps per scheduler): 64 ms -> see DESIGN.md 4.4
            float uv = 0.f, Lfast = 0.f;
            {
                float u0 = 0.f, u1 = 0.f, u2 = 0.f, u3 = 0.f, l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
                const float4* o4 = reinterpret_cast<const float4*>(&sVo[g][0]);
                const float4* c4 = reinterpret_cast<const float4*>(&sVf[EXACT ? 0 : g][0]);
#pragma unroll
                for (int q = 0; q < KP / 4; ++q) {
                    const float4 o = o4[q];
                    u0 = fmaf(uh[4 * q + 0], o.x, u0); u1 = fmaf(uh[4 * q + 1], o.y, u1);
                    u2 = fmaf(uh[4 * q + 2], o.z, u2); u3 = fmaf(uh[4 * q + 3], o.w, u3);
                    if (!EXACT) {
                        const float4 c = c4[q];
                        l0 = fmaf(uh[4 * q + 0], c.x, l0); l1 = fmaf(uh[4 * q + 1], c.y, l1);
                        l2 = fmaf(uh[4 * q + 2], c.z, l2); l3 = fmaf(uh[4 * q + 3], c.w, l3);
                    }
                }
                uv = (u0 + u1) + (u2 + u3);
                Lfast = (l0 + l1) + (l2 + l3);
            }
            float D = 1.f;
            if (!nz) {                                            // D_hat only matters on zeros (zigap.py:135-136)
                float e, ex;
                D = dropout_p(uv, slp[g], sfl[g], e, ex);
            }
            const bool masked = !(D > 0.5f);                      // base.py:67: UV[round(D_hat) == 0] = 0
            if (!EXACT && masked && !nz) {                        // rate 0 on a zero entry: l_uv = l_sat = log(1) = 0
                const float* gf = &sgf[EXACT ? 0 : g][0];
                ti[2] += (unsigned long long)(long long)(int)__logf(fmaf(gf[0], gf[5], gf[1]));
                continue;
            }
            double L = 0.0, logL = -INFINITY;
            if (!masked) {
                if (EXACT) {
                    const double2* c2 = reinterpret_cast<const double2*>(&sVc[EXACT ? g : 0][0]);
#pragma unroll
                    for (int q = 0; q < KP / 4; ++q) {
                        const double2 ca = c2[2 * q], cb = c2[2 * q + 1];
                        L = fma((double)uh[4 * q + 0], ca.x, L); L = fma((double)uh[4 * q + 1], ca.y, L);
                        L = fma((double)uh[4 * q + 2], cb.x, L); L = fma((double)uh[4 * q + 3], cb.y, L);
                    }
                    logL = log(L);
                } else {
                    const float Lf = Lfast;
                    if (Lf >= 1e-30f) {
                        // everything in float32: terms below 2^23 in magnitude are truncated exactly like their float64
                        // twins except within ~1e-2 of an integer (a +-1 on a term of 1e3 ... 1e5, unbiased)
                        const float* gf = &sgf[EXACT ? 0 : g][0];
                        float f_uv, f_sat, f_mean;
                        if (!nz) {
                            f_uv = __logf(fmaf(gf[0], __expf(-Lf), gf[1]));
                            f_sat = 0.f;
                            f_mean = __logf(fmaf(gf[0], gf[5], gf[1]));
                        } else {
                            const int xi = (int)x;
                            const float logx = (x < (float)DEV_LOGX && (float)xi == x) ? slogx[EXACT ? 0 : xi] : logf(x);
                            f_uv = fmaf(x, __logf(Lf), gf[2] - Lf);
                            f_sat = fmaf(x, logx, gf[2] - x);
                            f_mean = fmaf(x, gf[4], gf[2] - gf[3]);
                        }
                        if (fabsf(f_uv) < 8e6f && fabsf(f_sat) < 8e6f && fabsf(f_mean) < 8e6f) {
                            ti[0] += (unsigned long long)(long long)(int)f_uv;
                            ti[1] += (unsigned long long)(long long)(int)f_sat;
                            ti[2] += (unsigned long long)(long long)(int)f_mean;
                            continue;
                        }
                        L = (double)Lf; logL = log(L);            // huge or non-finite term: the float64 path below
                    } else {                                      // rare: redo in float64 from the parameters
                        const long long gj = (long long)(j0 + g) * KP;
#pragma unroll
                        for (int k = 0; k < KP; ++k)
                            if (b2[gj + k] != 0.f)
                                L = fma((double)uh[k], (double)b1[gj + k] / (double)b2[gj + k] * (Sh ? (double)Sh[gj + k] : 1.0), L);
                        logL = log(L);
                    }
                }
            }
            double l_uv, l_sat, l_mean;
            if (!nz) {                                            // sparse_zigap.py:49
                if (EXACT) {
                    l_uv = log(pj * exp(-L) + (1.0 - pj));
                    l_sat = log(pj + (1.0 - pj));
                    l_mean = log(pj * exp(-cm) + (1.0 - pj));
                } else {
                    const float pf = (float)pj, qf = (float)(1.0 - pj);
                    l_uv = (double)logf(fmaf(pf, expf(-(float)L), qf));
                    l_sat = 0.0;
                    l_mean = (double)logf(fmaf(pf, expf(-(float)cm), qf));
                }
            } else {                                              // sparse_zigap.py:50
                const double lpi = slpi[g];
                const double logx = log(xd);
                l_uv = lpi - L + xd * logL;
                l_sat = lpi - xd + xd * logx;
                l_mean = lpi - cm + xd * slcm[g];
            }
            ti[0] += (unsigned long long)trunc_like_numpy(l_uv);
            ti[1] += (unsigned long long)trunc_like_numpy(l_sat);
            ti[2] += (unsigned long long)trunc_like_numpy(l_mean);
            if (EXACT) { tf[0] += l_uv; tf[1] += l_sat; tf[2] += l_mean; }
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ti[c] += __shfl_xor_sync(0xffffffffu, ti[c], o);
        if (lane == 0 && ti[c]) atomicAdd(out_int + c, ti[c]);
        if (EXACT) {
            const double r = block_reduce_sum(tf[c], sred);
            if (tid == 0) atomicAdd(out_f64 + c, r);
        }
    }
}

// ================================================================================================
// launchers
template <int KP>
static int pass_rows_kp(const ori_problem_t* P, int g, cudaStream_t st) {
    const int bx = cdiv(P->n_rows, PR_TR);
    constexpr int TGS = KP <= 32 ? PR_TG : 16;         // tile width of the sparse variant
    const bool sparse = P->flags & ORI_F_SPARSE;
    const int ntiles = cdiv(P->p, sparse ? TGS : PR_TG);
    int gy = 1;  // split the gene sweep until there are several waves of CTAs (3 resident per SM): a 1.8-wave grid idles
    while (bx * gy < 148 * 3 * 6 && gy * 2 <= ntiles) gy *= 2;   // most of the machine during its last wave
    const bool drop = P->flags & ORI_F_DROPOUT, elbo = P->flags & ORI_F_ELBO;
    const RedBufs red = red_carve(*P);
    double* colsum = red.colsum;
    double* part = red.part;
    // ORI_F_DETERMINISTIC: one CTA per row block (a single add per Zi / a2s element), per-CTA slots for the rest
    double* det_cs = nullptr; double* det_part = nullptr;
    if ((P->flags & ORI_F_DETERMINISTIC) && P->det_ws) {
        if (!det_simt_ok(P->n_rows, P->p)) return set_error(ORI_EUNSUPPORTED, "ORI_F_DETERMINISTIC on the CUDA-core kernels: problem too large");
        gy = 1;
        const DetWs d = det_carve(P->det_ws, P->n_rows, P->p);
        det_cs = d.simt_colsum;
        det_part = d.simt_elbo;
    }
    auto det_sums = [&]() -> int {
        if (!det_cs) return ORI_OK;
        int nk = 0;
        if (drop) { k_det_sum_cols<<<cdiv(P->p, 128), 128, 0, st>>>(colsum, det_cs, bx, P->p); ++nk; }
        if (elbo) { if (launch_det_sum_pairs(det_part, bx, part + ORI_R64_XLOGDEN, part + ORI_R64_ENT, st) != ORI_OK) return ORI_ECUDA; }
        return nk ? check_launch("k_det_sum_cols", nk) : ORI_OK;
    };
    dim3 grid(bx, gy);
    // sparse model (without ORI_F_DROPOUT: the operator seam, api.cu, D_hat folded into X): the masked operands of
    // k_pass_rows; ORI_F_SPARSE excludes ORI_F_ELBO
    const float* eV = sparse ? P->eVd : P->eV;
    const float* Vh = sparse ? P->Vh_old : P->V_hat;
    const float* eVz = sparse ? P->eVz : P->eV;
    with_counts(P, [&](auto X) {
#define ORI_LAUNCH_PR(D, E, S)                                                                                  \
        k_pass_rows<KP, D, E, S, S ? TGS : PR_TG, count_t<decltype(X)>><<<grid, PR_TR, 0, st>>>(X, P->ldx,         \
            P->n_rows, P->p, P->eU[g], P->U_hat[g], eV, Vh, eVz, P->V_hat, P->lp, P->pfloor, P->Zi, P->a2s, colsum, part, \
            (P->thrU && P->thrV) ? P->thrU + (long long)g * P->n_rows : nullptr, P->thrU ? P->thrV : nullptr,    \
            det_cs, det_part)
        if (sparse && drop) ORI_LAUNCH_PR(true, false, true);
        else if (sparse) ORI_LAUNCH_PR(false, false, true);
        else if (drop && elbo) ORI_LAUNCH_PR(true, true, false);
        else if (drop) ORI_LAUNCH_PR(true, false, false);
        else if (elbo) ORI_LAUNCH_PR(false, true, false);
        else ORI_LAUNCH_PR(false, false, false);
#undef ORI_LAUNCH_PR
        return ORI_OK;
    });
    if (check_launch("k_pass_rows") != ORI_OK) return ORI_ECUDA;
    return det_sums();
}

int launch_pass_rows_simt(const ori_problem_t* P, int g, cudaStream_t st) {
    switch (P->KP) {
        case 8: return pass_rows_kp<8>(P, g, st);
        case 16: return pass_rows_kp<16>(P, g, st);
        case 32: return pass_rows_kp<32>(P, g, st);
        case 64: return pass_rows_kp<64>(P, g, st);
    }
    return set_error(ORI_EINVAL, "KP must be 8, 16, 32 or 64 (got %d)", P->KP);
}

template <int KP>
static int pass_genes_kp(const ori_problem_t* P, int g, cudaStream_t st) {
    const int bx = cdiv(P->p, PG_TG);
    long long chunks = 1;
    while (bx * chunks < 148 * 4 && P->n_rows / (chunks * 2) >= 64) chunks *= 2;
    long long rpc = (P->n_rows + chunks - 1) / chunks;
    rpc = (rpc + PG_TR - 1) / PG_TR * PG_TR;
    if (rpc > 8192) rpc = 8192;  // bound the fp32 running sums
    const bool third = P->eUl[g] != nullptr;      // the third sum Zl into red32 block 2
    // ORI_F_DETERMINISTIC: nominal chunks only (their number bounds the scratch), every chunk stores to its own slot
    float* det_z = nullptr;
    const long long det_stride = ORI_RED32_FLOATS(P->p, P->KP, third);
    if ((P->flags & ORI_F_DETERMINISTIC) && P->det_ws) {
        if (!det_simt_ok(P->n_rows, P->p)) return set_error(ORI_EUNSUPPORTED, "ORI_F_DETERMINISTIC on the CUDA-core kernels: problem too large");
        rpc = DET_SIMT_CHUNK_ROWS;
        det_z = det_carve(P->det_ws, P->n_rows, P->p).simt_gene;
    }
    const int gy = cdiv(P->n_rows, rpc);
    dim3 grid(bx, gy);
    const bool drop = P->flags & ORI_F_DROPOUT, quirk = (P->flags & ORI_F_QUIRK) != 0;
    const RedBufs red = red_carve(*P);
    auto det_sums = [&]() -> int {
        if (!det_z) return ORI_OK;
        // blocks of the [Zj | b2s | Zl] scratch that this launch did not write (no dropout) are never read: sum what exists
        const long long total = drop ? det_stride : (long long)P->p * P->KP;
        k_det_sum_chunks_strided<<<cdiv(total, 256), 256, 0, st>>>(red.Zj, det_z, gy, total, det_stride);
        return check_launch("k_det_sum_chunks");
    };
    // sparse model (without ORI_F_DROPOUT: the operator seam, api.cu, D_hat folded into X): the masked denominator
    // operand and the previous effective V_hat; the quirk weight and the third sum are never asked for together
    const bool sparse = P->flags & ORI_F_SPARSE;
    const float* eV = sparse ? P->eVd : P->eV;
    const float* Vh = sparse ? P->Vh_old : P->V_hat;
    with_counts(P, [&](auto X) {
#define ORI_LAUNCH_PG(D, Q, T)                                                                                  \
        k_pass_genes<KP, D, Q, T, count_t<decltype(X)>><<<grid, PG_TG, 0, st>>>(X, P->ldx, P->n_rows, P->p, (int)rpc, \
            P->eU[g], P->eUw, P->U_hat[g], P->U_hat[1 - g], P->eUl[g], eV, Vh, P->lp, P->pfloor, red.Zj, red.b2s, red.Zl, \
            (P->thrU && P->thrV) ? P->thrU + (long long)g * P->n_rows : nullptr, P->thrU ? P->thrV : nullptr,    \
            det_z, det_stride)
        if (third && drop) ORI_LAUNCH_PG(true, false, true);
        else if (third) ORI_LAUNCH_PG(false, false, true);
        else if (drop && quirk) ORI_LAUNCH_PG(true, true, false);
        else if (drop) ORI_LAUNCH_PG(true, false, false);
        else if (quirk) ORI_LAUNCH_PG(false, true, false);
        else ORI_LAUNCH_PG(false, false, false);
#undef ORI_LAUNCH_PG
        return ORI_OK;
    });
    if (check_launch("k_pass_genes") != ORI_OK) return ORI_ECUDA;
    return det_sums();
}

int launch_pass_genes_simt(const ori_problem_t* P, int g, cudaStream_t st) {
    switch (P->KP) {
        case 8: return pass_genes_kp<8>(P, g, st);
        case 16: return pass_genes_kp<16>(P, g, st);
        case 32: return pass_genes_kp<32>(P, g, st);
        case 64: return pass_genes_kp<64>(P, g, st);
    }
    return set_error(ORI_EINVAL, "KP must be 8, 16, 32 or 64 (got %d)", P->KP);
}

// ORI_F_DETERMINISTIC: the per-block partials of k_factor_update, added block by block in index order
__global__ void k_det_sum_blocks(const double* __restrict__ blk_part, int nblocks, int K,
                                 double* __restrict__ Slog, double* __restrict__ Shat,
                                 double* __restrict__ Hsum, double* __restrict__ PUVsum)
{
    const int t = threadIdx.x;
    if (t >= DET_FU_SLOTS) return;
    double s = 0.0;
    for (int b = 0; b < nblocks; ++b) s += blk_part[(long long)b * DET_FU_SLOTS + t];
    if (t < 64) { if (Slog && t < K) Slog[t] += s; }
    else if (t < 128) { if (Slog && t - 64 < K) Shat[t - 64] += s; }
    else if (t == 128) { if (Slog && Hsum) *Hsum += s; }
    else if (PUVsum) *PUVsum += s;
}

static int update_grid(long long total) {
    long long b = (total + 255) / 256;
    return (int)(b < 1 ? 1 : (b > DET_FU_BLOCKS ? DET_FU_BLOCKS : b));
}

// write_state: 1 = regular update into generation 1-gen_old; 0 = only the ELBO term sum D_hat*uv of
// the swept state (finalize); 2 = expectations of generation gen_old from (a1,a2) with their column sums
// (init); 3 = the same expectations without touching any sum (host-streamed slabs).
int launch_row_update(const ori_problem_t* P, int g, int write_state, cudaStream_t st) {
    const int K = P->K, KP = P->KP;
    const RedBufs red = red_carve(*P);
    double* Hrow = red.part + ORI_R64_HROW;
    const bool drop = P->flags & ORI_F_DROPOUT, sparse = P->flags & ORI_F_SPARSE;
    const bool det = (P->flags & ORI_F_DETERMINISTIC) && P->det_ws;
    double* fu = det ? det_carve(P->det_ws, P->n_rows, P->p).fu_part : nullptr;
    const int grid = update_grid(P->n_rows * KP);
    if (write_state >= 2) {
        const bool sums = write_state == 2;
        k_factor_update<true><<<grid, 256, 0, st>>>(P->n_rows, K, KP, nullptr, nullptr, nullptr, nullptr,
            nullptr, nullptr, nullptr, P->a1, P->a2, P->U_hat[g], P->eU[g], sparse ? P->eUl[g] : nullptr, P->xrow,
            sums ? red.SlogU : nullptr, red.SU, Hrow, nullptr, 1, P->thrU ? P->thrU + (long long)g * P->n_rows : nullptr,
            sums ? fu : nullptr);
        if (det && sums) k_det_sum_blocks<<<1, 256, 0, st>>>(fu, grid, K, red.SlogU, red.SU, Hrow, nullptr);
    } else {
        // GaP: rate = alpha2 + sum_j V_hat_jk (gap.py:98)
        k_factor_update<false><<<grid, 256, 0, st>>>(P->n_rows, K, KP, P->Zi, P->eU[g],
            drop ? P->a2s : nullptr, red.SV, P->hyper, P->hyper + K, P->U_hat[g],
            P->a1, P->a2, P->U_hat[1 - g], P->eU[1 - g], sparse ? P->eUl[1 - g] : nullptr, P->xrow, red.SlogU, red.SU,
            Hrow, red.part + ORI_R64_PUV, write_state, P->thrU ? P->thrU + (long long)(1 - g) * P->n_rows : nullptr, fu);
        if (det) k_det_sum_blocks<<<1, 256, 0, st>>>(fu, grid, K, red.SlogU, red.SU, Hrow, red.part + ORI_R64_PUV);
    }
    return check_launch("k_factor_update(rows)", det ? 2 : 1);
}

int launch_gene_update(const ori_problem_t* P, int write_state, cudaStream_t st) {
    const int p = P->p, K = P->K, KP = P->KP;
    const bool drop = P->flags & ORI_F_DROPOUT;
    const RedBufs red = red_carve(*P);
    double* Hgene = red.gpart + ORI_GSUM_HGENE;
    const bool det = (P->flags & ORI_F_DETERMINISTIC) && P->det_ws;
    double* fu = det ? det_carve(P->det_ws, P->n_rows, P->p).fu_part : nullptr;
    const int grid = update_grid((long long)p * KP);
    if (P->flags & ORI_F_SPARSE) {
        const int gs = cdiv(p, 128);
        if (det && gs > DET_FU_BLOCKS) return set_error(ORI_EUNSUPPORTED, "ORI_F_DETERMINISTIC: too many genes for the sparse update");
        if (write_state == 2) k_sparse_gene_update<true><<<gs, 128, 0, st>>>(*P, fu);
        else k_sparse_gene_update<false><<<gs, 128, 0, st>>>(*P, fu);
        if (det) k_det_sum_blocks<<<1, 256, 0, st>>>(fu, gs, K, red.SlogV, red.SV, nullptr, nullptr);
        return check_launch("k_sparse_gene_update", det ? 2 : 1);
    }
    if (write_state == 2) {
        k_factor_update<true><<<grid, 256, 0, st>>>(p, K, KP, nullptr, nullptr, nullptr, nullptr,
            nullptr, nullptr, nullptr, P->b1, P->b2, P->V_hat, P->eV, nullptr, P->xcol, red.SlogV, red.SV, Hgene, nullptr, 1,
            P->thrV, fu);
    } else {
        // GaP: rate = beta2 + sum_i U_hat_ik (gap.py:106) with the NEW U_hat
        k_factor_update<false><<<grid, 256, 0, st>>>(p, K, KP, red.Zj, P->eV, drop ? red.b2s : nullptr,
            red.SU, P->hyper + 2 * K, P->hyper + 3 * K, nullptr,
            P->b1, P->b2, P->V_hat, P->eV, nullptr, P->xcol, red.SlogV, red.SV, Hgene, nullptr, write_state, P->thrV, fu);
    }
    if (det) k_det_sum_blocks<<<1, 256, 0, st>>>(fu, grid, K, red.SlogV, red.SV, Hgene, nullptr);
    return check_launch("k_factor_update(genes)", det ? 2 : 1);
}

int launch_mstep(const ori_problem_t* P, int mode, cudaStream_t st) {
    k_mstep<<<1, 1024, 0, st>>>(*P, mode);
    return check_launch("k_mstep");
}

int launch_count_stats(const ori_problem_t* P, cudaStream_t st) {
    const int bx = cdiv(P->p, 128);
    long long chunks = 1;
    while (bx * chunks < 148 * 4 && P->n_rows / (chunks * 2) >= 16) chunks *= 2;
    const long long rpc = (P->n_rows + chunks - 1) / chunks;
    dim3 grid(bx, cdiv(P->n_rows, rpc));
    const RedBufs red = red_carve(*P);
    with_counts(P, [&](auto X) {
        k_count_stats<<<grid, 128, 0, st>>>(X, P->ldx, P->n_rows, P->p, (int)rpc, red.colsum, red.part);
        return ORI_OK;
    });
    return check_launch("k_count_stats");
}

int launch_quirk_weights(const ori_problem_t* P, int g, cudaStream_t st) {
    const long long total = P->n_rows * P->KP;
    with_counts(P, [&](auto X) {
        k_quirk_weights<<<cdiv(total, 256), 256, 0, st>>>(X, P->ldx, P->n_rows, P->K, P->KP, P->eU[g],
                                                          P->U_hat[g], P->V_hat, P->lp, P->pfloor, P->eUw);
        return ORI_OK;
    });
    return check_launch("k_quirk_weights");
}

int launch_dropout_posterior(const ori_problem_t* P, int g, float* out, long long ldo, long long row0,
                             long long nrows, cudaStream_t st) {
    const long long total = nrows * P->p;
    if (total == 0) return ORI_OK;
    with_counts(P, [&](auto X) {
        k_dropout_posterior<<<cdiv(total, 256), 256, 0, st>>>(X, P->ldx, P->p, P->K, P->KP, P->U_hat[g],
                                                              (P->flags & ORI_F_SPARSE) ? P->Vh_old : P->V_hat, P->lp,
                                                              P->pfloor, out, ldo, row0, nrows);
        return ORI_OK;
    });
    return check_launch("k_dropout_posterior");
}

template <class XT>
int launch_col_sums(const XT* X, long long ldx, long long n_rows, int p, double* out, cudaStream_t st) {
    if (n_rows == 0) return ORI_OK;
    const int bx = cdiv(p, 128);
    long long chunks = 1;
    while (bx * chunks < 148 * 4 && n_rows / (chunks * 2) >= 16) chunks *= 2;
    const long long rpc = (n_rows + chunks - 1) / chunks;
    dim3 grid(bx, cdiv(n_rows, rpc));
    k_col_sums<<<grid, 128, 0, st>>>(X, ldx, n_rows, p, (int)rpc, out);
    return check_launch("k_col_sums");
}

template <class XT>
int launch_row_sums(const XT* X, long long ldx, long long n_rows, int p, float* out, cudaStream_t st) {
    if (n_rows == 0) return ORI_OK;
    k_row_sums<<<cdiv(n_rows, 8), 256, 0, st>>>(X, ldx, n_rows, p, out);
    return check_launch("k_row_sums");
}
template int launch_col_sums(const float*, long long, long long, int, double*, cudaStream_t);
template int launch_col_sums(const uint16_t*, long long, long long, int, double*, cudaStream_t);
template int launch_row_sums(const float*, long long, long long, int, float*, cudaStream_t);
template int launch_row_sums(const uint16_t*, long long, long long, int, float*, cudaStream_t);

template <int KP>
static int deviance_kp(const ori_problem_t* P, int g, const double* pi, const double* cmean, long long* out_int,
                       double* out_f64, cudaStream_t st) {
    const int bx = cdiv(P->n_rows, PR_TR);
    const int ntiles = cdiv(P->p, PR_TG);
    // the gene sweep is split so that there are >= 8 waves of CTAs (4 resident per SM): the per-tile global loads are
    // exposed, so resident warps are what hides them, and a 1.3-wave grid leaves two thirds of the machine idle at the end
    int gy = 1;
    while (bx * gy < 148 * 4 * 8 && gy * 2 <= ntiles) gy *= 2;
    const bool sparse = P->flags & ORI_F_SPARSE;
    with_counts(P, [&](auto X) {
        using XT = count_t<decltype(X)>;
        if (out_f64)
            k_deviance<KP, true, XT><<<dim3(bx, gy), PR_TR, 0, st>>>(X, P->ldx, P->n_rows, P->p, P->U_hat[g], P->b1, P->b2,
                sparse ? P->p_s : nullptr, sparse ? P->Vh_old : P->V_hat, P->lp, P->pfloor, pi, cmean,
                (unsigned long long*)out_int, out_f64);
        else
            k_deviance<KP, false, XT><<<dim3(bx, gy), PR_TR, 0, st>>>(X, P->ldx, P->n_rows, P->p, P->U_hat[g], P->b1, P->b2,
                sparse ? P->p_s : nullptr, sparse ? P->Vh_old : P->V_hat, P->lp, P->pfloor, pi, cmean,
                (unsigned long long*)out_int, nullptr);
        return ORI_OK;
    });
    return check_launch("k_deviance");
}

int launch_deviance(const ori_problem_t* P, int g, const double* pi, const double* cmean, long long* out_int,
                    double* out_f64, cudaStream_t st) {
    switch (P->KP) {
        case 8: return deviance_kp<8>(P, g, pi, cmean, out_int, out_f64, st);
        case 16: return deviance_kp<16>(P, g, pi, cmean, out_int, out_f64, st);
        case 32: return deviance_kp<32>(P, g, pi, cmean, out_int, out_f64, st);
        case 64: return deviance_kp<64>(P, g, pi, cmean, out_int, out_f64, st);
    }
    return set_error(ORI_EINVAL, "KP must be 8, 16, 32 or 64 (got %d)", P->KP);
}

}  // namespace ori
