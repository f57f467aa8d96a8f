// synth.cu -- synthetic zero-inflated negative-binomial counts generated on the device (bench only;
// SURVEY.md section 8d).  The host cannot hold BASELINE.json's larger configurations (1M x 20k int64 is
// 160 GB), so each rank generates its own row block from a counter-based RNG.
#include "common.cuh"

namespace ori {

struct Philox {
    uint32_t k0, k1;
    __device__ Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
    __device__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
            const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
            c0 = h1 ^ c1 ^ a; c1 = l1; c2 = h0 ^ c3 ^ b; c3 = l0;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};

__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }  // (0,1)

// Gamma(2, 1/2) = (E1 + E2) / 2
__global__ void k_synth_factor(float* __restrict__ out, long long rows, int K, long long row0, uint64_t seed, uint32_t tag) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * K) return;
    const long long i = row0 + idx / K; const int k = (int)(idx % K);
    const uint4 r = Philox(seed)((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)k, tag);
    out[idx] = -0.5f * (__logf(u01(r.x)) + __logf(u01(r.y)));
}

__global__ void k_synth_pi(float* __restrict__ pi, int p, float z, uint64_t seed) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    const uint4 r = Philox(seed)((uint32_t)j, 0u, 0u, 0x50u);
    const float b = 1.f / z - 1.f;   // Beta(1, b): inverse CDF
    pi[j] = (z >= 1.f) ? 1.f : 1.f - __powf(1.f - u01(r.x), 1.f / b);
}

__global__ void __launch_bounds__(256)
k_synth_counts(float* __restrict__ X, long long ldx, long long row0, long long n_rows, int p, int K,
               const float* __restrict__ Us, const float* __restrict__ Vs, const float* __restrict__ pi,
               uint64_t seed, int nb)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows * ldx) return;
    const long long il = idx / ldx; const int j = (int)(idx % ldx);
    if (j >= p) { X[idx] = 0.f; return; }
    const long long i = row0 + il;
    const Philox ph(seed);
    uint4 r = ph((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)j, 0x58u);
    float x = 0.f;
    if (u01(r.x) < pi[j]) {
        float lam = 0.f;
        for (int k = 0; k < K; ++k) lam = fmaf(Us[il * K + k], Vs[(long long)j * K + k], lam);
        if (nb) lam *= -0.5f * (__logf(u01(r.y)) + __logf(u01(r.z)));
        if (lam > 60.f) {   // normal approximation (Box-Muller)
            const uint4 q = ph((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)j, 0x59u);
            const float zn = sqrtf(-2.f * __logf(u01(q.x))) * __cosf(6.2831853f * u01(q.y));
            x = fmaxf(0.f, rintf(lam + sqrtf(lam) * zn));
        } else {            // Knuth's product method
            const float L = __expf(-lam);
            float prod = u01(r.w);
            uint32_t ctr = 0x100u;
            int cnt = 0;
            while (prod > L && cnt < 400) {
                const uint4 q = ph((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)j, ctr++);
                const float u[4] = {u01(q.x), u01(q.y), u01(q.z), u01(q.w)};
#pragma unroll
                for (int t = 0; t < 4; ++t) if (prod > L) { ++cnt; prod *= u[t]; }
            }
            x = (float)cnt;
        }
    }
    X[idx] = x;
}

}  // namespace ori

using namespace ori;

extern "C" int ori_synth_counts_f32(float* X, int64_t ldx, int64_t row0, int64_t n_rows, int32_t p, int32_t K,
                                    uint64_t seed, float zero_level, int nb, float* Ustar, float* Vstar,
                                    float* pi, void* stream)
{
    if (!X || !Ustar || !Vstar || !pi || ldx < p || p <= 0 || K <= 0 || n_rows < 0 || !(zero_level > 0.f))
        return set_error(ORI_EINVAL, "ori_synth_counts_f32: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_rows == 0) return ORI_OK;
    k_synth_factor<<<cdiv(n_rows * K, 256), 256, 0, st>>>(Ustar, n_rows, K, row0, seed, 0x55u);
    k_synth_factor<<<cdiv((long long)p * K, 256), 256, 0, st>>>(Vstar, p, K, 0, seed, 0x56u);
    k_synth_pi<<<cdiv(p, 256), 256, 0, st>>>(pi, p, zero_level, seed);
    k_synth_counts<<<cdiv(n_rows * ldx, 256), 256, 0, st>>>(X, ldx, row0, n_rows, p, K, Ustar, Vstar, pi, seed, nb);
    return check_launch("k_synth_counts", 4);
}

// ---- compact count storage -> float32 (count-matrix ingest, oriana/singlecell/cmatrix.py:56-61 as_array) --------
// Counts are small integers: a host that keeps X as uint16 / uint8 halves / quarters the bytes that cross PCIe
// every step of the host-streamed iteration; the kernels still see the float32 matrix of zigap.py:112.
template <typename T>
__global__ void __launch_bounds__(256)
k_widen_counts(const T* __restrict__ src, long long lds, float* __restrict__ dst, long long ldd, long long rows, int p)
{
    const int p4 = (p + 3) >> 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * p4) return;
    const long long r = idx / p4;
    const int c = (int)(idx - r * p4) * 4;
    const T* s = src + r * lds + c;
    float* d = dst + r * ldd + c;
    if (c + 3 < p && ((lds * sizeof(T)) % (4 * sizeof(T)) == 0) && (((uintptr_t)s) % (4 * sizeof(T)) == 0)) {
        T v[4];
        if (sizeof(T) == 2) *reinterpret_cast<uint2*>(v) = *reinterpret_cast<const uint2*>(s);
        else *reinterpret_cast<uint32_t*>(v) = *reinterpret_cast<const uint32_t*>(s);
        *reinterpret_cast<float4*>(d) = make_float4((float)v[0], (float)v[1], (float)v[2], (float)v[3]);   // ldd % 4 == 0
    } else {
        for (int q = 0; q < 4 && c + q < p; ++q) d[q] = (float)s[q];
    }
}

extern "C" int ori_widen_counts_f32(const void* src, int elem_bytes, int64_t lds, float* dst, int64_t ldd,
                                    int64_t rows, int32_t p, void* stream)
{
    if (!src || !dst || lds < p || ldd < p || (ldd & 3) || ((uintptr_t)dst & 15) || p <= 0 || rows < 0 ||
        (elem_bytes != 1 && elem_bytes != 2))
        return set_error(ORI_EINVAL, "ori_widen_counts_f32: bad argument");
    if (rows == 0) return ORI_OK;
    const long long n = rows * ((p + 3) >> 2);
    if (elem_bytes == 2)
        k_widen_counts<uint16_t><<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((const uint16_t*)src, lds, dst, ldd, rows, p);
    else
        k_widen_counts<uint8_t><<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)src, lds, dst, ldd, rows, p);
    return check_launch("k_widen_counts");
}

// ---- bitmap + non-zero bytes -> float32 (sparse count-matrix ingest) ---------------------------------------------
// Single-cell count matrices are mostly zeros (cmatrix.py:100-104 as_sparse_matrix): a host that keeps, per cell, one
// bit per gene plus the non-zero counts as saturating bytes in gene order streams p / 8 + nnz bytes per cell per step
// instead of p.  Bit l of word w of a row = gene 32 w + l; rowoff[r] - base = position of row r's first non-zero byte.
// One CTA per row: (1) popcount prefix over the row's words, (2) lane l of a warp expands bit l of one word at a time,
// so every store is one coalesced 128-byte line and the bytes a word needs are consecutive.
constexpr int XB_WORDS = 1024;       // bitmap words per block of a row (256 threads x 4 words)
__global__ void __launch_bounds__(256)
k_expand_bitmap(const uint32_t* __restrict__ bm, long long wpr, const uint8_t* __restrict__ nz,
                const long long* __restrict__ rowoff, long long base, float* __restrict__ dst, long long ldd,
                long long rows, int p)
{
    __shared__ uint32_t s_word[XB_WORDS];
    __shared__ uint32_t s_off[XB_WORDS];
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = (p + 31) >> 5;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const uint8_t* src = nz + (rowoff[r] - base);
        const uint32_t* brow = bm + r * wpr;
        float* drow = dst + r * ldd;
        uint32_t carry = 0;
        for (int w0 = 0; w0 < W; w0 += XB_WORDS) {
            uint32_t wv[4], pre[4], sum = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int w = w0 + 4 * tid + i;
                wv[i] = w < W ? brow[w] : 0u;
                pre[i] = sum;
                sum += __popc(wv[i]);
            }
            uint32_t inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += v;
            }
            if (lane == 31) s_warp[warp] = inc;
            __syncthreads();
            uint32_t wbase = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) if (q < warp) wbase += s_warp[q];
            if (tid == 255) s_total = wbase + inc;
            const uint32_t excl = carry + wbase + inc - sum;
#pragma unroll
            for (int i = 0; i < 4; ++i) { s_word[4 * tid + i] = wv[i]; s_off[4 * tid + i] = excl + pre[i]; }
            __syncthreads();
            const int nw = min(XB_WORDS, W - w0);
            for (int j = warp; j < nw; j += 8) {
                const uint32_t word = s_word[j];
                const int col = (w0 + j) * 32 + lane;
                const bool bit = (word >> lane) & 1u;
                float v = 0.f;
                if (bit) v = (float)src[s_off[j] + __popc(word & ((1u << lane) - 1u))];
                if (col < p) drow[col] = v;
            }
            carry += s_total;
            __syncthreads();
        }
    }
}

extern "C" int ori_expand_bitmap_counts_f32(const uint32_t* bitmap, int64_t words_per_row, const uint8_t* nz,
                                            const int64_t* rowoff, int64_t base, float* dst, int64_t ldd,
                                            int64_t rows, int32_t p, void* stream)
{
    if (!bitmap || !rowoff || !dst || p <= 0 || rows < 0 || ldd < p || words_per_row < (p + 31) / 32)
        return set_error(ORI_EINVAL, "ori_expand_bitmap_counts_f32: bad argument");
    if (rows == 0) return ORI_OK;
    const int grid = (int)(rows < 148 * 64 ? rows : 148 * 64);
    k_expand_bitmap<<<grid, 256, 0, (cudaStream_t)stream>>>(bitmap, words_per_row, nz, (const long long*)rowoff, base, dst, ldd, rows, p);
    return check_launch("k_expand_bitmap");
}

// ---- CSR row slab -> X (sparse count-matrix ingest, cmatrix.py:39-54 as_sparse_matrix) -------------------------------
// Real single-cell matrices arrive as CSR (10x / Matrix Market, AnnData .X) with 2-10 % non-zeros: the host sends each
// non-zero as a column index and a count instead of the whole row.  One CTA per row: zero-fill the row's ldd elements
// with 16-byte stores (pad columns included, so the caller needs no memset), then scatter its non-zeros.  The indices of
// a row are distinct (canonical CSR), so the scattered stores never collide; the column guard keeps every store in its
// row's first p elements.  PCIe-bound where it is used (ingest, host-streamed slabs): no further tuning.
template <typename I, typename V, typename D>
__global__ void __launch_bounds__(256)
k_expand_csr(const long long* __restrict__ indptr, long long base, const I* __restrict__ idx, const V* __restrict__ val,
             D* __restrict__ dst, long long ldd, long long rows, int p)
{
    const int n16 = (int)(ldd * (long long)sizeof(D) / 16);        // ldd * sizeof(D) is a multiple of 16
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        D* drow = dst + r * ldd;
        uint4* d16 = reinterpret_cast<uint4*>(drow);
        for (int i = threadIdx.x; i < n16; i += blockDim.x) d16[i] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
        const long long lo = indptr[r] - base, hi = indptr[r + 1] - base;
        for (long long e = lo + threadIdx.x; e < hi; e += blockDim.x) {
            const long long c = (long long)idx[e];
            if (c >= 0 && c < p) drow[c] = (D)val[e];
        }
    }
}

template <typename I, typename V, typename D>
static void launch_expand_csr(const int64_t* indptr, int64_t base, const void* indices, const void* values, void* dst,
                              int64_t ldd, int64_t rows, int32_t p, cudaStream_t st)
{
    const int grid = (int)(rows < 148 * 64 ? rows : 148 * 64);
    k_expand_csr<I, V, D><<<grid, 256, 0, st>>>((const long long*)indptr, base, (const I*)indices, (const V*)values,
                                                (D*)dst, ldd, rows, p);
}

template <typename I, typename D>
static void launch_expand_csr_values(int32_t val_type, const int64_t* indptr, int64_t base, const void* indices,
                                     const void* values, void* dst, int64_t ldd, int64_t rows, int32_t p, cudaStream_t st)
{
    if (val_type == ORI_CSR_U8) launch_expand_csr<I, uint8_t, D>(indptr, base, indices, values, dst, ldd, rows, p, st);
    else if (val_type == ORI_CSR_U16) launch_expand_csr<I, uint16_t, D>(indptr, base, indices, values, dst, ldd, rows, p, st);
    else launch_expand_csr<I, float, float>(indptr, base, indices, values, dst, ldd, rows, p, st);   // D = float (checked)
}

extern "C" int ori_expand_csr_counts(const int64_t* indptr, int64_t base, const void* indices, int32_t idx_bytes,
                                     const void* values, int32_t val_type, void* dst, int32_t dst_bytes, int64_t ldd,
                                     int64_t rows, int32_t p, void* stream)
{
    if (!indptr || !dst || p <= 0 || rows < 0 || ldd < p || (idx_bytes != 2 && idx_bytes != 4) ||
        (val_type != ORI_CSR_U8 && val_type != ORI_CSR_U16 && val_type != ORI_CSR_F32) ||
        (dst_bytes != 2 && dst_bytes != 4) || (ldd % (16 / dst_bytes)) || ((uintptr_t)dst & 15) ||
        (val_type == ORI_CSR_F32 && dst_bytes == 2))
        return set_error(ORI_EINVAL, "ori_expand_csr_counts: bad argument");
    if (rows == 0) return ORI_OK;
    const cudaStream_t st = (cudaStream_t)stream;
    if (idx_bytes == 2) {
        if (dst_bytes == 4) launch_expand_csr_values<uint16_t, float>(val_type, indptr, base, indices, values, dst, ldd, rows, p, st);
        else launch_expand_csr_values<uint16_t, uint16_t>(val_type, indptr, base, indices, values, dst, ldd, rows, p, st);
    } else {
        if (dst_bytes == 4) launch_expand_csr_values<int32_t, float>(val_type, indptr, base, indices, values, dst, ldd, rows, p, st);
        else launch_expand_csr_values<int32_t, uint16_t>(val_type, indptr, base, indices, values, dst, ldd, rows, p, st);
    }
    return check_launch("k_expand_csr");
}

// Escapes of the saturating uint8 encoding: X[row[e] - row0, col[e]] = val[e] for the entries whose count does not
// fit a byte (stored as 255 in the compact matrix).  row is the GLOBAL cell index, row0 the first cell of the slab.
__global__ void __launch_bounds__(256)
k_scatter_counts(float* __restrict__ X, long long ldx, long long row0, long long rows, int p,
                 const int* __restrict__ row, const int* __restrict__ col, const float* __restrict__ val, long long count)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= count) return;
    const long long r = (long long)row[e] - row0;
    const int c = col[e];
    if (r >= 0 && r < rows && c >= 0 && c < p) X[r * ldx + c] = val[e];
}

extern "C" int ori_scatter_counts_f32(float* X, int64_t ldx, int64_t row0, int64_t rows, int32_t p, const int32_t* row,
                                      const int32_t* col, const float* val, int64_t count, void* stream)
{
    if (!X || ldx < p || p <= 0 || rows < 0 || count < 0 || (count && (!row || !col || !val)))
        return set_error(ORI_EINVAL, "ori_scatter_counts_f32: bad argument");
    if (count == 0 || rows == 0) return ORI_OK;
    k_scatter_counts<<<cdiv(count, 256), 256, 0, (cudaStream_t)stream>>>(X, ldx, row0, rows, p, row, col, val, count);
    return check_launch("k_scatter_counts");
}
