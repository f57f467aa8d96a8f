// kernels_tc.cu -- the two X-streaming passes of the CAVI iteration on the sm_100a tensor path:
// TMA-staged tiles, tcgen05.mma kind::tf32 with fp32 accumulators in TMEM, the ratio / dropout posterior
// computed between the two groups of contractions on the TMEM-resident tile (A operands from TMEM).
//
// Per tile of 128 "own" x SW "sweep" entries (own = cells in the row pass, genes in the gene pass; SW = 64 for a
// padded latent dimension KP = 32, SW = 32 for KP = 64, so that the tile always fits the same TMEM / smem plan):
//   S:  den = eO . eS^T     (hi.hi in tf32 + hi.lo + lo.hi in bf16)  zigap.py:86-90
//       uv  = Oh . Sh^T     (same split)                             zigap.py:131 (U_hat V_hat^T)
//   E:  R = X / den ; D = X != 0 ? 1 : max(sigmoid(lp - uv), floor)  zigap.py:91-92, :131-136
//       (written back over den / uv in TMEM, rounded to tf32 to nearest)
//   P:  acc1 += R . S1 ; acc2 += D . S2                              zigap.py:93-94 / :116, :124
// where S1, S2 are the transposed (K-major) copies of exp(E log .) and of the matching U_hat / V_hat.
//
// Data movement per CTA (one CTA per SM, persistent over work items = own tile x chunk of the sweep):
//   own side   the 128 own rows of exp(E log .) and E[.] are read once per work item from the raw factor
//              arrays, split hi/lo in registers and parked in TMEM (4 * KP columns): every S contraction takes
//              its A operand from TMEM, so shared memory only carries the streamed side;
//   sweep side three independent TMA rings: K-major hi/lo operands (consumed by S, freed as soon as S has
//              run), transposed operands (consumed by P) and the X tile (+ logit pi) for the element-wise
//              warps, so that a stage is recycled as early as its own consumer allows.
// MN-major tf32 operands would need the SWIZZLE_128B_ATOM_32B smem layout, which no K-major operand accepts,
// hence the transposed copies (prepared by k_tc_prep_*) and K-major descriptors everywhere
// (scripts/tc_probe.cu checks every descriptor form used here against the CPU).
//
// CTA pairs: two CTAs of a cluster sweep the same chunk with neighbouring own tiles; every MMA is a cta_group::2
// instruction of M = 256 issued by the pair's leader, each CTA stages only half of every streamed operand tile and
// TMA credits both halves to the leader's barrier; completion is multicast back.
//
// Warp roles (320 threads):
//   warp 0       TMA producer (whole warp walks the rings, one elected lane issues)
//   warp 1       MMA issuer + TMEM owner (warp-uniform control flow, one elected lane issues)
//   warps 2..9   element-wise warps; warp w owns TMEM lanes 32*(w%4).. and half of the tile's columns
#include <cstring>
#include "common.cuh"
#include "tc_ptx.cuh"

namespace ori {
using namespace tc;

constexpr int TC_OWN = 128;
constexpr int NEW = 8;                // element-wise warps, two per TMEM lane quarter
constexpr int TC_THREADS = 64 + 32 * NEW;
constexpr int NCTA = 2;               // CTAs of a cluster (pair)

// Plan of one kernel variant.  KP: padded latent dimension (32 or 64).  The CTA pair (cta_group::2, M = 256 over two
// SMs) stages only half of every streamed operand tile per CTA (the pair's MMA reads both halves), which halves the TMA
// fill and the tensor-core operand reads per SM and leaves room for deeper rings.
// The cross terms hi.lo + lo.hi of every 3xTF32 contraction run as ONE bf16 chain over [hi | lo] . [lo | hi] (error
// 2^-9 of a 2^-12 term): 4 instead of 6 MMA chains per tile.
//
// PRECISE (KP = 32): the accumulating contractions R . S1 and D . S2 are split-precision too -- R, D and the factor operands
// as tf32 hi plus a bf16 [hi | lo] . [lo | hi] chain for the two cross terms, like den / uv -- so every sum is fp32-grade
// (~2^-21) instead of TF32-grade (~2^-12 per term).  The tile keeps R16 / D16 (the packed bf16 pairs) beside R / D in TMEM,
// which halves the sweep width (32) to stay inside 512 columns.
template <int KP, bool PRECISE = false, bool DEVI = false>
struct Cfg {
    static_assert(KP == 32 || KP == 64, "tensor path: KP is 32 or 64");
    static_assert(!PRECISE || KP == 32, "the fp32-grade plan exists for KP = 32");
    static constexpr int SW = PRECISE ? 32 : 2048 / KP;   // sweep entries per tile
    static constexpr int NS = 2;                          // TMEM stages of [den/R | uv/D]
    static constexpr int KB = KP / 32;                    // 128-byte K blocks of a K-major row
    static constexpr int KST = 3, TST = 3, XST = 4;       // ring depths
    static constexpr int NTA = PRECISE ? 4 : 2;           // transposed operand arrays per stage: e, E [, bf16 pairs of e, of E]
    // K-major operand array of one tile: [KB blocks][SW / NCTA sweep rows][32 floats], 128-byte swizzled
    static constexpr uint32_t K_BLK = (SW / NCTA) * 128;
    static constexpr uint32_t K_ARR = KB * K_BLK;
    static constexpr uint32_t K_STAGE = 4 * K_ARR;        // hi(e) lo(e) hi(E) lo(E)
    // transposed operand array of one tile: [SW / 32 chunks][KP / NCTA latent rows][32 sweep columns]
    static constexpr uint32_t T_CHUNK = (KP / NCTA) * 128;
    static constexpr uint32_t T_ARR = (SW / 32) * T_CHUNK;
    static constexpr uint32_t T_STAGE = NTA * T_ARR;      // transposed e and transposed E (+ their bf16 [lo | hi] pairs)
    static constexpr uint32_t X_STAGE = TC_OWN * SW * 4;  // X tile
    // per-gene constants of a tile: lp2[SW] | floor[SW] | (1-pi)/pi [SW]; deviance pass: 8 arrays (k_tc_prep_dev)
    static constexpr uint32_t LP_STAGE = (DEVI ? 8 : 3) * SW * 4;
    static constexpr uint32_t OFF_K = 0;
    static constexpr uint32_t OFF_T = OFF_K + KST * K_STAGE;
    static constexpr uint32_t OFF_X = OFF_T + TST * T_STAGE;
    static constexpr uint32_t OFF_LP = OFF_X + XST * X_STAGE;
    static constexpr uint32_t OFF_BAR = OFF_LP + XST * LP_STAGE;
    static constexpr uint32_t SMEM_BYTES = OFF_BAR + 512 + 1024;   // + barriers + alignment slack
    // TMEM columns: NS stages of [den/R SW | uv/D SW], accumulators [acc1 KP | acc2 KP], own operands 4 x KP
    // stage: [den/R SW | uv/D SW], or with PRECISE [den/R SW | R16 SW | uv/D SW | D16 SW]
    static constexpr uint32_t TM_UV = PRECISE ? 2 * SW : SW;
    static constexpr uint32_t TM_STAGE = PRECISE ? 4 * SW : 2 * SW;
    static constexpr uint32_t TM_ACC = NS * TM_STAGE;
    static constexpr uint32_t TM_A = TM_ACC + 2 * KP;
    static constexpr uint32_t TM_COLS = 512;
    static_assert(TM_A + 4 * KP <= TM_COLS, "TMEM plan");
    // mbarriers.  KFULL / TFULL / PREADY / ACC_FREE / A_READY are used in the leader CTA only
    // (the peer's TMA bytes and warp arrivals are credited there); the others are per CTA.
    static constexpr int B_KFULL = 0, B_KEMPTY = B_KFULL + KST, B_TFULL = B_KEMPTY + KST, B_TEMPTY = B_TFULL + TST,
                         B_XFULL = B_TEMPTY + TST, B_XEMPTY = B_XFULL + XST, B_SREADY = B_XEMPTY + XST,
                         B_PREADY = B_SREADY + NS, B_ACC_READY = B_PREADY + NS, B_ACC_FREE = B_ACC_READY + 1,
                         B_A_READY = B_ACC_FREE + 1, NBARS = B_A_READY + 1;
    static_assert(NBARS * 8 + 8 <= 512, "barrier area");
    static_assert(SMEM_BYTES <= 232448, "shared memory");
};

struct TcMaps { CUtensorMap swK, swT, X; };

struct TcArgs {
    long long own_total, sw_total;   // valid extents (cells / genes)
    long long sw_pad;                // padded sweep extent (multiple of 128): q-th operand array starts at row q*pad
    int n_own_tiles, n_own_units, n_chunks, tiles_per_chunk, n_sw_tiles, n_items;   // unit = pair of own tiles
    const float* own_e;              // [own_total x KP] exp(E log .) of the own side (raw factor array)
    const float* own_E;              // [own_total x KP] E[.] of the own side
    const float* lp2w;               // [genes_pad] logit(pi) * log2(e); -inf: D_hat = (X>0)
    const float* flw;                // [genes_pad] floor (1e-10 where pi <= 0)
    const float* cw;                 // [genes_pad] exp(-logit(pi)) = (1 - pi) / pi
    const int* any_floor;            // != 0 when some gene has a floor
    float* acc1;                     // [own_total x KP]  sum_sweep R  * S1
    float* acc2;                     // [own_total x KP]  sum_sweep D  * S2
    double* colsum;                  // gene pass: [genes] += sum_i D_hat
    double* part64;                  // gene pass: ELBO partial sums
    // deviance pass (DEVI): per-gene constants, tile-major [n_sw_tiles][8][SW]; float64 fallback operands; int64 sums
    const float* devlp;
    const float* dev_b1; const float* dev_b2; const float* dev_ps;     // V' = b1 / b2 (* S_hat) [genes x KP]
    unsigned long long* dev_out;     // [3] truncated log-likelihood sums at the rates U V^T (masked), X, column means
    // float32-underflow emulation (special.cuh: underflow_thr_f32; zigap.py:86-90), all NULL = off: an entry with
    // den < thr_own * thr_sw assigns its count to no component.  The fast path only compares the smallest denominator of
    // a group with thr_own * max(thr_sw) -- no instruction per entry -- and sends the group to the general path.
    const float* thr_own;            // [own_total]
    const float* thr_sw;             // [sw_total]
    const float* thr_sw_max;         // [1] largest thr_sw
    // ORI_F_DETERMINISTIC (both NULL otherwise): the chunk items of an own tile add their accumulators in chunk order
    // -- tickets[tile] counts the element-wise warps that have finished, item by item -- and the ELBO terms of every
    // (item, CTA, warp) go to their own slot of item_part instead of one atomic target (k_det_sum_items adds them in order)
    int* tickets;                    // [n_own_tiles], zero before the launch
    double* item_part;               // [n_items][DET_ITEM_SLOTS]
    double* colsum2;                 // [genes] column sums of the second column slice: a gene's two warps never share a target
};

__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// tf32 round-to-nearest (ties away) for an operand the tensor core will truncate: one integer add
__device__ __forceinline__ uint32_t tf32_bias(float x) { return __float_as_uint(x) + 0x1000u; }

// ld.shared on explicit shared-window addresses (the aligned dynamic-smem pointer has lost its address space)
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
// x != 0 ? a : b, twice with differently spelled tests: each predicate dies at its select, so sixteen of them
// never have to be parked in a bit mask across the MUFU latency
__device__ __forceinline__ float sel_nz_a(float x, float a, float b) {
    float d;
    asm("{\n\t.reg .pred q;\n\tsetp.neu.f32 q, %1, 0f00000000;\n\tselp.f32 %0, %2, %3, q;\n\t}" : "=f"(d) : "f"(x), "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ float sel_nz_b(float x, float a, float b) {
    float d;
    asm("{\n\t.reg .pred q;\n\t.reg .f32 t;\n\tabs.f32 t, %1;\n\tsetp.gtu.f32 q, t, 0f00000000;\n\tselp.f32 %0, %2, %3, q;\n\t}"
        : "=f"(d) : "f"(x), "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ float is_zero_f(float x) {          // 1.0f where x == 0, else 0.0f (one FSET)
    float d;
    asm("set.eq.f32.f32 %0, %1, 0f00000000;" : "=f"(d) : "f"(x));
    return d;
}
__device__ __forceinline__ void kahan_add(float& s, float& c, float v) {
    const float y = v - c;
    const float u = s + y;
    c = (u - s) - y;
    s = u;
}

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

// Walks the tiles of the work items of this CTA pair: item = chunk * n_own_units + own_unit (chunk-major, so
// that the CTAs running at the same time sweep the same chunk and share its operands in L2).  The two CTAs of a
// cluster walk the same items; CTA `rank` owns own tile 2 * own_unit + rank.
struct TileIter {
    int item, stride, t, t_begin, t_end, own0, ncta, rank;
    __device__ __forceinline__ void load(const TcArgs& a) {
        if (item < a.n_items) {
            const int chunk = item / a.n_own_units, own_unit = item - chunk * a.n_own_units;
            own0 = (own_unit * ncta + rank) * TC_OWN;
            t_begin = chunk * a.tiles_per_chunk;
            t_end = min(t_begin + a.tiles_per_chunk, a.n_sw_tiles);
            t = t_begin;
        }
    }
    __device__ __forceinline__ void init(const TcArgs& a, int ncta_, int rank_) {
        ncta = ncta_; rank = rank_;
        item = blockIdx.x / ncta; stride = gridDim.x / ncta;
        load(a);
    }
    __device__ __forceinline__ bool valid(const TcArgs& a) const { return item < a.n_items; }
    __device__ __forceinline__ bool first() const { return t == t_begin; }
    __device__ __forceinline__ bool last() const { return t == t_end - 1; }
    __device__ __forceinline__ void next(const TcArgs& a) {
        if (++t >= t_end) { item += stride; load(a); }
    }
};

// UFL: underflow-emulation hooks (TcArgs::thr_*).  A separate instantiation: two more live registers in the element-wise
// loop cost the plain kernels 7 % (row pass) / 3 % (gene pass) when the hooks were runtime-switched.
// DET: the ORI_F_DETERMINISTIC epilogue (TcArgs::tickets / item_part), a separate instantiation for the same reason (runtime-
// switched it cost the plain kernels 2.6 % / 3.4 %).
template <bool GENES, bool DROPOUT, bool ELBO, int KP, bool PRECISE, bool DEVI = false, bool UFL = false, bool DET = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_pass(const __grid_constant__ TcMaps maps, const TcArgs a)
{
    using C = Cfg<KP, PRECISE, DEVI>;
    static_assert(!DEVI || (!GENES && DROPOUT && !ELBO && !PRECISE), "deviance pass: row orientation, two contractions");
    constexpr int SW = C::SW, NS = C::NS;
    constexpr uint32_t TM_UV = C::TM_UV;
    constexpr int KST = C::KST, TST = C::TST, XST = C::XST;
    constexpr uint32_t K_STAGE = C::K_STAGE, T_STAGE = C::T_STAGE, X_STAGE = C::X_STAGE, LP_STAGE = C::LP_STAGE;
    constexpr uint32_t OFF_K = C::OFF_K, OFF_T = C::OFF_T, OFF_X = C::OFF_X, OFF_LP = C::OFF_LP, OFF_BAR = C::OFF_BAR;
    constexpr uint32_t TM_STAGE = C::TM_STAGE, TM_ACC = C::TM_ACC, TM_A = C::TM_A, TM_COLS = C::TM_COLS;
    constexpr int B_KFULL = C::B_KFULL, B_KEMPTY = C::B_KEMPTY, B_TFULL = C::B_TFULL, B_TEMPTY = C::B_TEMPTY,
                  B_XFULL = C::B_XFULL, B_XEMPTY = C::B_XEMPTY, B_SREADY = C::B_SREADY, B_PREADY = C::B_PREADY,
                  B_ACC_READY = C::B_ACC_READY, B_ACC_FREE = C::B_ACC_FREE, B_A_READY = C::B_A_READY, NBARS = C::NBARS;
    constexpr int CW = SW / 2;                // tile columns per element-wise warp: 32 or 16
    constexpr int G = CW / 16;                // groups of 16 columns per tile for one warp
    constexpr int NQ = DROPOUT ? 4 : 2;       // K-major operand arrays in use
    constexpr int NT = DROPOUT ? 2 : 1;       // transposed operand arrays in use
    const int rank = (int)cluster_ctarank();  // CTA of the pair; rank 0 leads (issues every MMA)

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + OFF_BAR);
    uint32_t* tmem_slot = (uint32_t*)(bars + NBARS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < KST; ++s) { mbar_init(&bars[B_KFULL + s], 1); mbar_init(&bars[B_KEMPTY + s], 1); }
        for (int s = 0; s < TST; ++s) { mbar_init(&bars[B_TFULL + s], 1); mbar_init(&bars[B_TEMPTY + s], 1); }
        for (int s = 0; s < XST; ++s) { mbar_init(&bars[B_XFULL + s], 1); mbar_init(&bars[B_XEMPTY + s], NEW); }
        for (int s = 0; s < NS; ++s) { mbar_init(&bars[B_SREADY + s], 1); mbar_init(&bars[B_PREADY + s], NEW * NCTA); }
        mbar_init(&bars[B_ACC_READY], 1);
        mbar_init(&bars[B_ACC_FREE], NEW * NCTA);
        mbar_init(&bars[B_A_READY], NEW * NCTA);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc_pair(tmem_slot, TM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                    // both CTAs' barriers are initialised before any remote arrive / TMA credit
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ============================================ TMA producer ============================================
        // The whole warp walks the rings (warp-uniform control flow keeps every TMA operand in uniform
        // registers); one elected lane issues.
        if (elect_one()) { tma_prefetch_desc(&maps.swK); tma_prefetch_desc(&maps.swT); tma_prefetch_desc(&maps.X); }
        // Issue order K(j), X(j), T(j-1): the order in which the stages are released in steady state (the K stage
        // when S(j-2) has run, the X stage when the element-wise warps are done with tile j-3, the T stage when
        // P(j-3) has run), so the blocking waits below never hold back a load whose stage is already free.
        TileIter ik, it_;
        ik.init(a, NCTA, rank); it_.init(a, NCTA, rank);
        uint32_t nk = 0, nt = 0;
        auto load_T = [&]() {
            if (DEVI) { ++nt; it_.next(a); return; }       // no accumulating contraction: no transposed operands
            const uint32_t s = nt % TST;
            mbar_wait(&bars[B_TEMPTY + s], ((nt / TST) & 1) ^ 1, 12);
            if (elect_one()) {
                uint8_t* st = smem + OFF_T + s * T_STAGE;
                uint64_t* bar = &bars[B_TFULL + s];
                const int sw0 = it_.t * SW;
                constexpr int NTP = PRECISE ? 2 : 1;                            // + the bf16 [lo | hi] pairs of each array
                if (rank == 0) mbar_expect_tx(bar, NTP * NT * C::T_ARR * NCTA);       // the whole pair's bytes land on the leader's barrier
#pragma unroll
                for (int h = 0; h < NTP; ++h)
#pragma unroll
                    for (int q0 = 0; q0 < NT; ++q0)
#pragma unroll
                        for (int c = 0; c < SW / 32; ++c) {
                            const int q = 2 * h + q0;                               // slot in the stage = array in global memory
                            uint8_t* dst = st + q * C::T_ARR + c * C::T_CHUNK;
                            const int row = q * KP + (KP / NCTA) * rank;            // this CTA's latent rows of array q
                            tma_load_2d_pair(dst, &maps.swT, bar, sw0 + 32 * c, row, L2_EVICT_LAST);
                        }
            }
            __syncwarp();
            ++nt; it_.next(a);
        };
        while (ik.valid(a)) {
            {
                const uint32_t s = nk % KST;
                mbar_wait(&bars[B_KEMPTY + s], ((nk / KST) & 1) ^ 1, 10);
                if (elect_one()) {
                    uint8_t* st = smem + OFF_K + s * K_STAGE;
                    uint64_t* bar = &bars[B_KFULL + s];
                    const int sw0 = ik.t * SW;
                    if (rank == 0) mbar_expect_tx(bar, NQ * C::K_ARR * NCTA);
#pragma unroll
                    for (int q = 0; q < NQ; ++q)
#pragma unroll
                        for (int kb = 0; kb < C::KB; ++kb) {
                            uint8_t* dst = st + q * C::K_ARR + kb * C::K_BLK;
                            const int row = (int)(q * a.sw_pad + sw0 + (SW / NCTA) * rank);   // this CTA's sweep rows
                            tma_load_2d_pair(dst, &maps.swK, bar, 32 * kb, row, L2_EVICT_LAST);
                        }
                }
                __syncwarp();
            }
            {
                const uint32_t s = nk % XST;
                mbar_wait(&bars[B_XEMPTY + s], ((nk / XST) & 1) ^ 1, 11);
                if (elect_one()) {
                    uint8_t* st = smem + OFF_X + s * X_STAGE;
                    uint64_t* bar = &bars[B_XFULL + s];
                    const int sw0 = ik.t * SW;
                    mbar_expect_tx(bar, X_STAGE + ((!GENES && DROPOUT) ? LP_STAGE : 0));
                    if (DEVI) bulk_load(smem + OFF_LP + s * LP_STAGE, a.devlp + (long long)ik.t * (8 * SW), LP_STAGE, bar);
                    if (!GENES) {          // [128 cells][32 genes] boxes
#pragma unroll
                        for (int c = 0; c < SW / 32; ++c)
                            tma_load_2d_hint(st + c * (TC_OWN * 128), &maps.X, bar, sw0 + 32 * c, ik.own0, L2_EVICT_FIRST);
                        if (DROPOUT && !DEVI) {
                            bulk_load(smem + OFF_LP + s * LP_STAGE, a.lp2w + sw0, SW * 4, bar);
                            bulk_load(smem + OFF_LP + s * LP_STAGE + SW * 4, a.flw + sw0, SW * 4, bar);
                            bulk_load(smem + OFF_LP + s * LP_STAGE + SW * 8, a.cw + sw0, SW * 4, bar);
                        }
                    } else {               // [SW cells][32 genes] boxes, one per TMEM lane quarter
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            tma_load_2d_hint(st + c * (SW * 128), &maps.X, bar, ik.own0 + 32 * c, sw0, L2_EVICT_FIRST);
                    }
                }
                __syncwarp();
            }
            if (nk > 0) load_T();
            ++nk; ik.next(a);
        }
        if (nk > 0) load_T();
    } else if (warp == 1 || false) {      // `|| false` (and the mma / commit lambdas below) only fix the block layout
                                          // nvcc picks: written plainly, some instances compile to a different schedule
        // ============================================ MMA issuer ============================================
        // Warp-uniform control flow, one elected lane issues: descriptors and TMEM addresses stay in uniform
        // registers (a divergent single-lane loop makes the compiler wrap every tcgen05.mma in a
        // register->uniform-register broadcast loop, which throttles the issue rate).
        // Only the leader CTA issues: cta_group::2 MMAs of M = 256 span both CTAs' TMEM and read each CTA's half
        // of the B tile; completion is multicast to the barriers of both CTAs.
        if (rank == 0) {
            constexpr uint32_t idescS = make_idesc_tf32(TC_OWN * NCTA, SW, false, false);
            constexpr uint32_t idescP = make_idesc_tf32(TC_OWN * NCTA, KP, false, false);
            constexpr uint32_t idescS16 = make_idesc_bf16(TC_OWN * NCTA, SW);
            const uint32_t sbase = smem_u32(smem);
            const uint64_t kdesc0 = make_smem_desc(sbase + OFF_K, 16, 1024);
            const uint64_t tdesc0 = make_smem_desc(sbase + OFF_T, 16, 1024);
            auto mma = [&](uint32_t d, uint32_t at, uint64_t bd, uint32_t idesc, bool acc) {
                mma_tf32_ts_pair(d, at, bd, idesc, acc);
            };
            auto mma16 = [&](uint32_t d, uint32_t at, uint64_t bd, uint32_t idesc, bool acc) {
                mma_bf16_ts_pair(d, at, bd, idesc, acc);
            };
            auto commit = [&](uint64_t* bar) { tc_commit_pair(bar); };
            auto issue_P = [&](uint32_t it, bool first, bool last, int li) {
                const uint32_t s = it % NS, ts = it % TST;
                mbar_wait(&bars[B_PREADY + s], (it / NS) & 1, 20);
                mbar_wait(&bars[B_TFULL + ts], (it / TST) & 1, 24);
                if (first) mbar_wait(&bars[B_ACC_FREE], (li & 1) ^ 1, 21);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t td = tdesc0 + (uint64_t)((ts * T_STAGE) >> 4);
                    // contraction over the SW sweep entries of the tile, 8 per MMA: chunk ks / 4, 32 bytes per step
                    // the two accumulators are independent chains: issued alternately, so that an MMA never has to wait
                    // for the write-back of the one just before it (dependent MMAs of N <= 64 cost their latency, not
                    // their throughput)
#pragma unroll
                    for (int ks = 0; ks < SW / 8; ++ks) {
                        mma(tmem + TM_ACC, tmem + s * TM_STAGE + ks * 8,
                            td + (uint64_t)(((ks >> 2) * C::T_CHUNK + (ks & 3) * 32) >> 4), idescP, !(first && ks == 0));
                        if (DROPOUT)
                            mma(tmem + TM_ACC + KP, tmem + s * TM_STAGE + TM_UV + ks * 8,
                                td + (uint64_t)((C::T_ARR + (ks >> 2) * C::T_CHUNK + (ks & 3) * 32) >> 4), idescP,
                                !(first && ks == 0));
                    }
                    if (PRECISE) {
                        // cross terms hi.lo + lo.hi of both accumulations: A = the bf16 pairs [hi | lo] of R / D beside them in
                        // TMEM (SW words = 2 SW bf16), B = the bf16 pairs [lo | hi] of the transposed operands (slots 2, 3)
                        constexpr uint32_t idescP16 = make_idesc_bf16(TC_OWN * NCTA, KP);
#pragma unroll
                        for (int ks = 0; ks < SW / 8; ++ks) {
                            mma16(tmem + TM_ACC, tmem + s * TM_STAGE + SW + ks * 8,
                                  td + (uint64_t)((2 * C::T_ARR + (ks >> 2) * C::T_CHUNK + (ks & 3) * 32) >> 4), idescP16, true);
                            if (DROPOUT)
                                mma16(tmem + TM_ACC + KP, tmem + s * TM_STAGE + TM_UV + SW + ks * 8,
                                      td + (uint64_t)((3 * C::T_ARR + (ks >> 2) * C::T_CHUNK + (ks & 3) * 32) >> 4), idescP16, true);
                        }
                    }
                    commit(&bars[B_TEMPTY + ts]);
                    if (last) commit(&bars[B_ACC_READY]);
                }
                __syncwarp();
            };
            // S runs NS - 1 tiles ahead of P: S(it) overwrites the TMEM stage P(it - NS) has read (the tensor pipe executes in
            // issue order), so each loop iteration issues S(it) and then P(it - (NS - 1)); `tp` trails `ti` for the latter
            TileIter ti, tp;
            ti.init(a, NCTA, rank); tp.init(a, NCTA, rank);
            uint32_t it = 0, itp = 0;
            int li = 0, lip = 0;
            auto trail_P = [&]() {
                const bool pl = tp.last();
                if (DEVI) {     // nothing to accumulate: only wait until the element-wise warps have read the stage S will reuse
                    mbar_wait(&bars[B_PREADY + itp % NS], (itp / NS) & 1, 20);
                } else
                issue_P(itp, tp.first(), pl, lip);
                if (pl) ++lip;
                ++itp; tp.next(a);
            };
            while (ti.valid(a)) {
                const uint32_t s = it % NS, ks_ = it % KST;
                const bool first = ti.first(), last = ti.last();
                mbar_wait(&bars[B_KFULL + ks_], (it / KST) & 1, 23);
                if (first) mbar_wait(&bars[B_A_READY], li & 1, 22);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t kd = kdesc0 + (uint64_t)((ks_ * K_STAGE) >> 4);
                    // den (and uv) of this tile: hi.hi in tf32, A operand from TMEM; contraction over the KP latent
                    // components, 8 per MMA: K block kk / 4, 32 bytes per step
#define ORI_CHAIN(D_, Q)                                                                                          \
                    _Pragma("unroll") for (int kk = 0; kk < KP / 8; ++kk)                                         \
                        mma((D_), tmem + TM_A + (Q) * KP + kk * 8,                                                \
                            kd + (uint64_t)(((Q) * C::K_ARR + (kk >> 2) * C::K_BLK + (kk & 3) * 32) >> 4), idescS, kk != 0)
                    // arrays 1 and 3 hold bf16 pairs: own side [hi | lo], sweep side [lo | hi] (2 KP elements, the
                    // same bytes and the same 8-column / 32-byte steps as a tf32 array)
#define ORI_CHAIN16(D_, Q)                                                                                        \
                    _Pragma("unroll") for (int kk = 0; kk < KP / 8; ++kk)                                         \
                        mma16((D_), tmem + TM_A + (Q) * KP + kk * 8,                                              \
                              kd + (uint64_t)(((Q) * C::K_ARR + (kk >> 2) * C::K_BLK + (kk & 3) * 32) >> 4), idescS16, true)
                    ORI_CHAIN(tmem + s * TM_STAGE, 0);
                    ORI_CHAIN16(tmem + s * TM_STAGE, 1);
                    if (DROPOUT) {
                        ORI_CHAIN(tmem + s * TM_STAGE + TM_UV, 2);
                        ORI_CHAIN16(tmem + s * TM_STAGE + TM_UV, 3);
                    }
#undef ORI_CHAIN16
#undef ORI_CHAIN
                    commit(&bars[B_SREADY + s]);
                    commit(&bars[B_KEMPTY + ks_]);
                }
                __syncwarp();
                if (it >= (uint32_t)(NS - 1)) trail_P();
                if (last) ++li;
                ++it;
                ti.next(a);
            }
            while (itp < it) trail_P();
        }
    } else {
        // ======================================= element-wise stage + epilogue =================================
        const int ew = warp - 2;
        const int quarter = warp & 3;                 // TMEM lane quarter this warp may touch
        // slice: which half of the tile's columns, and which own-side array and accumulator
        // (0: exp(E log .) and accumulator 1; 1: E[.] and accumulator 2)
        const int slice = ew >> 2;
        const int lrow = quarter * 32 + lane;         // own index inside the tile = TMEM lane
        const int colbase = slice * CW;
        const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16);
        const uint32_t sbase = smem_u32(smem);
        const bool any_floor = DROPOUT && (*a.any_floor != 0);

        // own-side operands of one work item -> TMEM: slice 0 writes hi / lo of exp(E log .), slice 1 (dropout only)
        // hi / lo of E[.], for this warp's 32 lanes, 16 latent components at a time
        auto a_load_store = [&](int own0) {
            if (slice * 2 < NQ) {
                const long long idx = (long long)own0 + lrow;
                const float* src = (slice ? a.own_E : a.own_e) + idx * KP;
                const bool ok = idx < a.own_total;
                const bool scale = GENES && slice;                 // uv is kept in log2 units: V_hat side * log2(e)
#pragma unroll
                for (int c16 = 0; c16 < KP / 16; ++c16) {
                    float av[16];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 v = ok ? __ldg(reinterpret_cast<const float4*>(src + 16 * c16) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                        av[4 * c] = v.x; av[4 * c + 1] = v.y; av[4 * c + 2] = v.z; av[4 * c + 3] = v.w;
                    }
                    uint32_t whi[16], wlo[16];
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const float v = scale ? av[e] * LOG2E : av[e];
                        const float hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
                        whi[e] = __float_as_uint(hi);
                        wlo[e] = __float_as_uint(v - hi);
                    }
                    tmem_st16(tlane + TM_A + (2 * slice) * KP + 16 * c16, whi);
                    // cross-term operand [hi | lo] as bf16 pairs: these 16 components -> 8 + 8 columns
                    uint32_t phi[8], plo[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        phi[e] = pack_bf16x2(__uint_as_float(whi[2 * e]), __uint_as_float(whi[2 * e + 1]));
                        plo[e] = pack_bf16x2(__uint_as_float(wlo[2 * e]), __uint_as_float(wlo[2 * e + 1]));
                    }
                    tmem_st8(tlane + TM_A + (2 * slice + 1) * KP + 8 * c16, phi);
                    tmem_st8(tlane + TM_A + (2 * slice + 1) * KP + KP / 2 + 8 * c16, plo);
                }
            }
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&bars[B_A_READY], 0);
        };

        // gene pass: X is staged [cell][gene]; lane (gene) reads one float per cell, 128-byte swizzle undone here
        uint32_t xoff[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) xoff[k] = (uint32_t)(quarter * (SW * 128) + ((((lane >> 2) ^ k)) << 4) + (lane & 3) * 4);

        TileIter ti;
        ti.init(a, NCTA, rank);
        uint32_t it = 0;                              // tiles of this CTA so far: TMEM stage it & 1, X stage it % XST
        int li = 0;
        if (ti.valid(a)) a_load_store(ti.own0);
        while (ti.valid(a)) {
            const long long own_idx = (long long)ti.own0 + lrow;
            const bool own_ok = own_idx < a.own_total;
            const int next_item = ti.item + ti.stride;
            const bool has_next = next_item < a.n_items;
            const int next_own0 = ((next_item % a.n_own_units) * NCTA + rank) * TC_OWN;
            float lp2j = 0.f, flj = 0.f, cj = 0.f, ulim = 127.f;
            if (GENES && DROPOUT) {                   // padded arrays: always in range
                lp2j = a.lp2w[own_idx]; flj = a.flw[own_idx];
                cj = ex2_approx(-lp2j);               // (1 - pi) / pi
                ulim = fminf(127.f, 127.f + lp2j);    // uv * log2(e) beyond this: D_hat = 0 either way
            }
            // pi_j = 1 (a gene without a single zero, logit = +inf): every entry has D_hat = 1 and contributes
            // (1 - D) * e2 = 0 * -inf to the entropy sum; a finite stand-in keeps that product at 0
            const float lp2f = fminf(lp2j, 3.0e38f);
            // underflow emulation: this row's threshold factor and the bound under which a denominator needs the exact test
            float thr_o = 0.f, den_lim = 0.f;             // compile-time zeros without UFL
            if constexpr (UFL) {
                thr_o = own_ok ? a.thr_own[own_idx] : 0.f;
                den_lim = thr_o * __ldg(a.thr_sw_max);
                den_lim = den_lim == den_lim ? fminf(den_lim, 3.0e38f) : 0.f;
            }
            // genes / columns with a floor (pi <= 0, zigap.py:133) or with the initial indicator state (logit pi = -inf,
            // zigap.py:77) take the general path
            const bool slow_item = DROPOUT && (GENES ? (__any_sync(0xffffffffu, flj != 0.f || lp2j == -INFINITY) != 0) : any_floor);
            float cs = 0.f;
            float xl_s = 0.f, xl_c = 0.f, ent_s = 0.f, ent_c = 0.f;     // compensated fp32 sums over the item
            const int t_end = ti.t_end;
            // ---- tiles of the item.  Two register buffers of 16 columns are in flight per warp.
            uint32_t dr[2][16], ur[2][16];
            float x[2][16];
            struct Tile { uint32_t xs_addr, lp_addr, tden, s, xs; int valid; bool slow; long long sw0; };
            auto tile_of = [&](uint32_t it_, int t_) {
                Tile c;
                c.s = it_ % NS; c.xs = it_ % XST;
                c.xs_addr = sbase + OFF_X + c.xs * X_STAGE;
                c.lp_addr = sbase + OFF_LP + c.xs * LP_STAGE;
                c.valid = (int)min((long long)SW, a.sw_total - (long long)t_ * SW);   // gene pass: real cells
                c.sw0 = (long long)t_ * SW;
                c.slow = slow_item || (GENES && c.valid != SW);
                c.tden = tlane + c.s * TM_STAGE;                                      // uv / D_hat: + TM_UV
                return c;
            };
            // X tile (and lp) visible to this thread; den / uv complete in TMEM
            auto wait_tile = [&](uint32_t it_) {
                const uint32_t s = it_ % NS, sph = (it_ / NS) & 1, xs = it_ % XST, xph = (it_ / XST) & 1;
                mbar_wait2(&bars[B_XFULL + xs], xph, &bars[B_SREADY + s], sph, 30);
                tc_fence_after();
            };
            auto ld_group = [&](const Tile& c, int g, int b) {
                tmem_ld16(c.tden + colbase + g * 16, dr[b]);
                if (DROPOUT) tmem_ld16(c.tden + TM_UV + colbase + g * 16, ur[b]);
            };
            // PRECISE: v -> tf32 hi (written where the MMA reads R / D) and the bf16 pairs of (hi, lo) of two neighbouring
            // entries (written beside them): words 0..7 of a group = hi pairs, pk[8..15] = lo pairs
            uint32_t pkr_h[8], pkr_l[8], pkd_h[8], pkd_l[8];
            auto split_store = [&](uint32_t (&w)[16], uint32_t (&ph)[8], uint32_t (&pl)[8]) {
#pragma unroll
                for (int e = 0; e < 16; e += 2) {
                    const float v0 = __uint_as_float(w[e]), v1 = __uint_as_float(w[e + 1]);
                    const float h0 = __uint_as_float((w[e] + 0x1000u) & 0xffffe000u), h1 = __uint_as_float((w[e + 1] + 0x1000u) & 0xffffe000u);
                    w[e] = __float_as_uint(h0); w[e + 1] = __float_as_uint(h1);
                    ph[e >> 1] = pack_bf16x2(h0, h1);
                    pl[e >> 1] = pack_bf16x2(v0 - h0, v1 - h1);
                }
            };
            auto load_x = [&](const Tile& c, int g, int b) {
                const int c0 = colbase + g * 16;
                if (!GENES) {
                    const uint32_t base = c.xs_addr + (c0 >> 5) * (TC_OWN * 128) + lrow * 128;
                    const int cb = (c0 & 31) >> 2;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 v = lds128(base + (((cb + q) ^ (lrow & 7)) << 4));
                        x[b][4 * q] = v.x; x[b][4 * q + 1] = v.y; x[b][4 * q + 2] = v.z; x[b][4 * q + 3] = v.w;
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int i = c0 + e;
                        x[b][e] = lds32(c.xs_addr + xoff[i & 7] + i * 128);
                    }
                }
            };
            // general path: den guard, floors, ragged last tile (zigap.py:90, :133); rare
            auto slow_group = [&](const Tile& c, int g, int b, float& t_xl, float& t_ent) {
                const int c0 = colbase + g * 16;
                tmem_ld16(c.tden + c0, dr[b]);
                if (DROPOUT) tmem_ld16(c.tden + TM_UV + c0, ur[b]);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float den = __uint_as_float(dr[b][e]);
                    const float xe = x[b][e];
                    const bool nz = xe != 0.f;
                    // every term of the entry underflows in the reference's float32 exp: no count assigned (zigap.py:90)
                    float xr = xe;
                    if constexpr (UFL)
                        if (den_lim > 0.f && nz && (c0 + e) < c.valid && den < thr_o * __ldg(a.thr_sw + c.sw0 + c0 + e)) xr = 0.f;
                    const float dg = den > 0.f ? den : 1.f;
                    float tt = dg, e2 = 0.f, D = 1.f;
                    if (DROPOUT) {
                        const float lp2 = GENES ? lp2j : lds32(c.lp_addr + 4 * (c0 + e));
                        const float fl = GENES ? flj : lds32(c.lp_addr + SW * 4 + 4 * (c0 + e));
                        e2 = fminf(__uint_as_float(ur[b][e]) - lp2, 127.f);
                        tt = nz ? dg : 1.f + ex2_approx(e2);
                        const float r = rcp_approx(tt);
                        D = fmaxf(nz ? 1.f : r, fl);
                        dr[b][e] = PRECISE ? __float_as_uint(xr * r) : tf32_bias(xr * r);
                        ur[b][e] = PRECISE ? __float_as_uint(D) : tf32_bias(D);
                    } else {
                        const float R = xr * rcp_approx(tt);
                        dr[b][e] = PRECISE ? __float_as_uint(R) : tf32_bias(R);
                    }
                    if (GENES && (c0 + e) < c.valid) {
                        if (DROPOUT) cs += D;
                        if (ELBO) {
                            const float l2 = lg2_approx(tt);
                            t_xl = fmaf(xe, l2, t_xl);
                            if (DROPOUT && !nz) t_ent += l2 - (1.f - D) * e2;      // non-zeros: D_hat = 1, no entropy
                        }
                    }
                }
            };
            // lean path: full tile, no floors; returns the smallest denominator seen
            auto fast_group = [&](const Tile& c, int g, int b, float& g_cs, float& g_xl, float& g_ent) -> float {
                const int c0 = colbase + g * 16;
                float cc[16];
                if (DROPOUT && !GENES) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 v = lds128(c.lp_addr + SW * 8 + 4 * (c0 + 4 * q));
                        cc[4 * q] = v.x; cc[4 * q + 1] = v.y; cc[4 * q + 2] = v.z; cc[4 * q + 3] = v.w;
                    }
                }
                float dmin = 1.f;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float den = __uint_as_float(dr[b][e]);
                    const float xe = x[b][e];
                    dmin = fminf(dmin, den);                  // den <= 0 (zigap.py:90): the group is redone below
                    float tt = den, uvp = 0.f;
                    if (DROPOUT) {
                        uvp = __uint_as_float(ur[b][e]);                          // U_hat.V_hat * log2(e)
                        if (GENES && ELBO) uvp = fminf(uvp, ulim);                // keeps 2^uv, tz and e2 finite
                        const float tz = fmaf(ex2_approx(uvp), GENES ? cj : cc[e], 1.f);   // 1 + exp(uv - logit pi)
                        tt = sel_nz_a(xe, den, tz);
                    }
                    const float r = rcp_approx(tt);
                    dr[b][e] = PRECISE ? __float_as_uint(xe * r) : tf32_bias(xe * r);   // R = X / den; 0 where X == 0
                    float D = 1.f;
                    if (DROPOUT) {
                        D = sel_nz_b(xe, 1.f, r);                                 // zigap.py:131-136
                        ur[b][e] = PRECISE ? __float_as_uint(D) : tf32_bias(D);
                    }
                    if (GENES) {
                        if (DROPOUT) g_cs += D;
                        if (ELBO) {
                            const float l2 = lg2_approx(tt);
                            g_xl = fmaf(xe, l2, g_xl);
                            if (DROPOUT) {
                                g_ent = fmaf(is_zero_f(xe), l2, g_ent);           // log2(1 + 2^e2) on zeros
                                const float e2 = uvp - lp2f;                      // <= 127 (uvp was clamped)
                                const float w = 1.f - D;                          // 0 on non-zeros
                                g_ent = fmaf(-w, e2, g_ent);
                            }
                        }
                    }
                }
                return dmin;
            };

            auto st_group = [&](const Tile& c, int g, int b) {
                const int c0 = colbase + g * 16;
                if (PRECISE) {
                    split_store(dr[b], pkr_h, pkr_l);
                    tmem_st8(c.tden + SW + (c0 >> 1), pkr_h);
                    tmem_st8(c.tden + SW + SW / 2 + (c0 >> 1), pkr_l);
                    if (DROPOUT) {
                        split_store(ur[b], pkd_h, pkd_l);
                        tmem_st8(c.tden + TM_UV + SW + (c0 >> 1), pkd_h);
                        tmem_st8(c.tden + TM_UV + SW + SW / 2 + (c0 >> 1), pkd_l);
                    }
                }
                tmem_st16(c.tden + c0, dr[b]);
                if (DROPOUT) tmem_st16(c.tden + TM_UV + c0, ur[b]);
            };
            // R / D_hat of the tile are in TMEM (after tcgen05.wait::st): P may run; the X stage may be refilled
            auto hand_off = [&](const Tile& c) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive_cluster(&bars[B_PREADY + c.s], 0);
                    mbar_arrive(&bars[B_XEMPTY + c.xs]);
                }
            };
            long long dv0 = 0, dv1 = 0, dv2 = 0;      // deviance pass: truncated log-likelihood sums of this thread and item
            if constexpr (DEVI) {
                // components of this cell's U_hat that are not exactly zero (bit k & 31): see k_tc_prep_dev
                uint32_t mU = 0;
                if (own_ok) {
                    const float* uh = a.own_E + own_idx * KP;
#pragma unroll 8
                    for (int k = 0; k < KP; ++k) if (__ldg(uh + k) != 0.f) mU |= 1u << (k & 31);
                }
                // ---- deviance pass (base.py:58-82, sparse_zigap.py:44-51): "den" = the rate L = U_hat . V_hat^T, "uv" = the
                //      contraction that generates D_hat (log2 units).  Per entry, like k_deviance's integer mode:
                //        zero, round(D_hat) = 0 (uv >= logit pi):  l_uv = 0
                //        zero, kept:   l_uv = log(pi e^-L + 1 - pi);     l_sat = 0;   l_mean = log(pi e^-mean + 1 - pi)
                //        non-zero:     l = log pi - rate + x log rate    at the rates L, x, mean
                //      every term truncated toward zero before it is summed (sparse_zigap.py:45).  float32 with a float64
                //      redo of the entries whose rate underflows or whose terms leave the exact range; nothing is written back.
                for (int t = ti.t_begin; t < t_end; ++t, ++it) {
                    const bool last = (t == t_end - 1);
                    const Tile c = tile_of(it, t);
                    wait_tile(it);
                    if (last && has_next) a_load_store(next_own0);
                    ld_group(c, 0, 0);
                    load_x(c, 0, 0);
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        const int b = g & 1;
                        const int c0 = colbase + g * 16;
                        if (g + 1 < G) load_x(c, g + 1, b ^ 1);
                        tmem_wait_ld();
                        if (g + 1 < G) ld_group(c, g + 1, b ^ 1);
                        int s0 = 0, s1 = 0, s2 = 0;       // <= 16 terms of magnitude < 8e6 each
                        uint32_t bad = 0;                 // entries that need the float64 redo (kept out of the unrolled code)
                        const int nvalid = (int)min((long long)16, a.sw_total - ((long long)t * SW + c0));
#pragma unroll
                        for (int e = 0; e < 16; ++e) {
                            const uint32_t ca = c.lp_addr + 32 * (c0 + e);        // 8 constants per gene (k_tc_prep_dev)
                            const float L = __uint_as_float(dr[b][e]), uvp = __uint_as_float(ur[b][e]), xe = x[b][e];
                            const float4 ga = lds128(ca), gb = lds128(ca + 16);
                            const float lp2 = ga.x, pj = ga.y, qj = ga.z, lpi = ga.w, mj = gb.x, lmj = gb.y, lm0 = gb.z;
                            const bool nz = xe != 0.f;
                            const bool kept = uvp < lp2;                           // round(D_hat) = 1 on a zero entry
                            // both branches for every lane, selected afterwards: 4 MUFU per entry, no divergence
                            const float lnL = lg2_approx(L) * LN2, lnx = lg2_approx(xe) * LN2;
                            const float z0 = lg2_approx(fmaf(pj, ex2_approx(-L * LOG2E), qj)) * LN2;
                            const float f0 = nz ? fmaf(xe, lnL, lpi - L) : (kept ? z0 : 0.f);
                            const float f1 = nz ? fmaf(xe, lnx, lpi - xe) : 0.f;
                            const float f2 = nz ? fmaf(xe, lmj, lpi - mj) : lm0;
                            const bool ok = (!nz || L >= 1e-30f) && fmaxf(fmaxf(fabsf(f0), fabsf(f1)), fabsf(f2)) < 8e6f;
                            const bool live = own_ok && e < nvalid;
                            if (live && ok) { s0 += (int)f0; s1 += (int)f1; s2 += (int)f2; }
                            if (live && !ok) bad |= 1u << e;
                        }
                        if (__any_sync(0xffffffffu, bad != 0)) {
                            // rare: the float32 rate underflowed under an observed count (the reference's float64 product does
                            // not), or a term is huge / not finite: float64 from the parameters, numpy's cast rules
                            float xs_[16], us_[16];
#pragma unroll
                            for (int e = 0; e < 16; ++e) { xs_[e] = x[b][e]; us_[e] = __uint_as_float(ur[b][e]); }
#pragma unroll 1
                            for (int e = 0; e < 16; ++e) {
                                if (!((bad >> e) & 1u)) continue;
                                const long long j = (long long)t * SW + c0 + e;
                                const uint32_t ca = c.lp_addr + 32 * (c0 + e);
                                const float4 ga = lds128(ca), gb = lds128(ca + 16);
                                const float xe = xs_[e], uvp = us_[e];
                                const bool nz = xe != 0.f, kept = uvp < ga.x;
                                // every product U_hat_ik V_hat_jk is exactly zero (a masked gene of the sparse model, mostly): the
                                // float64 rate is 0 and the term of the observed count -inf, which the reference's int64 buffer
                                // holds as INT64_MIN (trunc64 below gives the same); the other two sums as on the fast path
                                if (nz && (mU & __float_as_uint(gb.w)) == 0u) {
                                    const float g1 = fmaf(xe, lg2_approx(xe) * LN2, ga.w - xe), g2 = fmaf(xe, gb.y, ga.w - gb.x);
                                    if (fmaxf(fabsf(g1), fabsf(g2)) < 8e6f) {
                                        dv0 = (long long)((unsigned long long)dv0 + 0x8000000000000000ull);
                                        dv1 += (int)g1; dv2 += (int)g2;
                                        continue;
                                    }
                                }
                                double Ld = 0.0;
                                const float* uh = a.own_E + own_idx * KP;
                                for (int k = 0; k < KP; ++k) {
                                    const long long gk = j * KP + k;
                                    if (a.dev_b2[gk] != 0.f)
                                        Ld = fma((double)uh[k], (double)a.dev_b1[gk] / (double)a.dev_b2[gk] * (a.dev_ps ? (double)a.dev_ps[gk] : 1.0), Ld);
                                }
                                const double xd = (double)xe;
                                double l0, l1, l2;
                                if (nz) {
                                    l0 = (double)ga.w - Ld + xd * log(Ld);
                                    l1 = (double)ga.w - xd + xd * log(xd);
                                    l2 = (double)ga.w - (double)gb.x + xd * (double)gb.y;
                                } else {
                                    l0 = kept ? (double)logf(fmaf(ga.y, expf(-(float)Ld), ga.z)) : 0.0;
                                    l1 = 0.0;
                                    l2 = (double)gb.z;
                                }
                                auto trunc64 = [](double v) -> long long {
                                    return (fabs(v) < 9.2233720368547758e18) ? (long long)v : (long long)0x8000000000000000ull;
                                };
                                dv0 += trunc64(l0); dv1 += trunc64(l1); dv2 += trunc64(l2);
                            }
                        }
                        dv0 += s0; dv1 += s1; dv2 += s2;
                    }
                    hand_off(c);
                }
            } else {
                // ---- every warp owns G groups of the tile; the next group's loads fly during the current one;
                //      the tile is handed to the MMA warp as soon as its last group is stored
                for (int t = ti.t_begin; t < t_end; ++t, ++it) {
                    const bool last = (t == t_end - 1);
                    const Tile c = tile_of(it, t);
                    wait_tile(it);
                    if (last && has_next) a_load_store(next_own0);   // every S of this item has completed: A can be replaced
                    if (!c.slow) ld_group(c, 0, 0);
                    load_x(c, 0, 0);
                    float t_xl = 0.f, t_ent = 0.f;
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        const int b = g & 1;
                        bool redo = c.slow;
                        if (g + 1 < G) load_x(c, g + 1, b ^ 1);
                        if (!c.slow) {
                            tmem_wait_ld();
                            if (g + 1 < G) ld_group(c, g + 1, b ^ 1);
                            float g_cs = 0.f, g_xl = 0.f, g_ent = 0.f;
                            const float dmin = fast_group(c, g, b, g_cs, g_xl, g_ent);
                            redo = __any_sync(0xffffffffu, dmin <= den_lim) != 0;
                            if (GENES && !redo) { cs += g_cs; t_xl += g_xl; t_ent += g_ent; }
                        }
                        if (redo) slow_group(c, g, b, t_xl, t_ent);
                        st_group(c, g, b);
                    }
                    if (GENES && ELBO) { kahan_add(xl_s, xl_c, t_xl); if (DROPOUT) kahan_add(ent_s, ent_c, t_ent); }
                    tmem_wait_st();
                    hand_off(c);
                }
            }
            if constexpr (DEVI) {
                unsigned long long r0 = (unsigned long long)dv0, r1 = (unsigned long long)dv1, r2 = (unsigned long long)dv2;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    r0 += __shfl_xor_sync(0xffffffffu, r0, o); r1 += __shfl_xor_sync(0xffffffffu, r1, o);
                    r2 += __shfl_xor_sync(0xffffffffu, r2, o);
                }
                if (lane == 0) {
                    if (r0) atomicAdd(a.dev_out, r0);
                    if (r1) atomicAdd(a.dev_out + 1, r1);
                    if (r2) atomicAdd(a.dev_out + 2, r2);
                }
                ++li;
                ti.item += ti.stride;
                ti.load(a);
                continue;
            }
            double acc_xl = (double)xl_s - (double)xl_c, acc_ent = (double)ent_s - (double)ent_c;
            // ---- epilogue of the work item: accumulators -> global (atomics: the sweep of one own tile is split);
            //      slice 0 drains acc1, slice 1 acc2
            mbar_wait(&bars[B_ACC_READY], li & 1, 32);
            tc_fence_after();
            const int det_tile = ti.own0 / TC_OWN;
            if (DET && a.tickets) {          // wait until every warp of the previous chunk item of this own tile has added its sums
                const int want = (ti.item / a.n_own_units) * NEW;
                if (lane == 0) {
                    volatile int* tk = a.tickets + det_tile;
                    while (*tk < want) __nanosleep(200);
                }
                __syncwarp();
                __threadfence();
            }
            if (slice == 0 || DROPOUT) {
                float* out = (slice == 0 ? a.acc1 : a.acc2) + own_idx * KP;
#pragma unroll
                for (int g = 0; g < KP / 16; ++g) {
                    uint32_t v[16];
                    tmem_ld16(tlane + TM_ACC + slice * KP + g * 16, v);
                    tmem_wait_ld();
                    if (own_ok) {
#pragma unroll
                        for (int e = 0; e < 16; ++e) atomicAdd(out + g * 16 + e, __uint_as_float(v[e]));
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&bars[B_ACC_FREE], 0);
            if (GENES) {
                if (DROPOUT && own_ok) atomicAdd(((DET && slice) ? a.colsum2 : a.colsum) + own_idx, (double)cs);
                if (ELBO) {
                    if (!own_ok) { acc_xl = 0.0; acc_ent = 0.0; }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        acc_xl += __shfl_xor_sync(0xffffffffu, acc_xl, o);
                        acc_ent += __shfl_xor_sync(0xffffffffu, acc_ent, o);
                    }
                    if (lane == 0) {
                        if (DET && a.item_part) {
                            double* slot = a.item_part + ((long long)ti.item * DET_ITEM_SLOTS + (rank * NEW + ew) * 2);
                            slot[0] = acc_xl * (double)LN2;
                            slot[1] = DROPOUT ? acc_ent * (double)LN2 : 0.0;
                        } else {
                            atomicAdd(a.part64 + R64_XLOGDEN, acc_xl * (double)LN2);
                            if (DROPOUT) atomicAdd(a.part64 + R64_ENT, acc_ent * (double)LN2);
                        }
                    }
                }
            }
            if (DET && a.tickets) {          // this warp's sums are in: let the next chunk item of the tile proceed
                __threadfence();
                __syncwarp();
                if (lane == 0) atomicAdd(a.tickets + det_tile, 1);
            }
            ++li;
            ti.item += ti.stride;
            ti.load(a);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                    // the leader's MMAs read the peer's shared memory and TMEM until the very end
    if (warp == 1) tmem_dealloc_pair(tmem, TM_COLS);
}

// ---- operand preparation -------------------------------------------------------------------------------------
// K-major operand arrays: out[q][pad][KP], q = 0: hi(e) 1: bf16 pairs of lo(e) | hi(e) 2: hi(E) 3: the same pairs of E;
// hi = tf32 round-to-nearest (the tensor core truncates fp32 operands to tf32: scripts/tc_probe.cu T4), lo = x - hi.
// Pad rows are zero.
__global__ void __launch_bounds__(256)
k_tc_prep_K(const float* __restrict__ e, const float* __restrict__ E, float Escale, float* __restrict__ out, long long n,
            long long pad, int KP)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= pad * KP) return;
    const bool ok = idx < n * KP;
    const float v = ok ? e[idx] : 0.f;
    const float hv = to_tf32_rna(v);
    out[idx] = hv;
    // arrays 1 and 3: row i = 2 KP bf16 [lo(0..KP-1) | hi(0..KP-1)], i.e. KP 32-bit words; this thread writes word w
    const long long i = idx / KP;
    const int w = (int)(idx - i * KP), half = KP / 2;
    const int k0 = 2 * (w < half ? w : w - half);
    auto word = [&](const float* src, float scale) -> uint32_t {
        const float a = ok ? src[i * KP + k0] * scale : 0.f, b = ok ? src[i * KP + k0 + 1] * scale : 0.f;
        const float ha = to_tf32_rna(a), hb = to_tf32_rna(b);
        return w < half ? pack_bf16x2(a - ha, b - hb) : pack_bf16x2(ha, hb);
    };
    reinterpret_cast<uint32_t*>(out)[pad * KP + idx] = word(e, 1.f);
    if (E) {
        const float x = ok ? E[idx] * Escale : 0.f;
        out[2 * pad * KP + idx] = to_tf32_rna(x);
        reinterpret_cast<uint32_t*>(out)[3 * pad * KP + idx] = word(E, Escale);
    }
}
// transposed operand: out[k][i] = tf32(src[i][k]),  src [n x KP], out [KP x pad]; grid (pad / 32, KP / 32).
// out16 (PRECISE, else NULL): the bf16 pairs [lo | hi] of the same values, 32 words per block of 32 sweep entries:
// word w < 16 = (lo[2w], lo[2w+1]), word w >= 16 = (hi[2(w-16)], hi[2(w-16)+1]); hi = tf32 round-to-nearest, lo = v - hi
__global__ void __launch_bounds__(256)
k_tc_prep_T(const float* __restrict__ src, float* __restrict__ out, uint32_t* __restrict__ out16, long long n, long long pad, int KP)
{
    __shared__ float tile[32][33];
    const long long i0 = (long long)blockIdx.x * 32;
    const int k0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const long long i = i0 + r;
        tile[r][threadIdx.x] = i < n ? src[i * KP + k0 + threadIdx.x] : 0.f;
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += 8) {
        const long long i = i0 + threadIdx.x;
        if (i < pad) {
            out[(long long)(k0 + k) * pad + i] = to_tf32_rna(tile[threadIdx.x][k]);
            if (out16) {
                const int w = threadIdx.x, e = 2 * (w & 15);
                const float a = tile[e][k], b = tile[e + 1][k];
                const float ha = to_tf32_rna(a), hb = to_tf32_rna(b);
                out16[(long long)(k0 + k) * pad + i] = w < 16 ? pack_bf16x2(a - ha, b - hb) : pack_bf16x2(ha, hb);
            }
        }
    }
}
__global__ void k_tc_prep_lp(const float* __restrict__ lp, const float* __restrict__ fl, float* __restrict__ lp2w,
                             float* __restrict__ flw, float* __restrict__ cw, int* __restrict__ any_floor, int p, int pad)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= pad) return;
    const float f = j < p ? fl[j] : 0.f;
    const float l2 = j < p ? lp[j] * LOG2E : -INFINITY;
    lp2w[j] = l2;
    flw[j] = f;
    cw[j] = exp2f(-l2);
    if (f != 0.f) *any_floor = 1;
}

// largest underflow threshold of a side (non-negative floats order like their bit patterns)
__global__ void k_tc_thr_max(const float* __restrict__ thr, long long n, int* __restrict__ out)
{
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) m = fmaxf(m, thr[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_int(m));
}

// deviance pass: 8 constants per gene, tile-major [tile][SW][8]:
//   logit(pi_gen) * log2(e) | pi | 1 - pi | log pi | mean | log mean | trunc(log(pi e^-mean + 1 - pi)) | mask
// pi = the finalised Bernoulli prior, pi_gen (through lp) the one that generated D_hat, mean = column mean of X;
// mask (bit pattern in a float slot): bit k & 31 set when component k of the gene's effective V_hat = b1 / b2 (* S_hat) is
// not exactly zero in float64 -- with the matching mask of the cell's U_hat an empty intersection means the rate is
// EXACTLY zero (masked genes of the sparse model, sparse_zigap.py:103), which the element-wise warps then know without
// the float64 redo
__global__ void k_tc_prep_dev(const float* __restrict__ lp, const double* __restrict__ pi, const double* __restrict__ cmean,
                              float* __restrict__ out, int p, int pad, const float* __restrict__ b1,
                              const float* __restrict__ b2, const float* __restrict__ ps, int KP)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= pad) return;
    float4 a = make_float4(-INFINITY, 0.5f, 0.5f, 0.f), b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < p) {
        const double pj = pi[j], mj = cmean[j];
        a.x = lp[j] * LOG2E; a.y = (float)pj; a.z = (float)(1.0 - pj); a.w = (float)log(pj);
        b.x = (float)mj; b.y = (float)log(mj);
        const float lm = logf(fmaf((float)pj, (float)exp(-mj), (float)(1.0 - pj)));     // as k_deviance's integer mode
        b.z = (float)(int)lm;
        uint32_t mask = 0;
        for (int k = 0; k < KP; ++k) {
            const long long gk = (long long)j * KP + k;
            if (b2[gk] != 0.f && b1[gk] != 0.f && (!ps || ps[gk] != 0.f)) mask |= 1u << (k & 31);
        }
        b.w = __uint_as_float(mask);
    }
    reinterpret_cast<float4*>(out)[2 * (long long)j] = a;
    reinterpret_cast<float4*>(out)[2 * (long long)j + 1] = b;
}

// ORI_F_DETERMINISTIC: the per-(item, CTA, warp) ELBO terms of the gene pass, added in index order by one block
__global__ void __launch_bounds__(1024)
k_det_sum_items(const double* __restrict__ item_part, long long n_slots, double* __restrict__ dst0, double* __restrict__ dst1)
{
    __shared__ double s0[1024], s1[1024];
    double a = 0.0, b = 0.0;
    // thread t owns the contiguous range [t * per, (t + 1) * per): a fixed order whatever the timing
    const long long per = (n_slots + 1023) / 1024;
    const long long lo = (long long)threadIdx.x * per, hi = lo + per < n_slots ? lo + per : n_slots;
    for (long long i = lo; i < hi; ++i) { a += item_part[2 * i]; b += item_part[2 * i + 1]; }
    s0[threadIdx.x] = a; s1[threadIdx.x] = b;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if (threadIdx.x < w) { s0[threadIdx.x] += s0[threadIdx.x + w]; s1[threadIdx.x] += s1[threadIdx.x + w]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { *dst0 += s0[0]; *dst1 += s1[0]; }
}

__global__ void k_det_add(double* __restrict__ dst, const double* __restrict__ src, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}

// ---- host side ---------------------------------------------------------------------------------------------------
// accumulation chunk lengths in sweep entries (see tc_partition)
#ifndef ORI_TC_CHUNK
#define ORI_TC_CHUNK 16384
#endif
#ifndef ORI_TC_CHUNK_PRECISE
#define ORI_TC_CHUNK_PRECISE 2048
#endif
static long long pad128(long long v) { return (v + 127) / 128 * 128; }

long long det_max_items(long long n_rows, int p) {
    // items = own units x sweep chunks; the shortest nominal chunk is ORI_TC_CHUNK_PRECISE sweep entries, own units are at
    // least 128 wide, and the small-problem splitting of tc_partition stops below one item per SM
    const long long np = pad128(n_rows), pp = pad128(p);
    const long long a = (np / 128) * (pp / ORI_TC_CHUNK_PRECISE + 1), b = (pp / 128) * (np / ORI_TC_CHUNK_PRECISE + 1);
    long long m = a > b ? a : b;
    return m > 2 * 148 ? m : 2 * 148;
}
long long det_simt_offset(long long n_rows, int p) {
    const long long tiles = (pad128(n_rows) + pad128(p)) / 128 + 64;
    return (long long)DET_FU_BLOCKS * DET_FU_SLOTS + pad128(p) + det_max_items(n_rows, p) * DET_ITEM_SLOTS + (tiles + 1) / 2 + 2;
}
long long det_workspace_doubles(long long n_rows, int p, int KP) {
    (void)KP;
    long long simt = 0;
    if (det_simt_ok(n_rows, p)) {
        const long long nb = (n_rows + 127) / 128, chunks = (n_rows + 8191) / 8192;
        simt = nb * p + 2 * nb + 2 + (chunks * 3 * p * 64 + 1) / 2 + 8;
    }
    return det_simt_offset(n_rows, p) + simt;
}
int launch_det_sum_pairs(const double* src, long long n, double* dst0, double* dst1, cudaStream_t st) {
    k_det_sum_items<<<1, 1024, 0, st>>>(src, n, dst0, dst1);
    return check_launch("k_det_sum_items");
}

long long tc_workspace_floats(long long n_rows, int p, int KP) {
    const long long np = pad128(n_rows), pp = pad128(p);
    return 8LL * KP * (np + pp) + 3 * pp + 32;      // K-major 4 arrays + transposed 2 tf32 + 2 bf16-pair arrays per side
}

struct TcWs { float *rowK, *rowT, *geneK, *geneT, *lp2w, *flw, *cw; int* flags; long long np, pp; };
static TcWs tc_carve(const ori_problem_t* P) {
    TcWs w;
    w.np = pad128(P->n_rows); w.pp = pad128(P->p);
    const long long KP = P->KP;
    float* f = P->tc_ws;
    w.rowK = f; f += 4 * w.np * KP;
    w.rowT = f; f += 4 * KP * w.np;        // [e | E] tf32, then [e | E] bf16 pairs (PRECISE)
    w.geneK = f; f += 4 * w.pp * KP;
    w.geneT = f; f += 4 * KP * w.pp;
    w.lp2w = f; f += w.pp;
    w.flw = f; f += w.pp;
    w.cw = f; f += w.pp;
    w.flags = (int*)f;
    return w;
}

bool tc_eligible(const ori_problem_t* P) {
    if ((P->flags & (ORI_F_SPARSE | ORI_F_PRECISE)) && P->KP != 32) return false;
    return P->tc_ws != nullptr && (P->KP == 32 || P->KP == 64) && !(P->flags & ORI_F_NO_TENSOR) && P->n_rows > 0 &&
           P->tc_ws_floats >= tc_workspace_floats(P->n_rows, P->p, P->KP) && get_encode_fn() != nullptr;
}

static int num_sms() {
    static int n = 0;
    if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = 148; }
    return n;
}

// gene-side operands (+ padded logit(pi)): the sweep side of the row pass; run once per iteration before it
int launch_tc_prep_genes(const ori_problem_t* P, cudaStream_t st) {
    const TcWs w = tc_carve(P);
    const bool drop = P->flags & ORI_F_DROPOUT, sparse = P->flags & ORI_F_SPARSE;
    const int KP = P->KP;
    const dim3 tg(cdiv(w.pp, 32), KP / 32);
    // sparse model (sparse_zigap.py:100-116, :140-142, :166): the denominator operand carries the mask, the row sums
    // contract with eVz, D_hat is rebuilt from the PREVIOUS effective V_hat, the rate sums contract with the current one
    const float* e_den = sparse ? P->eVd : P->eV;
    const float* e_acc = sparse ? P->eVz : P->eV;
    const float* E_uv = sparse ? P->Vh_old : P->V_hat;
    k_tc_prep_K<<<cdiv(w.pp * KP, 256), 256, 0, st>>>(e_den, drop ? E_uv : nullptr, LOG2E, w.geneK, P->p, w.pp, KP);
    const bool precise = (P->flags & ORI_F_PRECISE) != 0;
    auto t16 = [&](float* base, long long pad, int q) -> uint32_t* {      // bf16-pair twin of transposed array q (PRECISE)
        return precise ? reinterpret_cast<uint32_t*>(base + (long long)(2 + q) * KP * pad) : nullptr;
    };
    k_tc_prep_T<<<tg, dim3(32, 8), 0, st>>>(e_acc, w.geneT, t16(w.geneT, w.pp, 0), P->p, w.pp, KP);
    {
        const cudaError_t e_ = cudaMemsetAsync(w.flags, 0, 32 * sizeof(int), st);
        if (e_ != cudaSuccess) return set_error(ORI_ECUDA, "cudaMemsetAsync(tc flags): %s", cudaGetErrorString(e_));
    }
    if (drop) {
        k_tc_prep_T<<<tg, dim3(32, 8), 0, st>>>(P->V_hat, w.geneT + (long long)KP * w.pp, t16(w.geneT, w.pp, 1), P->p, w.pp, KP);
        k_tc_prep_lp<<<cdiv(w.pp, 256), 256, 0, st>>>(P->lp, P->pfloor, w.lp2w, w.flw, w.cw, w.flags, P->p, (int)w.pp);
    }
    const bool ufl = P->thrU && P->thrV;
    if (ufl) k_tc_thr_max<<<(cdiv(P->p, 256) < 296 ? (int)cdiv(P->p, 256) : 296), 256, 0, st>>>(P->thrV, P->p, w.flags + 1);
    return check_launch("k_tc_prep(genes)", (drop ? 4 : 2) + (ufl ? 1 : 0));
}
// row-side operands, the sweep side of the gene pass: K-major hi/lo of generation g (the state that generated
// D_hat), transposed Zj weight (eU, or eU * D_hat[:, :K] under the quirk) and transposed NEW U_hat
// (zigap.py:124); run after the U update
int launch_tc_prep_rows(const ori_problem_t* P, int g, cudaStream_t st) {
    const TcWs w = tc_carve(P);
    const bool drop = P->flags & ORI_F_DROPOUT;
    const int KP = P->KP;
    const dim3 tg(cdiv(w.np, 32), KP / 32);
    k_tc_prep_K<<<cdiv(w.np * KP, 256), 256, 0, st>>>(P->eU[g], drop ? P->U_hat[g] : nullptr, 1.f, w.rowK, P->n_rows, w.np, KP);
    const float* wsrc = (P->flags & ORI_F_QUIRK) ? P->eUw : P->eU[g];
    const bool precise = (P->flags & ORI_F_PRECISE) != 0;
    uint32_t* r16 = precise ? reinterpret_cast<uint32_t*>(w.rowT + 2ll * KP * w.np) : nullptr;
    k_tc_prep_T<<<tg, dim3(32, 8), 0, st>>>(wsrc, w.rowT, r16, P->n_rows, w.np, KP);
    if (drop) k_tc_prep_T<<<tg, dim3(32, 8), 0, st>>>(P->U_hat[1 - g], w.rowT + (long long)KP * w.np,
                                                      precise ? r16 + (long long)KP * w.np : nullptr, P->n_rows, w.np, KP);
    const bool ufl = P->thrU && P->thrV;
    if (ufl) k_tc_thr_max<<<(cdiv(P->n_rows, 256) < 296 ? (int)cdiv(P->n_rows, 256) : 296), 256, 0, st>>>(
        P->thrU + (long long)g * P->n_rows, P->n_rows, w.flags + 2);
    return check_launch("k_tc_prep(rows)", (drop ? 3 : 2) + (ufl ? 1 : 0));
}

// sparse model, third gene-side sum (sparse_zigap.py:116): the transposed operand of accumulator 1 becomes eU * E[log U]
int launch_tc_prep_rows_logsum(const ori_problem_t* P, int g, cudaStream_t st) {
    const TcWs w = tc_carve(P);
    const dim3 tg(cdiv(w.np, 32), P->KP / 32);
    const bool precise = (P->flags & ORI_F_PRECISE) != 0;
    k_tc_prep_T<<<tg, dim3(32, 8), 0, st>>>(P->eUl[g], w.rowT, precise ? reinterpret_cast<uint32_t*>(w.rowT + 2ll * P->KP * w.np) : nullptr,
                                            P->n_rows, w.np, P->KP);
    return check_launch("k_tc_prep(rows, logsum)");
}

// Split the sweep into chunks of a FIXED length: the accumulators of a work item live in TMEM, and the tensor core's fp32
// accumulation truncates -- a chain of S accumulating MMAs comes out about S * 3e-8 low (measured: sum_ij D_ij (U V^T)_ij
// at 100k x 20k differed by 8e-6 between a 2504-step and an 830-step chaining of the same state, and with it the ELBO by
// 2e-5).  Items therefore hand their partial sums to global memory (round-to-nearest float atomics) every ORI_TC_CHUNK
// sweep entries and, because the chunk length depends on nothing but the kernel plan, every cell and gene sees the same
// chaining whatever the number of ranks or slabs the matrix is split into: the same state evaluated by the device model
// and by host-streamed slabs gives the same ELBO to 1e-8 (it differed by 2e-5 ... 1e-4 when the chunking followed the
// load balance).  Every item boundary drains the pipeline and reloads the own-side operands; measured at config 4
// (1M x 20k, K = 32, one GPU, ms per step / row pass / gene pass): 4096: 53.9 / 21.0 / 31.5, 8192: 52.8 / 20.5 / 30.9,
// 16384: 51.9 / 20.2 / 30.3.  The TF32-operand mode takes 16384 (2048 accumulating steps: a bias of ~3e-5, an order of
// magnitude below its operand rounding); the fp32-grade mode 2048 (256 + 256 steps, ~4e-6).  Cutting the chain inside an
// item instead (two accumulator sets in TMEM, the element-wise warps flushing one while the other accumulates) was built
// and measured: 60.2 / 24.3 / 34.4 ms -- the flush code in the element-wise loop costs more than the drains it saves.
// Problems too small to give every SM (pair) an item are split further.
static void tc_partition(TcArgs& a, bool genes, int units, int sw, bool precise, bool fixed_chain) {
    // the row pass sweeps the genes: its chaining depends on p only (not on the sharding / slabbing of the cells), so its
    // chunks may be twice as long -- one item per row block up to p = 32768 -- at the same accumulation bias
    int tpc = (precise ? ORI_TC_CHUNK_PRECISE : (genes ? ORI_TC_CHUNK : 2 * ORI_TC_CHUNK)) / sw;
    if (tpc < 1) tpc = 1;
    if (tpc > a.n_sw_tiles) tpc = a.n_sw_tiles;
    const int min_tpc = (128 / sw) > 1 ? 128 / sw : 1;
    // small problems: split further, but only when fewer than half of the units would get an item -- a 16384-row slab
    // (64 row-block pairs) keeps the chaining of a large matrix
    // (never for a slab of a larger matrix -- ORI_F_FIXED_CHAIN -- whose sums must be chained like the resident matrix's)
    while (!fixed_chain && (long long)a.n_own_units * cdiv(a.n_sw_tiles, tpc) < units / 2 && tpc > min_tpc) tpc = (tpc + 1) / 2;
    a.tiles_per_chunk = tpc;
    a.n_chunks = cdiv(a.n_sw_tiles, a.tiles_per_chunk);
    a.n_items = a.n_own_units * a.n_chunks;
}

template <bool GENES, bool D, bool E, int KP, bool PRECISE, bool DEVI, bool UFL, bool DET>
static int launch_tc_variant(const TcMaps& maps, const TcArgs& a, int grid, cudaStream_t st) {
    auto kern = k_tc_pass<GENES, D, E, KP, PRECISE, DEVI, UFL, DET>;
    constexpr uint32_t smem = Cfg<KP, PRECISE, DEVI>::SMEM_BYTES;
    static bool attr_done = false;
    if (!attr_done) {
        cudaError_t e_ = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e_ != cudaSuccess) return set_error(ORI_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e_));
        attr_done = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = NCTA; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e_ = cudaLaunchKernelEx(&cfg, kern, maps, a);
    if (e_ != cudaSuccess) return set_error(ORI_ECUDA, "cudaLaunchKernelEx(k_tc_pass): %s", cudaGetErrorString(e_));
    return ORI_OK;
}

// the instance of a pass for its (dropout, ELBO) flags
template <bool GENES, int KP, bool PRECISE, bool UFL, bool DET>
static int launch_tc_flags(bool drop, bool elbo, const TcMaps& maps, const TcArgs& a, int grid, cudaStream_t st) {
    if (drop && elbo) return launch_tc_variant<GENES, true, true, KP, PRECISE, false, UFL, DET>(maps, a, grid, st);
    if (drop) return launch_tc_variant<GENES, true, false, KP, PRECISE, false, UFL, DET>(maps, a, grid, st);
    if (elbo) return launch_tc_variant<GENES, false, true, KP, PRECISE, false, UFL, DET>(maps, a, grid, st);
    return launch_tc_variant<GENES, false, false, KP, PRECISE, false, UFL, DET>(maps, a, grid, st);
}

// logsum: the dropout-free sweep of the sparse model's third gene-side sum into red32 block 2
template <bool GENES, int KP, bool PRECISE>
static int launch_tc_pass_p(const ori_problem_t* P, int gen_old, cudaStream_t st, bool logsum = false) {
    using C = Cfg<KP, PRECISE>;
    const TcWs w = tc_carve(P);
    const bool sparse = P->flags & ORI_F_SPARSE;
    const bool drop = (P->flags & ORI_F_DROPOUT) && !logsum, elbo = (P->flags & ORI_F_ELBO) && !logsum;
    constexpr int SW = C::SW;
    TcMaps maps;
    TcArgs a;
    bool ok;
    // streamed-operand boxes: K-major [32 latent x SW / NCTA sweep rows] per K block, transposed
    // [32 sweep x KP / NCTA latent rows] per chunk (a CTA of a pair stages half of the rows)
    if (!GENES) {
        ok = make_tmap_f32(&maps.swK, w.geneK, 4 * w.pp, KP, KP, 32, SW / NCTA) &&
             make_tmap_f32(&maps.swT, w.geneT, C::NTA * KP, w.pp, w.pp, 32, KP / NCTA) &&
             make_tmap_f32(&maps.X, P->X, P->n_rows, P->p, P->ldx, 32, TC_OWN);
        a.own_total = P->n_rows; a.sw_total = P->p; a.sw_pad = w.pp;
        a.own_e = P->eU[gen_old]; a.own_E = P->U_hat[gen_old];
        a.acc1 = P->Zi; a.acc2 = P->a2s;
    } else {
        ok = make_tmap_f32(&maps.swK, w.rowK, 4 * w.np, KP, KP, 32, SW / NCTA) &&
             make_tmap_f32(&maps.swT, w.rowT, C::NTA * KP, w.np, w.np, 32, KP / NCTA) &&
             make_tmap_f32(&maps.X, P->X, P->n_rows, P->p, P->ldx, 32, SW);
        a.own_total = P->p; a.sw_total = P->n_rows; a.sw_pad = w.np;
        a.own_e = sparse ? P->eVd : P->eV; a.own_E = sparse ? P->Vh_old : P->V_hat;
        a.acc1 = P->red32 + (logsum ? 2ll * P->p * KP : 0ll); a.acc2 = P->red32 + (long long)P->p * KP;
    }
    if (!ok) return set_error(ORI_ECUDA, "cuTensorMapEncodeTiled failed");
    a.lp2w = w.lp2w; a.flw = w.flw; a.cw = w.cw; a.any_floor = w.flags;
    const bool ufl = P->thrU && P->thrV;          // underflow emulation (thresholds reduced by the prep launches)
    const float* thr_rows = ufl ? P->thrU + (long long)gen_old * P->n_rows : nullptr;     // thresholds of generation gen_old
    a.thr_own = ufl ? (GENES ? P->thrV : thr_rows) : nullptr;
    a.thr_sw = ufl ? (GENES ? thr_rows : P->thrV) : nullptr;
    a.thr_sw_max = ufl ? reinterpret_cast<const float*>(w.flags + (GENES ? 2 : 1)) : nullptr;
    a.colsum = P->red64; a.part64 = P->red64 + P->p + 2 * P->KP;
    a.n_own_tiles = cdiv(a.own_total, TC_OWN);
    a.n_own_units = cdiv(a.n_own_tiles, NCTA);
    a.n_sw_tiles = cdiv(a.sw_total, SW);
    const int units = num_sms() / NCTA;
    tc_partition(a, GENES, units, SW, PRECISE, (P->flags & ORI_F_FIXED_CHAIN) != 0);
    const int grid = NCTA * (a.n_items < units ? a.n_items : units);
    a.tickets = nullptr; a.item_part = nullptr; a.colsum2 = nullptr;
    const bool det = (P->flags & ORI_F_DETERMINISTIC) && P->det_ws;
    if (det) {
        if (ufl) return set_error(ORI_EUNSUPPORTED, "ORI_F_DETERMINISTIC and the underflow thresholds cannot be combined on the tensor path");
        if (a.n_items > det_max_items(P->n_rows, P->p)) return set_error(ORI_EINVAL, "det_ws too small for %d items", a.n_items);
        a.colsum2 = P->det_ws + (long long)DET_FU_BLOCKS * DET_FU_SLOTS;
        a.item_part = a.colsum2 + pad128(P->p);
        if (GENES && drop) {
            const cudaError_t e2 = cudaMemsetAsync(a.colsum2, 0, sizeof(double) * (size_t)P->p, st);
            if (e2 != cudaSuccess) return set_error(ORI_ECUDA, "cudaMemsetAsync(colsum2): %s", cudaGetErrorString(e2));
        }
        a.tickets = reinterpret_cast<int*>(a.item_part + det_max_items(P->n_rows, P->p) * DET_ITEM_SLOTS);
        cudaError_t e_ = cudaMemsetAsync(a.tickets, 0, sizeof(int) * (size_t)(a.n_own_tiles + 2), st);
        if (e_ != cudaSuccess) return set_error(ORI_ECUDA, "cudaMemsetAsync(tickets): %s", cudaGetErrorString(e_));
        if (!(GENES && elbo)) a.item_part = nullptr;
        else {      // the kernel writes every (CTA, warp) slot of an item; zeroed all the same, so no stale value is ever summed
            e_ = cudaMemsetAsync(a.item_part, 0, sizeof(double) * (size_t)a.n_items * DET_ITEM_SLOTS, st);
            if (e_ != cudaSuccess) return set_error(ORI_ECUDA, "cudaMemsetAsync(item_part): %s", cudaGetErrorString(e_));
        }
    }
    const int rc = det ? launch_tc_flags<GENES, KP, PRECISE, false, true>(drop, elbo, maps, a, grid, st)
                 : ufl ? launch_tc_flags<GENES, KP, PRECISE, true, false>(drop, elbo, maps, a, grid, st)
                       : launch_tc_flags<GENES, KP, PRECISE, false, false>(drop, elbo, maps, a, grid, st);
    if (rc != ORI_OK) return rc;
    int extra = 0;
    if (det && GENES && drop) { k_det_add<<<cdiv(P->p, 256), 256, 0, st>>>(P->red64, a.colsum2, P->p); ++extra; }
    if (a.item_part) {
        double* part = P->red64 + P->p + 2 * P->KP;
        k_det_sum_items<<<1, 1024, 0, st>>>(a.item_part, (long long)a.n_items * (DET_ITEM_SLOTS / 2), part + R64_XLOGDEN, part + R64_ENT);
        ++extra;
    }
    if (extra) return check_launch("k_tc_pass + deterministic sums", 1 + extra);
    return check_launch(GENES ? "k_tc_pass(genes)" : "k_tc_pass(rows)");
}

template <bool GENES>
static int launch_tc_pass(const ori_problem_t* P, int gen_old, cudaStream_t st, bool logsum = false) {
    // fp32-grade contractions: KP = 32 plan with 32-wide sweep tiles (tc_eligible checks KP)
    if (P->flags & ORI_F_PRECISE) return launch_tc_pass_p<GENES, 32, true>(P, gen_old, st, logsum);
    if (P->KP == 64) return launch_tc_pass_p<GENES, 64, false>(P, gen_old, st, logsum);
    return launch_tc_pass_p<GENES, 32, false>(P, gen_old, st, logsum);
}

// The three truncated log-likelihood sums behind reconstruction_deviance / explained_deviance (base.py:58-82) on the
// tensor path: a row-oriented pass whose two contractions are the rate U_hat . V_hat^T and the one that generates D_hat.
template <int KP>
static int launch_deviance_tc_kp(const ori_problem_t* P, int g, const double* pi, const double* cmean, long long* out_int,
                                 cudaStream_t st) {
    using C = Cfg<KP, false, true>;
    constexpr int SW = C::SW;
    const TcWs w = tc_carve(P);
    const bool sparse = P->flags & ORI_F_SPARSE;
    // gene-side K-major operands: [hi | lo] of the effective V_hat (rate) and of the V_hat that generates D_hat (log2 units)
    k_tc_prep_K<<<cdiv(w.pp * KP, 256), 256, 0, st>>>(P->V_hat, sparse ? P->Vh_old : P->V_hat, LOG2E, w.geneK, P->p, w.pp, KP);
    float* devlp = w.geneT;                 // the transposed-operand area is free here (no accumulating contraction)
    k_tc_prep_dev<<<cdiv(w.pp, 256), 256, 0, st>>>(P->lp, pi, cmean, devlp, P->p, (int)w.pp, P->b1, P->b2, sparse ? P->p_s : nullptr, KP);
    {
        const cudaError_t e_ = cudaMemsetAsync(w.flags, 0, 32 * sizeof(int), st);
        if (e_ != cudaSuccess) return set_error(ORI_ECUDA, "cudaMemsetAsync(tc flags): %s", cudaGetErrorString(e_));
    }
    if (check_launch("k_tc_prep(deviance)", 2) != ORI_OK) return ORI_ECUDA;
    TcMaps maps;
    TcArgs a;
    memset(&a, 0, sizeof(a));
    const bool ok = make_tmap_f32(&maps.swK, w.geneK, 4 * w.pp, KP, KP, 32, SW / NCTA) &&
                    make_tmap_f32(&maps.swT, w.geneT, C::NTA * KP, w.pp, w.pp, 32, KP / NCTA) &&
                    make_tmap_f32(&maps.X, P->X, P->n_rows, P->p, P->ldx, 32, TC_OWN);
    if (!ok) return set_error(ORI_ECUDA, "cuTensorMapEncodeTiled failed");
    a.own_total = P->n_rows; a.sw_total = P->p; a.sw_pad = w.pp;
    a.own_e = P->U_hat[g]; a.own_E = P->U_hat[g];
    a.lp2w = w.lp2w; a.flw = w.flw; a.cw = w.cw; a.any_floor = w.flags;
    a.devlp = devlp;
    a.dev_b1 = P->b1; a.dev_b2 = P->b2; a.dev_ps = sparse ? P->p_s : nullptr;
    a.dev_out = (unsigned long long*)out_int;
    a.n_own_tiles = cdiv(a.own_total, TC_OWN);
    a.n_own_units = cdiv(a.n_own_tiles, NCTA);
    a.n_sw_tiles = cdiv(a.sw_total, SW);
    const int units = num_sms() / NCTA;
    // one chunk per row block where that fills the machine: nothing accumulates in TMEM here
    a.tiles_per_chunk = a.n_sw_tiles;
    while ((long long)a.n_own_units * cdiv(a.n_sw_tiles, a.tiles_per_chunk) < 2LL * units && a.tiles_per_chunk > 4)
        a.tiles_per_chunk = (a.tiles_per_chunk + 1) / 2;
    a.n_chunks = cdiv(a.n_sw_tiles, a.tiles_per_chunk);
    a.n_items = a.n_own_units * a.n_chunks;
    const int grid = NCTA * (a.n_items < units ? a.n_items : units);
    const int rc = launch_tc_variant<false, true, false, KP, false, true, false, false>(maps, a, grid, st);
    if (rc != ORI_OK) return rc;
    return check_launch("k_tc_pass(deviance)");
}

// integer sums only (the float64 sums stay on the CUDA-core kernel); `pi`, `cmean` as for launch_deviance
int launch_deviance_tc(const ori_problem_t* P, int g, const double* pi, const double* cmean, long long* out_int, cudaStream_t st) {
    if (P->KP == 64) return launch_deviance_tc_kp<64>(P, g, pi, cmean, out_int, st);
    return launch_deviance_tc_kp<32>(P, g, pi, cmean, out_int, st);
}

int launch_pass_rows_tc(const ori_problem_t* P, int gen_old, cudaStream_t st) { return launch_tc_pass<false>(P, gen_old, st); }
int launch_pass_genes_tc(const ori_problem_t* P, int gen_old, cudaStream_t st) { return launch_tc_pass<true>(P, gen_old, st); }
int launch_pass_genes_logsum_tc(const ori_problem_t* P, int gen_old, cudaStream_t st) { return launch_tc_pass<true>(P, gen_old, st, true); }

}  // namespace ori
