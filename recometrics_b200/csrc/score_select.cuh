// score_select.cuh -- fused "score -> exclude train -> running top-K (+ rank counting)" kernel.
//
// Replaces, for a tile of 128 users at a time, the per-user loop body of the reference:
//   candidate list      /root/reference/src/recometrics.hpp:491-497
//   dot1 scoring        /root/reference/src/recometrics.hpp:84-112, :499-512
//   partial_sort / sort /root/reference/src/recometrics.hpp:537-563
//   (the AUC walks of :795-865 become a counting pass over the same score tiles)
//
// Design (sm_100a; FP32 on the packed FFMA2 pipe, FP64 on DFMA):
//   * Factors are re-tiled once per call into slabs  At[user tile][k][128]  /  Bt[item tile][k][128]
//     (k-major inside a 128-wide tile), so the operand chunk of one pipeline stage is ONE contiguous
//     block: a single TMA bulk copy (cp.async.bulk, SASS UBLKCP) lands it in shared memory in
//     exactly the layout the FMA micro-kernel reads.
//   * CTA = 8 compute warps + 1 producer warp.  The producer's elected lane runs the TMA ring
//     (full/empty mbarriers, STAGES deep) over the flattened (item tile, k chunk) space; compute
//     warps never meet at a CTA barrier.
//   * CTA tile 128 users x 128 items; a compute warp OWNS 16 users x 128 items (thread micro-tile
//     8 users x 8 items in registers), so all per-user selection state is warp-private.
//     fp32: the 8x8 micro-tile is 32 packed accumulators updated with fma.rn.f32x2, user factor as
//     the scalar-broadcast operand (SASS: FFMA2 Rd, Ra.F32, Rb.F32x2, Rc.F32x2) -- half the issue
//     slots of FFMA and no register-bank conflicts (profiles/r01_ubench_fma.txt).
//   * The score tile never leaves registers: per user row a thread takes the max of its 8 scores
//     and compares it with the user's running K-th best (tau).  Survivors (~K ln(n/K) per user over
//     the whole catalogue) are checked against the user's train row (only in item tiles the sorted
//     train row intersects -- a per-row cursor keeps the next train item id) and appended to a
//     per-user candidate buffer of C entries in global memory (L2 resident).  When a buffer passes
//     C - BN entries its warp cuts it back to the best K with a bitwise radix select on the
//     order-preserving integer image of the scores (warp REDUX counts; ties at the cut resolved by
//     item id), which refreshes tau.  rank_topk_kernel finally orders the K survivors.
//   * AUC mode (ROC/PR requested): the warp stages its 16 x BN score block in shared memory, masks
//     train items there, and counts for every held-out item of its rows the candidates of the tile
//     that rank before it (score above, or equal with a smaller item id).  The held-out entries of
//     the warp's 16 rows form one list dealt out to the 32 lanes, so the work is the sum of the
//     rows' held-out counts, not 16 x their maximum; per score one compare on the ALU pipe and half
//     a packed add on the FMA pipe; counters in global memory, one owner each (no atomics).
//     Scores of held-out items are pre-computed with the same FMA order (prep.cuh) so comparisons
//     are exact.
//   * Everything outside the FMA loop is written as rolled loops / out-of-line calls: the epilogue
//     runs once per item tile and must not evict the FMA loop from the instruction cache.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <limits.h>
#include <string.h>

namespace rmb {

constexpr int BM = 128;             // users per CTA tile (items per tile: NumTraits<T>::BN)
constexpr int NCWARPS = 8;          // compute warps (16 user rows each)
constexpr int NTHREADS = (NCWARPS + 1) * 32;   // + 1 producer warp
// Rank-counting (AUC) mode is warp-specialised: next to the 8 FMA warps and the producer warp the CTA has 8 COUNTING warps.
// FMA warp w hands the 16 x BN score block of every item tile to counting warp w through shared memory (one block per pair,
// full / empty mbarriers) and goes on with the next tile's FMAs; the counting warp masks the train items, tracks the row
// minima and counts the held-out items' ranks on the ALU pipe while the FMA pipe keeps running.  Registers are moved to
// where they are needed with setmaxnreg (FMA warps 152 / counting warps 72 in float, 160 / 64 in double, producer warp group 32: exactly the 640 x 96 registers the CTA is launched with --
// setmaxnreg only redistributes the CTA's own allocation).
constexpr int AUC_THREADS = 640;    // 8 FMA warps + 8 counting warps + 1 producer warp (+ 3 idle warps: setmaxnreg works on groups of 4)
constexpr int AUC_PCAP = 384;       // held-out entries per counting warp whose score / item id are staged in shared memory (the rest: global)
constexpr int KPAD = 8;             // factors are zero-padded to a multiple of this
constexpr unsigned FULL = 0xffffffffu;
typedef unsigned long long u64;

template <typename T> struct NumTraits;
template <> struct NumTraits<float> {
    static constexpr int BN = 128;      // items per tile (thread micro-tile 8 users x 8 items)
    static constexpr int BK = 32;       // factors per pipeline stage
    static constexpr int STAGES = 4;
    typedef unsigned key_t;             // order-preserving integer image of a score
    static constexpr int KEYBITS = 32;
    __device__ __forceinline__ static key_t key(float x) { return (key_t)orderable(x); }
    __device__ __forceinline__ static float inf() { return CUDART_INF_F; }
    __device__ __forceinline__ static float nan() { return CUDART_NAN_F; }
    __device__ __forceinline__ static float fma(float a, float b, float c) { return fmaf(a, b, c); }
    __device__ __forceinline__ static u64 orderable(float x) {
        unsigned u = __float_as_uint(x);
        u ^= (u >> 31) ? 0xffffffffu : 0x80000000u;
        return (u64)u;
    }
    __host__ __device__ static float from_orderable(u64 o) {
        unsigned u = (unsigned)o;
        u ^= (u >> 31) ? 0x80000000u : 0xffffffffu;
#ifdef __CUDA_ARCH__
        return __uint_as_float(u);
#else
        float f; memcpy(&f, &u, 4); return f;
#endif
    }
};
template <> struct NumTraits<double> {
    static constexpr int BN = 64;       // items per tile (thread micro-tile 8 users x 4 items: the
                                        // register file of a 9-warp CTA holds 168 registers per thread)
    static constexpr int BK = 16;
    static constexpr int STAGES = 4;
    typedef u64 key_t;
    static constexpr int KEYBITS = 64;
    __device__ __forceinline__ static key_t key(double x) { return orderable(x); }
    __device__ __forceinline__ static double inf() { return CUDART_INF; }
    __device__ __forceinline__ static double nan() { return CUDART_NAN; }
    __device__ __forceinline__ static double fma(double a, double b, double c) { return ::fma(a, b, c); }
    __device__ __forceinline__ static u64 orderable(double x) {
        u64 u = (u64)__double_as_longlong(x);
        u ^= (u >> 63) ? 0xffffffffffffffffull : 0x8000000000000000ull;
        return u;
    }
    __host__ __device__ static double from_orderable(u64 u) {
        u ^= (u >> 63) ? 0x8000000000000000ull : 0xffffffffffffffffull;
#ifdef __CUDA_ARCH__
        return __longlong_as_double((long long)u);
#else
        double f; memcpy(&f, &u, 8); return f;
#endif
    }
};

// ------------------------------------------------------------------ ranking helpers
// total order used for ranking: score descending, ties by ascending item id
// (the reference's comparator is a strict '>' on the score, hpp:538-540 / :552-554; its tie order
//  is whatever libstdc++ does -- SURVEY quirk Q8 -- so a deterministic refinement is chosen here)
template <typename T>
__device__ __forceinline__ bool ranks_before(T sa, int ia, T sb, int ib)
{
    return (sa > sb) || (sa == sb && ia < ib);
}

// Bitonic sorting network over 32*E (score,item) pairs held E per lane (element i = e*32 + lane),
// best first.  Fully unrolled; strides >= 32 are register exchanges, strides < 32 are shuffles.
template <typename T, int E>
__device__ __forceinline__ void warp_sort_ranked(T (&s)[E], int (&it)[E], const int lane)
{
    constexpr int N = 32 * E;
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const int je = j >> 5;
#pragma unroll
                for (int e = 0; e < E; e++) {
                    if ((e & je) == 0) {
                        const int e2 = e | je;
                        const bool desc = (((e * 32) & k) == 0);
                        const bool first_better = ranks_before<T>(s[e], it[e], s[e2], it[e2]);
                        const bool sw = desc ? !first_better : first_better;
                        if (sw) {
                            const T ts = s[e]; s[e] = s[e2]; s[e2] = ts;
                            const int ti = it[e]; it[e] = it[e2]; it[e2] = ti;
                        }
                    }
                }
            } else {
#pragma unroll
                for (int e = 0; e < E; e++) {
                    const int i = e * 32 + lane;
                    const bool desc = ((i & k) == 0);
                    const bool lower = ((lane & j) == 0);
                    const T so = __shfl_xor_sync(FULL, s[e], j);
                    const int io = __shfl_xor_sync(FULL, it[e], j);
                    const bool mine_better = ranks_before<T>(s[e], it[e], so, io);
                    const bool keep_better = (lower == desc);
                    if (mine_better != keep_better) { s[e] = so; it[e] = io; }
                }
            }
        }
    }
}

template <typename T>
struct ScoreSelectParams {
    const T* __restrict__ At;      // [user tiles][p_pad][128]  user factors of this batch, zero padded
    const T* __restrict__ Bt;      // [item tiles][p_pad][128]  item factors, zero padded
    const T* __restrict__ bias;    // [item tiles * 128] item biases (zero padded) or nullptr
    int p_pad;
    int n;                          // items
    int mb;                         // users in this batch
    int user0;                      // row (of the CSR / status arrays) of the batch's first user
    const int* __restrict__ trp;    // train CSR
    const int* __restrict__ tri;
    const int* __restrict__ tep;    // test CSR indptr
    const int* __restrict__ ustatus;// [m] 0 = user is ranked, !=0 = NaN row decided before scoring
    T* cand_score;                  // [mb_pad][C]
    int* cand_item;                 // [mb_pad][C]
    int* cand_count;                // [mb_pad] entries left at the head of the buffer (<= K, unordered)
    int* uflags;                    // [m] bit0: a candidate score was NaN
    int K;
    // rank counting (AUC mode)
    const T* __restrict__ pos_sorted;   // [nnz_test] held-out item scores, ascending per user
    const int* __restrict__ pos_item;   // [nnz_test] their item ids
    unsigned int* auc_cnt;              // [nnz_test] number of candidates ranked before the j-th smallest held-out item
                                        // of the row: scoring above it, or equal with a smaller item id (zeroed)
    unsigned int* auc_near;             // optional [nnz_test] (break_ties_with_noise): number of candidates, the item itself included,
                                        // whose score lies within the reach of the tie-breaking noise of the held-out item's
                                        // (>= 2: the noise decides a rank of this user, api.cu hands the user to the full-order path)
    u64* umin;                          // [m] orderable(min candidate score), init ~0
    int slice_rows;                     // item slices (gridDim.y > 1: a call with fewer user tiles than SMs cuts the catalogue into ranges, one CTA per
                                        // (user tile, range)): rows of cand_score / cand_item / cand_count per slice -- slice y keeps the best K of its
                                        // range in rows [y * slice_rows, ...), merge_slices_kernel joins them; rank counts are then added atomically
    const int* __restrict__ umap;       // optional [mb]: row r of this launch is batch-local user umap[r] (CSR rows, status, flags and
                                        // candidate buffers are those of the mapped user; At holds the launch's rows in order).  Used
                                        // to re-run only the users the tensor-core filter handed back (api.cu)
};

// ------------------------------------------------------------------ PTX wrappers (TMA ring)
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(const unsigned bar, const unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(const unsigned bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(const unsigned bar, const unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(const unsigned bar, const unsigned parity)
{
    unsigned ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
// global -> shared bulk copy executed by the TMA unit, completion counted on an mbarrier
__device__ __forceinline__ void tma_bulk_g2s(const unsigned dst, const void* src, const unsigned bytes, const unsigned bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

__device__ __forceinline__ u64 pack2(const float lo, const float hi)
{
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(const u64 v, float& lo, float& hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
// d = a * b + d on two packed fp32 lanes (each lane an IEEE fma, same rounding as fmaf)
__device__ __forceinline__ void fma2(u64& d, const u64 a, const u64 b)
{
    asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}
__device__ __forceinline__ float max_nan(const float a, const float b)
{
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ double max_nan(const double a, const double b)
{
    return (a != a || b != b) ? CUDART_NAN : (a > b ? a : b);
}

__device__ __forceinline__ void lds_vec(const float* p, float (&v)[4])
{
    const float4 f = *reinterpret_cast<const float4*>(p);
    v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
}
__device__ __forceinline__ void lds_vec(const double* p, double (&v)[2])
{
    const double2 f = *reinterpret_cast<const double2*>(p);
    v[0] = f.x; v[1] = f.y;
}
__device__ __forceinline__ void sts4(float* p, const float* v)
{
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void sts4(double* p, const double* v)
{
    *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
    *reinterpret_cast<double2*>(p + 2) = make_double2(v[2], v[3]);
}

// ------------------------------------------------------------------ register micro-tiles
// Thread (ly = lane >> 4, lx = lane & 15) of a compute warp holds, of the warp's 16 x BN block,
//   rows  ly*4 + (i & 3) + (i >> 2) * 8      i = 0..7
//   cols  lx*4 + (c & 3) + (c >> 2) * 64     c = 0..NC-1   (NC = BN / 16: 8 for fp32, 4 for fp64)
template <typename T> struct MicroTile;

template <> struct MicroTile<float> {
    static constexpr int NC = 8;
    u64 acc[8][4];   // acc[i][c/2] = scores (i, c), (i, c+1)
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[i][q] = 0ull;
    }
    struct Frag { float a[8]; u64 b[4]; };
    // sA: the warp's 16 user values of factor k; sB: the tile's 128 item values of factor k
    __device__ __forceinline__ static void load(Frag& f, const float* __restrict__ sA, const float* __restrict__ sB, const int ly, const int lx)
    {
        const float4 a0 = *reinterpret_cast<const float4*>(sA + ly * 4);
        const float4 a1 = *reinterpret_cast<const float4*>(sA + 8 + ly * 4);
        const ulonglong2 b0 = *reinterpret_cast<const ulonglong2*>(sB + lx * 4);
        const ulonglong2 b1 = *reinterpret_cast<const ulonglong2*>(sB + 64 + lx * 4);
        f.a[0] = a0.x; f.a[1] = a0.y; f.a[2] = a0.z; f.a[3] = a0.w;
        f.a[4] = a1.x; f.a[5] = a1.y; f.a[6] = a1.z; f.a[7] = a1.w;
        f.b[0] = b0.x; f.b[1] = b0.y; f.b[2] = b1.x; f.b[3] = b1.y;
    }
    __device__ __forceinline__ void compute(const Frag& f)
    {
#pragma unroll
        for (int q = 0; q < 4; q++)
#pragma unroll
            for (int i = 0; i < 8; i++) fma2(acc[i][q], pack2(f.a[i], f.a[i]), f.b[q]);
    }
    __device__ __forceinline__ void row(const int i, float (&s)[8]) const
    {
#pragma unroll
        for (int q = 0; q < 4; q++) unpack2(acc[i][q], s[2 * q], s[2 * q + 1]);
    }
};

template <> struct MicroTile<double> {
    static constexpr int NC = 4;
    double acc[8][4];
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int c = 0; c < 4; c++) acc[i][c] = 0.;
    }
    struct Frag { double a[8]; double b[4]; };
    __device__ __forceinline__ static void load(Frag& f, const double* __restrict__ sA, const double* __restrict__ sB, const int ly, const int lx)
    {
#pragma unroll
        for (int g = 0; g < 2; g++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const double2 va = *reinterpret_cast<const double2*>(sA + g * 8 + ly * 4 + h * 2);
                f.a[g * 4 + h * 2] = va.x; f.a[g * 4 + h * 2 + 1] = va.y;
            }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const double2 vb = *reinterpret_cast<const double2*>(sB + lx * 4 + h * 2);
            f.b[h * 2] = vb.x; f.b[h * 2 + 1] = vb.y;
        }
    }
    __device__ __forceinline__ void compute(const Frag& f)
    {
#pragma unroll
        for (int c = 0; c < 4; c++)
#pragma unroll
            for (int i = 0; i < 8; i++) acc[i][c] = ::fma(f.a[i], f.b[c], acc[i][c]);
    }
    __device__ __forceinline__ void row(const int i, double (&s)[4]) const
    {
#pragma unroll
        for (int c = 0; c < 4; c++) s[c] = acc[i][c];
    }
};


// ------------------------------------------------------------------ per-CTA shared state
template <typename T>
struct RowState {
    T tau[BM];          // running K-th best score; +inf = row is not ranked (padding / NaN-row user)
    int cnt[BM];        // entries in the row's candidate buffer
    int nan[BM];        // a candidate score was NaN
    int nxt_train[BM];  // smallest train item id >= first item of the current tile (INT_MAX: none)
    int cur_train[BM];  // its position in the train CSR
    int end_train[BM];
    int tp0[BM];        // first entry of the held-out (test) row
    int npos[BM];       // its length (0 for rows that are not ranked)
    int urow[BM];       // batch-local user of the row (its candidate buffer, status, flags): the row itself unless ScoreSelectParams::umap
};

template <typename T, bool AUC>
struct SmemLayout {
    static constexpr int S = NumTraits<T>::STAGES, BN = NumTraits<T>::BN, BK = NumTraits<T>::BK;
    static constexpr size_t a_off = 0;                                            // [S][BK][BM]
    static constexpr size_t b_off = (size_t)S * BK * BM * sizeof(T);              // [S][BK][BN]
    static constexpr size_t rs_off = b_off + (size_t)S * BK * BN * sizeof(T);
    static constexpr size_t bar_off = rs_off + ((sizeof(RowState<T>) + 15) & ~size_t(15));   // full[S], empty[S] (AUC: + blk_full[NCWARPS], blk_empty[NCWARPS])
    static constexpr size_t plain_bytes = bar_off + 2 * S * sizeof(u64);
    // AUC mode only
    static constexpr int BNP = BN + 16 / (int)sizeof(T);                          // row pitch of a staged score block: consecutive rows
                                                                                  // start 16 bytes apart in the banks (lanes of the
                                                                                  // counting loop read several rows at once)
    static constexpr size_t blk_off = plain_bytes + 2 * NCWARPS * sizeof(u64);    // [NCWARPS][16][BNP] score blocks
    static constexpr size_t pref_off = blk_off + (size_t)NCWARPS * 16 * BNP * sizeof(T);  // [BM + 4] held-out entries before row r, [BM + 4] work units before row r
    static constexpr size_t pthr_off = (pref_off + (size_t)2 * (BM + 4) * sizeof(int) + 15) & ~size_t(15);      // [NCWARPS * AUC_PCAP] held-out scores
    static constexpr size_t pitem_off = pthr_off + (size_t)NCWARPS * AUC_PCAP * sizeof(T);     // [NCWARPS][AUC_PCAP] their item ids
    static constexpr size_t auc_bytes = pitem_off + (size_t)NCWARPS * AUC_PCAP * sizeof(int);
};

template <typename T, bool AUC>
inline size_t score_select_smem_bytes() { return AUC ? SmemLayout<T, AUC>::auc_bytes : SmemLayout<T, AUC>::plain_bytes; }

extern __shared__ __align__(128) unsigned char smem_raw[];


// ------------------------------------------------------------------ selection: out-of-line slow paths
// One warp: cut the first nv (>= K) entries of a user's candidate buffer back to the best K
// (score descending, ties at the cut by ascending item id -- the order of ranks_before), left
// unordered at the head; publish the K-th best score (tau) and the new count.
template <typename T, int C>
__device__ __noinline__ void compact_user(T* cs, int* ci, const int nv, const int K, const int lane,
                                          T* tau_out, int* cnt_out)
{
    typedef typename NumTraits<T>::key_t key_t;
    constexpr int E = C / 32;
    if (nv < K) return;                       // nothing to drop yet; tau stays -inf
    key_t key[E];
    int it[E];
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int idx = e * 32 + lane;
        const bool v = idx < nv;
        key[e] = v ? NumTraits<T>::key(cs[idx]) : (key_t)0;     // 0 sorts below every score (NaN is never stored)
        it[e] = v ? ci[idx] : INT_MAX;
    }
    __syncwarp();
    // K-th largest key, bit by bit from the top: the largest t with #(key >= t) >= K
    key_t t = 0;
    for (int b = NumTraits<T>::KEYBITS - 1; b >= 0; b--) {
        const key_t cand = t | ((key_t)1 << b);
        int c = 0;
#pragma unroll
        for (int e = 0; e < E; e++) c += (key[e] >= cand) ? 1 : 0;
        c = __reduce_add_sync(FULL, c);
        if (c >= K) t = cand;
    }
    int cgt = 0, cge = 0;
#pragma unroll
    for (int e = 0; e < E; e++) { cgt += (key[e] > t) ? 1 : 0; cge += (key[e] >= t) ? 1 : 0; }
    cgt = __reduce_add_sync(FULL, cgt);
    cge = __reduce_add_sync(FULL, cge);
    unsigned id_cut = 0x7fffffffu;            // keep tied entries with item id <= id_cut
    if (cge > K) {
        // more entries tie with the K-th score than fit: keep the (K - cgt) smallest item ids among them,
        // i.e. id_cut = max{x : #(tied, id < x) < need}
        const int need = K - cgt;
        unsigned x = 0;
        for (int b = 30; b >= 0; b--) {
            const unsigned cand = x | (1u << b);
            int c = 0;
#pragma unroll
            for (int e = 0; e < E; e++) c += (key[e] == t && (unsigned)it[e] < cand) ? 1 : 0;
            c = __reduce_add_sync(FULL, c);
            if (c < need) x = cand;
        }
        id_cut = x;
    }
    int base = 0;
#pragma unroll
    for (int e = 0; e < E; e++) {
        const bool keep = (key[e] > t) || (key[e] == t && (unsigned)it[e] <= id_cut);
        const unsigned mask = __ballot_sync(FULL, keep);
        if (keep) {
            const int pos = base + __popc(mask & ((1u << lane) - 1u));
            cs[pos] = NumTraits<T>::from_orderable((u64)key[e]);
            ci[pos] = it[e];
        }
        base += __popc(mask);
    }
    if (lane == 0) { *tau_out = NumTraits<T>::from_orderable((u64)t); *cnt_out = base; }
    __syncwarp();
}

// is `item` in the sorted train row segment [lo, hi) ?  (hpp:494-495 moves those out of the pool)
__device__ __forceinline__ bool in_train_segment(const int* __restrict__ tri, int lo, int hi, const int item)
{
    const int end = hi;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tri[mid] < item) lo = mid + 1; else hi = mid;
    }
    return lo < end && tri[lo] == item;
}

// Slow path of the selection filter (taken by ~K ln(n/K) scores per user): candidate checks, then
// append to the user's buffer (cs / ci = the row's candidate buffer).  Everything arrives by value:
// the kernel parameters live in constant memory, which an out-of-line function could only reach
// through a generic pointer.
template <typename T>
__device__ __forceinline__ void insert_candidate(RowState<T>* rs, T* cs, int* ci, const int* __restrict__ tri, const int n,
                                                 const T s, const int row, const int item, const int item_end)
{
    if (item >= n) return;                                      // padding column
    if (rs->nxt_train[row] < item_end &&                        // the train row intersects this tile
        in_train_segment(tri, rs->cur_train[row], rs->end_train[row], item)) return;   // not a candidate
    if (s != s) { rs->nan[row] = 1; return; }                   // NaN candidate score => NaN row
    const int slot = atomicAdd(&rs->cnt[row], 1);
    // slot < C always: the buffer holds <= C-BN entries when a tile starts and a tile adds <= BN
    cs[slot] = s;
    ci[slot] = item;
}

// A thread's scores of one user row in one item tile, at least one of which is not below tau.
// item_lo = id of the first of the four columns.
template <typename T>
__device__ __noinline__ void row_slow(RowState<T>* rs, T* cs, int* ci, const int* __restrict__ tri, const int n, const T tau, const int row,
                                      const int item_lo, const int item_end,
                                      const T s0, const T s1, const T s2, const T s3)
{
    if (tau == NumTraits<T>::inf()) return;                     // row is not ranked (padding / NaN-row user)
    if (!(s0 < tau)) insert_candidate<T>(rs, cs, ci, tri, n, s0, row, item_lo, item_end);
    if (!(s1 < tau)) insert_candidate<T>(rs, cs, ci, tri, n, s1, row, item_lo + 1, item_end);
    if (!(s2 < tau)) insert_candidate<T>(rs, cs, ci, tri, n, s2, row, item_lo + 2, item_end);
    if (!(s3 < tau)) insert_candidate<T>(rs, cs, ci, tri, n, s3, row, item_lo + 3, item_end);
}

// ---- rank counting: how many of the BN staged scores of a row lie strictly above a threshold ----
// float: the compare leaves 1.0f / 0.0f (FSET.BF, the only ALU-pipe instruction per score) and the ones are added as packed
// pairs on the FMA pipe (add.f32x2), four independent accumulators; a tile adds at most BN to each, exact in fp32.
__device__ __forceinline__ float gt_one(const float a, const float p)
{
    float r;
    asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(p));
    return r;
}
__device__ __forceinline__ u64 add2(const u64 a, const u64 b)
{
    u64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// NT thresholds at once: every 16-byte load of the row is compared with all of them (4 x NT independent compares per load).
// Only two counting warps share a scheduler, so latencies are not hidden by other warps: the instruction ORDER is pinned
// (volatile asm keeps program order) -- the next 16-byte load first, then all compares of the current one, then the packed
// adds, each of which then finds its compare results (~20 cycles of latency on FSET.BF) long finished.
__device__ __forceinline__ float gt_one_v(const float a, const float p)
{
    float r;
    asm volatile("set.gt.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(p));
    return r;
}
__device__ __forceinline__ u64 add2_v(const u64 a, const float lo, const float hi)
{
    u64 r;
    asm volatile("{\n\t.reg .b64 t;\n\tmov.b64 t, {%2, %3};\n\tadd.rn.f32x2 %0, %1, t;\n\t}" : "=l"(r) : "l"(a), "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float4 lds128_v(const float* p)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)));
    return v;
}
template <int NT>
__device__ __forceinline__ void count_above(const float* __restrict__ src, const float (&thr)[NT], unsigned (&cnt)[NT])
{
    constexpr int BN = NumTraits<float>::BN;
    u64 acc[NT][2];
#pragma unroll
    for (int t = 0; t < NT; t++) { acc[t][0] = 0ull; acc[t][1] = 0ull; }
    float4 v = lds128_v(src);
#pragma unroll 2
    for (int x = 0; x < BN; x += 4) {
        const float4 nv = lds128_v(src + ((x + 4) & (BN - 1)));      // next load in flight (wraps on the last one)
        float m[NT][4];
#pragma unroll
        for (int t = 0; t < NT; t++) {
            m[t][0] = gt_one_v(v.x, thr[t]); m[t][1] = gt_one_v(v.y, thr[t]);
            m[t][2] = gt_one_v(v.z, thr[t]); m[t][3] = gt_one_v(v.w, thr[t]);
        }
#pragma unroll
        for (int t = 0; t < NT; t++) {
            acc[t][0] = add2_v(acc[t][0], m[t][0], m[t][1]);
            acc[t][1] = add2_v(acc[t][1], m[t][2], m[t][3]);
        }
        v = nv;
    }
#pragma unroll
    for (int t = 0; t < NT; t++) {
        float lo, hi;
        unpack2(add2(acc[t][0], acc[t][1]), lo, hi);
        cnt[t] = (unsigned)(lo + hi);
    }
}
__device__ __forceinline__ unsigned gt_mask(const double a, const double p)
{
    unsigned r;
    asm("set.gt.u32.f64 %0, %1, %2;" : "=r"(r) : "d"(a), "d"(p));
    return r;
}
template <int NT>
__device__ __forceinline__ void count_above(const double* __restrict__ src, const double (&thr)[NT], unsigned (&cnt)[NT])
{
    constexpr int BN = NumTraits<double>::BN;
    unsigned c0[NT], c1[NT];
#pragma unroll
    for (int t = 0; t < NT; t++) { c0[t] = 0; c1[t] = 0; }
#pragma unroll 2
    for (int x = 0; x < BN; x += 2) {
        const double2 v = *reinterpret_cast<const double2*>(src + x);
#pragma unroll
        for (int t = 0; t < NT; t++) { c0[t] -= gt_mask(v.x, thr[t]); c1[t] -= gt_mask(v.y, thr[t]); }
    }
#pragma unroll
    for (int t = 0; t < NT; t++) cnt[t] = c0[t] + c1[t];
}
// How far apart two scores must be for the reference's tie-breaking noise (uniform in [-1e-12, 1e-12) added to each,
// hpp:531-534) to be unable to swap them, as seen from a held-out score p: 0 where adding the noise gives the score back
// (float: |p| >= 2^-13, double: |p| >= 2^16), else twice the noise plus the rounding of the two sums.
__device__ __forceinline__ float noise_reach(const float p) { return fabsf(p) < 1.220703125e-4f ? fmaf(fabsf(p), 4.8e-7f, 2.0e-12f) : 0.f; }
__device__ __forceinline__ double noise_reach(const double p) { return fabs(p) < 65536. ? fma(fabs(p), 8.9e-16, 2.0e-12) : 0.; }

// The largest value below x (IEEE nextafter towards -inf; x finite): "s >= x" is "s > next_below(x)".
template <typename T>
__device__ __forceinline__ T next_below(const T x)
{
    if (x == (T)0) return -NumTraits<T>::from_orderable(NumTraits<T>::orderable((T)0) + 1);     // -denorm_min (covers -0.0 as well)
    return NumTraits<T>::from_orderable(NumTraits<T>::orderable(x) - 1);
}

// Producer: one thread runs the TMA ring over (item tile, k chunk).
template <typename T, int S, int BK>
__device__ __forceinline__ void tma_producer_role(const ScoreSelectParams<T>& P, T* As, T* Bs, const unsigned bar_full, const unsigned bar_empty,
                                                  const int KC, const int total, const int tile0)
{
    constexpr int BN = NumTraits<T>::BN;
    const T* gA = P.At + (size_t)blockIdx.x * P.p_pad * BM;
    int tile = tile0, kc = 0;
    for (int it = 0; it < total; it++) {
        const int s = it % S;
        if (it >= S) mbar_wait(bar_empty + 8 * s, ((it / S) - 1) & 1);
        const int k0 = kc * BK;
        const int kcount = (P.p_pad - k0) < BK ? (P.p_pad - k0) : BK;
        const unsigned bytes_a = (unsigned)(kcount * BM * sizeof(T)), bytes_b = (unsigned)(kcount * BN * sizeof(T));
        mbar_arrive_expect_tx(bar_full + 8 * s, bytes_a + bytes_b);
        tma_bulk_g2s(smem_u32(As + (size_t)s * BK * BM), gA + (size_t)k0 * BM, bytes_a, bar_full + 8 * s);
        tma_bulk_g2s(smem_u32(Bs + (size_t)s * BK * BN), P.Bt + ((size_t)tile * P.p_pad + k0) * BN, bytes_b, bar_full + 8 * s);
        if (++kc == KC) { kc = 0; tile++; }
    }
}

// break_ties_with_noise: a held-out entry the noise can move takes a pass of its own -- its rank count, and the candidates of the
// tile inside [p - reach, p + reach] (auc_near: >= 2 over the catalogue = the noise decides a rank of this user, api.cu).
template <typename T>
__device__ __noinline__ void auc_count_banded(const ScoreSelectParams<T>& P, const T* __restrict__ src, const size_t e, const T p,
                                              const int colp)
{
    constexpr int BN = NumTraits<T>::BN;
    const T reach = noise_reach(p);
    const unsigned before1 = P.auc_cnt[e], near0 = P.auc_near[e];
    const T thr3[3] = {colp >= BN ? next_below<T>(p) : p, next_below<T>(p - reach), p + reach};
    unsigned c3[3];
    count_above<3>(src, thr3, c3);
    unsigned ct = c3[0];
    if (colp > 0 && colp < BN)
        for (int x = 0; x < colp; x++) ct += (src[x] == p);
    if (gridDim.y > 1) { atomicAdd(&P.auc_cnt[e], ct); atomicAdd(&P.auc_near[e], c3[1] - c3[2]); return; }
    P.auc_cnt[e] = before1 + ct;
    P.auc_near[e] = near0 + (c3[1] - c3[2]);
}

// The eight counting warps of the rank-counting kernel.  For every item tile:
//   * counting warp cw waits for the score block FMA warp cw staged for its 16 rows and masks (NaN: never above a threshold,
//     ignored by fmin) what is not a candidate -- the train items of rows whose train row intersects the tile (own cursors,
//     lane r <-> row r) and the padding columns of the last tile -- and tracks the smallest candidate score of its rows
//     (the full-order validity rule, hpp:555-562);
//   * the counting warps meet (named barrier): all 128 rows of the tile are staged and masked;
//   * counting: for every held-out entry of the CTA's rows, the candidates of the tile that rank before it -- scoring above
//     it, or equal with a smaller item id (the tie order of the top-K selection).  Tiles wholly before the entry's own item
//     count "s >= score" (as "s > next_below(score)"), tiles after it "s > score"; the item's own tile "s > score" plus the
//     equal scores in the columns before the item.  The held-out entries of the 128 rows form ONE list (pref[r] = entries
//     before row r), cut into work units of up to UN consecutive entries of one row; unit u belongs to counting thread
//     u % 256 for the whole kernel (it alone updates the entries' counters in global memory: plain read-modify-write).
//     A unit is one pass over its row's BN scores, every 16-byte load compared with the unit's thresholds.  The work of the
//     CTA -- the sum of its rows' held-out counts, heavy-tailed per row -- is spread evenly over all 256 counting lanes:
//     with per-warp lists the CTA ran at the pace of its heaviest warp;
//   * every counting warp releases all eight blocks (blk_empty[w] counts eight arrivals).
template <typename T>
__device__ __noinline__ void auc_count_role(const ScoreSelectParams<T>& P, RowState<T>* rs, T* blk_all, int* pref, T* pthr, int* pitem,
                                            const unsigned bar_blkf, const unsigned bar_blke, const int cw, const int lane,
                                            const int tile_u0, const int NT, const int t_begin)
{
    constexpr int BN = NumTraits<T>::BN;
    constexpr int BNP = SmemLayout<T, true>::BNP;
    constexpr int UN = sizeof(T) == 4 ? 4 : 2;                   // entries per work unit
    const bool sliced = gridDim.y > 1;                           // other CTAs count the same entries over other item ranges: atomic adds
    constexpr int NCT = NCWARPS * 32;                            // counting threads
    constexpr int PCAP = NCWARPS * AUC_PCAP;                     // entries staged in shared memory
    const int wrow0 = cw * 16;
    const int tc = cw * 32 + lane;
    T* blk = blk_all + (size_t)cw * 16 * BNP;
    int* upref = pref + BM + 4;                                  // [BM + 1] units before row r (pref: [BM + 1] entries before row r)
    auto count_sync = []() { asm volatile("bar.sync 1, %0;" ::"n"(NCWARPS * 32) : "memory"); };

    if (cw == 0) {                                               // prefix sums over the CTA's 128 rows (4 rows per lane)
        int np[4], nu[4], sp = 0, su = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) { np[i] = rs->npos[4 * lane + i]; nu[i] = (np[i] + UN - 1) / UN; sp += np[i]; su += nu[i]; }
        int ip = sp, iu = su;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int a = __shfl_up_sync(FULL, ip, o), b = __shfl_up_sync(FULL, iu, o);
            if (lane >= o) { ip += a; iu += b; }
        }
        int bp = ip - sp, bu = iu - su;                          // exclusive
#pragma unroll
        for (int i = 0; i < 4; i++) { pref[4 * lane + i] = bp; upref[4 * lane + i] = bu; bp += np[i]; bu += nu[i]; }
        if (lane == 31) { pref[BM] = bp; upref[BM] = bu; }
    }
    count_sync();
    const int total_pos = pref[BM], n_units = upref[BM];
    for (int q = tc; q < (total_pos < PCAP ? total_pos : PCAP); q += NCT) {      // the first PCAP entries: score and item id staged
        int lo = 0, hi = BM - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (pref[mid] <= q) lo = mid; else hi = mid - 1; }
        const size_t e = (size_t)rs->tp0[lo] + (size_t)(q - pref[lo]);
        pthr[q] = P.pos_sorted[e];
        pitem[q] = P.pos_item[e];
    }
    int unit_row[4];                                             // rows of the thread's first four units (further ones are looked up)
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int u = tc + NCT * j;
        int lo = 0, hi = BM - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (upref[mid] <= u) lo = mid; else hi = mid - 1; }
        unit_row[j] = lo;
    }
    // own train cursor of row `lane` of the warp's block (lanes 0..15), minimum of half a row (row lane >> 1, columns (lane & 1) * BN / 2 ...)
    int t_cur = 0, t_end = 0, t_nxt = INT_MAX;
    if (lane < 16 && tile_u0 + wrow0 + lane < P.mb && rs->npos[wrow0 + lane] > 0) {      // (ranked rows have held-out items)
        const int u = P.user0 + rs->urow[wrow0 + lane];
        t_cur = P.trp[u]; t_end = P.trp[u + 1];
        if (t_begin > 0) {
            int lo = t_cur, hi = t_end;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (P.tri[mid] < t_begin * BN) lo = mid + 1; else hi = mid; }
            t_cur = lo;
        }
        if (t_cur < t_end) t_nxt = P.tri[t_cur];
    }
    T rmin = NumTraits<T>::inf();
    // (pointers of the parameter block in registers: through the reference every use is a load from the parameter space)
    const int n_items = P.n;
    const int* const tri_g = P.tri;
    unsigned int* const cnt_g = P.auc_cnt;
    const unsigned int* const near_g = P.auc_near;
    const T* const sorted_g = P.pos_sorted;
    const int* const item_g = P.pos_item;
    count_sync();                                                // (the staged entries are visible)

    for (int tile = 0; tile < NT; tile++) {
        const int item0 = (t_begin + tile) * BN;
        mbar_wait(bar_blkf + 8 * cw, (unsigned)tile & 1u);
        if (lane < 16) {
            T* dst = blk + (size_t)lane * BNP;
            while (t_nxt < item0 + BN) {
                dst[t_nxt - item0] = NumTraits<T>::nan();
                t_cur++;
                t_nxt = t_cur < t_end ? tri_g[t_cur] : INT_MAX;
            }
            if (item0 + BN > n_items)
                for (int x = (n_items > item0 ? n_items - item0 : 0); x < BN; x++) dst[x] = NumTraits<T>::nan();
        }
        __syncwarp();
        const T* half_row = blk + (size_t)(lane >> 1) * BNP + (lane & 1) * (BN / 2);
        constexpr int VEC = 16 / (int)sizeof(T);
        T m0 = NumTraits<T>::inf(), m1 = NumTraits<T>::inf();
#pragma unroll 4
        for (int x = 0; x < BN / 2; x += 2 * VEC) {
            T v[VEC], w[VEC];
            lds_vec(half_row + x, v);
            lds_vec(half_row + x + VEC, w);
#pragma unroll
            for (int e = 0; e < VEC; e++) { m0 = fmin(m0, v[e]); m1 = fmin(m1, w[e]); }     // fmin ignores NaN
        }
        rmin = fmin(rmin, fmin(m0, m1));
        count_sync();                                            // all 128 rows of the tile are staged and masked
        for (int j = 0, u = tc; u < n_units; j++, u += NCT) {
            int row;
            if (j < 4) row = j == 0 ? unit_row[0] : (j == 1 ? unit_row[1] : (j == 2 ? unit_row[2] : unit_row[3]));
            else {
                int lo = 0, hi = BM - 1;
                while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (upref[mid] <= u) lo = mid; else hi = mid - 1; }
                row = lo;
            }
            const int q = pref[row] + UN * (u - upref[row]);                   // first entry of the unit
            const int run = min(pref[row + 1] - q, UN);
            const size_t e0 = (size_t)rs->tp0[row] + (size_t)(q - pref[row]);
            const T* src = blk_all + (size_t)row * BNP;
            // the unit's counters, scores and item ids: unconditional loads (entries past the unit's end re-read its first
            // one), all in flight together -- the counters come from L2, a dependent load per entry cost more than the counting
            unsigned before[UN];
            T thr[UN], eff[UN];
            int col[UN];
#pragma unroll
            for (int t = 0; t < UN; t++) before[t] = sliced ? 0u : cnt_g[e0 + (t < run ? t : 0)];
            if (q + UN <= PCAP) {
#pragma unroll
                for (int t = 0; t < UN; t++) { thr[t] = pthr[q + t]; col[t] = pitem[q + t] - item0; }
            } else {
#pragma unroll
                for (int t = 0; t < UN; t++) { thr[t] = sorted_g[e0 + (t < run ? t : 0)]; col[t] = item_g[e0 + (t < run ? t : 0)] - item0; }
            }
            unsigned banded = 0;                                          // entries within the noise's reach of other candidates: below
#pragma unroll
            for (int t = 0; t < UN; t++) {
                bool on = t < run;
                if (on && near_g != nullptr && noise_reach(thr[t]) > (T)0) { banded |= 1u << t; on = false; }
                if (!on) col[t] = 0;
                eff[t] = !on ? NumTraits<T>::inf() : (col[t] >= BN ? next_below<T>(thr[t]) : thr[t]);
            }
            unsigned c[UN];
            count_above<UN>(src, eff, c);
#pragma unroll
            for (int t = 0; t < UN; t++) {
                if (t < run && !((banded >> t) & 1u)) {
                    unsigned ct = c[t];
                    if (col[t] > 0 && col[t] < BN)
                        for (int x = 0; x < col[t]; x++) ct += (src[x] == thr[t]);
                    if (!sliced) cnt_g[e0 + t] = before[t] + ct;
                    else if (ct) atomicAdd(&cnt_g[e0 + t], ct);
                }
            }
            while (banded) {
                const int t = __ffs(banded) - 1;
                banded &= banded - 1;
                auc_count_banded<T>(P, src, e0 + t, t == 0 ? thr[0] : (t == 1 ? thr[1] : (UN > 2 && t == 2 ? thr[UN > 2 ? 2 : 0] : thr[UN - 1])),
                                    (q + t < PCAP ? pitem[q + t] : item_g[e0 + t]) - item0);
            }
        }
        __syncwarp();
        if (lane < NCWARPS) mbar_arrive(bar_blke + 8 * lane);    // this warp is done with all eight blocks of the tile
    }
    // smallest candidate score of every ranked row
    rmin = fmin(rmin, __shfl_xor_sync(FULL, rmin, 1));
    if ((lane & 1) == 0) {
        const int row = wrow0 + (lane >> 1);
        if (tile_u0 + row < P.mb && rs->npos[row] > 0 && rmin != NumTraits<T>::inf())
            atomicMin(&P.umin[P.user0 + rs->urow[row]], NumTraits<T>::orderable(rmin));
    }
}

template <typename T, int C, bool AUC>
__global__ void __launch_bounds__(AUC ? AUC_THREADS : NTHREADS, 1)
score_select_kernel(const __grid_constant__ ScoreSelectParams<T> P)
{
    typedef SmemLayout<T, AUC> L;
    constexpr int S = L::S;
    constexpr int BK = L::BK;
    constexpr int BN = NumTraits<T>::BN;
    constexpr int UM = BM;                           // users of this CTA
    constexpr int NW = NCWARPS;                      // FMA warps
    constexpr int NTHR = AUC ? AUC_THREADS : NTHREADS;
    constexpr int NC = MicroTile<T>::NC;            // item columns per thread

    T* As = reinterpret_cast<T*>(smem_raw + L::a_off);
    T* Bs = reinterpret_cast<T*>(smem_raw + L::b_off);
    RowState<T>* rs = reinterpret_cast<RowState<T>*>(smem_raw + L::rs_off);
    const unsigned bar_full = smem_u32(smem_raw + L::bar_off), bar_empty = bar_full + 8 * S;
    const unsigned bar_blkf = bar_empty + 8 * S, bar_blke = bar_blkf + 8 * NCWARPS;      // AUC: score block of warp w handed over / taken
    constexpr int BNP = L::BNP;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int tile_u0 = blockIdx.x * UM;            // first user (batch-local) of this CTA
    const int KC = (P.p_pad + BK - 1) / BK;
    const int NT_all = (P.n + BN - 1) / BN;
    const int t_begin = (int)((long long)NT_all * blockIdx.y / gridDim.y);          // this CTA's range of item tiles (the whole catalogue unless sliced)
    const int NT = (int)((long long)NT_all * (blockIdx.y + 1) / gridDim.y) - t_begin;
    const int total = NT * KC;
    const size_t slice_off = (size_t)blockIdx.y * (size_t)P.slice_rows;               // first row of this slice's candidate buffers

    // ---- one-time setup: per-row selection state, train cursors, barriers ----
    for (int r = tid; r < UM; r += NTHR) {
        const int ul0 = tile_u0 + r;
        const int ul = (ul0 < P.mb && P.umap != nullptr) ? P.umap[ul0] : ul0;
        const bool ranked = (ul0 < P.mb) && (P.ustatus[P.user0 + ul] == 0);
        rs->urow[r] = ul0 < P.mb ? ul : 0;
        rs->tau[r] = ranked ? -NumTraits<T>::inf() : NumTraits<T>::inf();
        rs->cnt[r] = 0;
        rs->nan[r] = 0;
        int cur = 0, end = 0, tp0 = 0, npos = 0;
        if (ranked) {
            const int u = P.user0 + ul;
            cur = P.trp[u]; end = P.trp[u + 1];
            tp0 = P.tep[u]; npos = P.tep[u + 1] - tp0;
            if (t_begin > 0) {                       // first train item inside this CTA's item range
                int lo = cur, hi = end;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (P.tri[mid] < t_begin * BN) lo = mid + 1; else hi = mid; }
                cur = lo;
            }
        }
        rs->cur_train[r] = cur;
        rs->end_train[r] = end;
        rs->nxt_train[r] = cur < end ? P.tri[cur] : INT_MAX;
        rs->tp0[r] = tp0;
        rs->npos[r] = npos;
    }
    if (tid == 0) {
        for (int s = 0; s < S; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, NW); }
        if (AUC)
            for (int w = 0; w < NCWARPS; w++) { mbar_init(bar_blkf + 8 * w, 1); mbar_init(bar_blke + 8 * w, NCWARPS); }
        mbar_fence_init();
    }
    __syncthreads();   // the only CTA-wide barrier

    if (AUC) {
        // registers to where they are needed (every warp of a group of four executes the same setmaxnreg)
        if (warp >= 2 * NCWARPS) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
            if (warp == 2 * NCWARPS && lane == 0) tma_producer_role<T, S, BK>(P, As, Bs, bar_full, bar_empty, KC, total, t_begin);
            return;
        }
        if (warp >= NCWARPS) {
            if (sizeof(T) == 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
            else asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
            auc_count_role<T>(P, rs, reinterpret_cast<T*>(smem_raw + L::blk_off), reinterpret_cast<int*>(smem_raw + L::pref_off),
                              reinterpret_cast<T*>(smem_raw + L::pthr_off), reinterpret_cast<int*>(smem_raw + L::pitem_off),
                              bar_blkf, bar_blke, warp - NCWARPS, lane, tile_u0, NT, t_begin);
            return;
        }
        if (sizeof(T) == 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 152;");
        else asm volatile("setmaxnreg.inc.sync.aligned.u32 160;");
    } else if (warp == NCWARPS) {
        if (lane == 0) tma_producer_role<T, S, BK>(P, As, Bs, bar_full, bar_empty, KC, total, t_begin);
        return;
    }

    // ===================== compute warps =====================
    const int ly = lane >> 4, lx = lane & 15;
    const int wrow0 = warp * 16;                    // first CTA row of this warp
    T* blk = reinterpret_cast<T*>(smem_raw + L::blk_off) + (size_t)warp * 16 * BNP;   // AUC only: [16][BNP]
    MicroTile<T> mt;
    typename MicroTile<T>::Frag frag;               // operand registers of one k step
    int it = 0;
    for (int tile = 0; tile < NT; tile++) {
        const int item0 = (t_begin + tile) * BN;
        mt.zero();
        for (int kc = 0; kc < KC; kc++, it++) {
            const int s = it % S;
            mbar_wait(bar_full + 8 * s, (it / S) & 1);
            const int k0 = kc * BK;
            const int kcount = (P.p_pad - k0) < BK ? (P.p_pad - k0) : BK;      // a multiple of KPAD
            const T* sA = As + (size_t)s * BK * UM + wrow0;
            const T* sB = Bs + (size_t)s * BK * BN;
            for (int kk0 = 0; kk0 < kcount; kk0 += KPAD) {
#pragma unroll
                for (int kk = 0; kk < KPAD; kk++) {
                    MicroTile<T>::load(frag, sA + (kk0 + kk) * UM, sB + (kk0 + kk) * BN, ly, lx);
                    mt.compute(frag);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + 8 * s);
        }

        // ---------------- epilogue of item tile `tile` (warp-private) ----------------
        T biasv[NC];
        if (P.bias != nullptr) {
#pragma unroll
            for (int c = 0; c < NC; c++) biasv[c] = P.bias[item0 + lx * 4 + (c & 3) + (c >> 2) * 64];
        }
        bool inserted = false;
        if (AUC && tile > 0) mbar_wait(bar_blke + 8 * warp, (unsigned)(tile - 1) & 1u);      // the counting warp is done with the previous block
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int row_l = ly * 4 + (i & 3) + (i >> 2) * 8;
            const int row = wrow0 + row_l;
            T s[NC];
            mt.row(i, s);
            if (P.bias != nullptr) {
#pragma unroll
                for (int c = 0; c < NC; c++) s[c] += biasv[c];
            }
            const T tau = rs->tau[row];
            T m = max_nan(max_nan(s[0], s[1]), max_nan(s[2], s[3]));
            if (NC == 8) m = max_nan(m, max_nan(max_nan(s[NC - 4], s[NC - 3]), max_nan(s[NC - 2], s[NC - 1])));
            if (!(m < tau)) {
                T* cs = P.cand_score + (slice_off + (size_t)rs->urow[row]) * C;
                int* ci = P.cand_item + (slice_off + (size_t)rs->urow[row]) * C;
                row_slow<T>(rs, cs, ci, P.tri, P.n, tau, row, item0 + lx * 4, item0 + BN, s[0], s[1], s[2], s[3]);
                if (NC == 8)
                    row_slow<T>(rs, cs, ci, P.tri, P.n, tau, row, item0 + 64 + lx * 4, item0 + BN, s[NC - 4], s[NC - 3], s[NC - 2], s[NC - 1]);
                inserted = true;
            }
            if (AUC) {
                T* dst = blk + (size_t)row_l * BNP + lx * 4;
                sts4(dst, &s[0]);
                if (NC == 8) sts4(dst + 64, &s[NC - 4]);
            }
        }
        __syncwarp();
        if (AUC && lane == 0) mbar_arrive(bar_blkf + 8 * warp);      // the tile's score block is the counting warp's now

        // advance the train cursors of the warp's rows past this tile (lanes 0..15, rare)
        if (lane < 16) {
            const int row = wrow0 + lane;
            int nxt = rs->nxt_train[row];
            if (nxt < item0 + BN) {
                int cur = rs->cur_train[row];
                const int end = rs->end_train[row];
                while (cur < end && (nxt = P.tri[cur]) < item0 + BN) cur++;
                rs->cur_train[row] = cur;
                rs->nxt_train[row] = cur < end ? nxt : INT_MAX;
            }
        }
        // cut back the buffers of this warp that passed the trigger (rare after the first few tiles)
        if (__any_sync(FULL, inserted)) {
            const int nv_l = lane < 16 ? rs->cnt[wrow0 + lane] : 0;
            unsigned need = __ballot_sync(FULL, nv_l > C - BN);
            while (need) {
                const int r = __ffs(need) - 1;
                need &= need - 1;
                const int row = wrow0 + r;
                const size_t base = (slice_off + (size_t)rs->urow[row]) * C;
                compact_user<T, C>(P.cand_score + base, P.cand_item + base, rs->cnt[row], P.K, lane, &rs->tau[row], &rs->cnt[row]);
            }
        }
        __syncwarp();
    }

    // ---- leave the best min(cnt, K) candidates of every user at the head of its buffer ----
    for (int r = 0; r < 16; r++) {
        const int row = wrow0 + r;
        if (tile_u0 + row < P.mb) {
            const int ul = rs->urow[row];
            const size_t base = (slice_off + (size_t)ul) * C;
            compact_user<T, C>(P.cand_score + base, P.cand_item + base, rs->cnt[row], P.K, lane, &rs->tau[row], &rs->cnt[row]);
            if (lane == 0) {
                P.cand_count[slice_off + ul] = rs->cnt[row];
                if (rs->nan[row]) atomicOr(&P.uflags[P.user0 + ul], 1);
            }
        }
    }
}

// One warp per user: order the (<= K <= 32*E) candidates score_select_kernel left at the head of the
// user's buffer (score descending, ties by ascending item id).
template <typename T, int E>
__global__ void rank_topk_kernel(T* __restrict__ cand_score, int* __restrict__ cand_item, const int* __restrict__ cand_count,
                                 const int C, const int mb)
{
    const int lane = threadIdx.x & 31;
    const int ul = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (ul >= mb) return;
    const int nv = cand_count[ul];
    T* cs = cand_score + (size_t)ul * C;
    int* ci = cand_item + (size_t)ul * C;
    T s[E];
    int it[E];
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int idx = e * 32 + lane;
        const bool v = idx < nv;
        s[e] = v ? cs[idx] : -NumTraits<T>::inf();
        it[e] = v ? ci[idx] : INT_MAX;
    }
    warp_sort_ranked<T, E>(s, it, lane);
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int idx = e * 32 + lane;
        if (idx < nv) { cs[idx] = s[e]; ci[idx] = it[e]; }
    }
}

// Item slices (ScoreSelectParams::slice_rows): join the heads the slices left for every user into slice 0's row -- the best K of the
// catalogue are among the best K of every range.  One warp per user.
template <typename T>
__global__ void merge_slices_kernel(T* __restrict__ cand_score, int* __restrict__ cand_item, int* __restrict__ cand_count,
                                    const int C, const int mb, const int slices, const int slice_rows)
{
    const int lane = threadIdx.x & 31;
    const int ul = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (ul >= mb) return;
    int total = cand_count[ul];
    for (int y = 1; y < slices; y++) {
        const size_t row = (size_t)y * slice_rows + ul;
        const int c = cand_count[row];
        for (int i = lane; i < c; i += 32) {
            cand_score[(size_t)ul * C + total + i] = cand_score[row * C + i];
            cand_item[(size_t)ul * C + total + i] = cand_item[row * C + i];
        }
        total += c;
    }
    __syncwarp();
    if (lane == 0) cand_count[ul] = total;
}

}  // namespace rmb
