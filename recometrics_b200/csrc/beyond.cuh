// beyond.cuh -- per-user beyond-accuracy metrics of the ranked top-K lists: Novelty@K, AvgPop@K and ILD@K (intra-list
// diversity), plus the item popularity they need.
//
//   item_popularity_kernel   column count of a CSR row range into a uint32 histogram [n] (widened by exposure_widen_kernel)
//   popularity_table_kernel  per item {-log2((pop + 1) / (U + 1)), pop} in double, once per call; flags counts outside [0, U]
//   unit_rows_kernel         unit-row image of B (item factors only, no bias), row pitch padded to 16 bytes, norm in double
//   beyond_accuracy_kernel   one warp per user of a batch, reading the ranked rows and list lengths of the metrics step
//
// Definitions (user's list j_1..j_L, L = list_len as user_metrics_kernel decides it; L = 0: every output is the NaN value):
//   Novelty@i = (1/i) sum_{r<=i} -log2((pop_{j_r} + 1) / (U + 1))      AvgPop@i = (1/i) sum_{r<=i} pop_{j_r}
//   ILD@i     = 1 - 2 P_i / (i (i - 1)),  u_r = b_{j_r} / ||b_{j_r}|| (a zero row gives u_r = 0),
//               s_0 = 0, P_0 = 0,  P_r = P_{r-1} + u_r . s_{r-1},  s_r = s_{r-1} + u_r       (ILD@1 is NaN)
// i.e. the mean pairwise cosine distance of the first i items in O(L p) per user; every new pair enters P as itself (no
// ||s||^2 - L cancellation).  Every sum is accumulated in double in rank order and cast to T once; the per-rank dot product is
// reduced across the warp by a fixed butterfly.  So column K of a cumulative row is bit-identical to the non-cumulative value,
// and a user's values do not depend on how the users are split into batches, shards or devices.
#pragma once
#include <cstdint>

namespace rmb {

constexpr int BEYOND_WARPS = 8;            // users (warps) per block of beyond_accuracy_kernel
constexpr int POPULARITY_THREADS = 256;

// Counts every entry idx[0..nnz) of a CSR row range.  __match_any_sync groups the lanes that hold the same item (a hot item
// of a skewed catalogue costs one atomic per warp, not one per entry); entries outside [0, n) are not counted.
__global__ void __launch_bounds__(POPULARITY_THREADS) item_popularity_kernel(const int* __restrict__ idx, const long long nnz,
                                                                              unsigned* __restrict__ hist, const int n)
{
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < nnz; i0 += stride) {   // warp-uniform
        const long long i = i0 + lane;
        int item = i < nnz ? idx[i] : -1;
        if (item >= n) item = -1;
        const unsigned grp = __match_any_sync(0xffffffffu, item);
        if (item >= 0 && lane == __ffs(grp) - 1) atomicAdd(&hist[item], (unsigned)__popc(grp));
    }
}

// {self-information, popularity} of every item, from int64 counts over U users; *bad = 1 when a count lies outside [0, U]
__global__ void popularity_table_kernel(const long long* __restrict__ pop, const int n, const long long U,
                                        double2* __restrict__ tab, int* __restrict__ bad)
{
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const long long c = pop[j];
        if (c < 0 || c > U) *bad = 1;
        tab[j] = make_double2(-log2((double)(c + 1) / (double)(U + 1)), (double)c);
    }
}

// One warp per item row: u = b / ||b|| in T, zero past k and for a zero row
template <typename T>
__global__ void unit_rows_kernel(const T* __restrict__ B, const size_t ldb, const int n, const int k, T* __restrict__ U, const int pitch)
{
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= n) return;
    const T* b = B + (size_t)j * ldb;
    double ss = 0.;
    for (int c = lane; c < k; c += 32) ss += (double)b[c] * (double)b[c];
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const double norm = sqrt(ss);
    T* u = U + (size_t)j * pitch;
    for (int c = lane; c < pitch; c += 32) u[c] = (c < k && norm > 0.) ? (T)((double)b[c] / norm) : (T)0;
}

template <typename T> struct Vec16;                          // 16 bytes of T
template <> struct Vec16<float> { using type = float4; };
template <> struct Vec16<double> { using type = double2; };

template <typename T>
struct BeyondParams {
    const int* items; int C;               // the batch's ranked rows (row pitch C)
    const int* list_len;                   // [nb]: L of every user of the batch (0: undefined)
    int nb, K, cumulative;
    const double2* pop;                    // [n] {self-information, popularity}; null: neither Novelty nor AvgPop requested
    const T* unit; int pitch;              // [n][pitch] unit rows of B; null: ILD not requested
    T *nov, *avgpop, *ild;                 // the batch's rows (row stride K if cumulative else 1); null: not requested
    T nan_value;
};

// Lane l owns 16-byte chunks l, l + 32, ... (NCH of them) of a unit row and the matching components of s, in double.  The
// row loads of the next D ranks are issued before a rank is processed (they do not depend on s): the kernel is bound by the
// bytes it gathers, so several rows per warp are kept in flight.
template <typename T, int NCH>
__global__ void __launch_bounds__(BEYOND_WARPS * 32, NCH == 1 ? 0 : 1) beyond_accuracy_kernel(const __grid_constant__ BeyondParams<T> P)
{
    using V16 = typename Vec16<T>::type;
    constexpr int V = 16 / (int)sizeof(T);
    constexpr int D = NCH >= 4 ? 1 : 4 / NCH;                // ranks in flight
    const int lane = threadIdx.x & 31;
    const int ul = blockIdx.x * BEYOND_WARPS + (threadIdx.x >> 5);
    if (ul >= P.nb) return;                                  // the whole warp leaves
    const int K = P.K;
    const size_t rs = P.cumulative ? (size_t)K : 1;
    const T NaN = P.nan_value;
    T* nov = P.nov ? P.nov + (size_t)ul * rs : nullptr;
    T* avg = P.avgpop ? P.avgpop + (size_t)ul * rs : nullptr;
    T* ild = P.ild ? P.ild + (size_t)ul * rs : nullptr;
    const int len = P.list_len[ul];
    // undefined users, and the columns past the list (none under the eligibility rules, which make L = K)
    for (int c = (len > 0 ? len : 0) + lane; c < (int)rs; c += 32) {
        if (nov) nov[c] = NaN;
        if (avg) avg[c] = NaN;
        if (ild) ild[c] = NaN;
    }
    if (len <= 0) return;
    const int* ci = P.items + (size_t)ul * P.C;

    if (nov || avg) {      // lane t of a round holds rank base + t; the sums run through the ranks in order
        double sn = 0., sp = 0.;
        for (int base = 0; base < len; base += 32) {
            const int r = base + lane;
            const double2 v = r < len ? P.pop[ci[r]] : make_double2(0., 0.);
            const int cnt = len - base < 32 ? len - base : 32;
            double my_n = 0., my_p = 0.;
            for (int t = 0; t < cnt; t++) {
                sn += __shfl_sync(0xffffffffu, v.x, t);
                sp += __shfl_sync(0xffffffffu, v.y, t);
                if (t == lane) { my_n = sn; my_p = sp; }
            }
            if (P.cumulative && r < len) {
                if (nov) nov[r] = (T)(my_n / (double)(r + 1));
                if (avg) avg[r] = (T)(my_p / (double)(r + 1));
            }
        }
        if (!P.cumulative && lane == 0) {
            if (nov) *nov = (T)(sn / (double)len);
            if (avg) *avg = (T)(sp / (double)len);
        }
    }

    if (ild) {
        const int nvec = P.pitch / V;                        // 16-byte chunks per unit row
        double s[NCH][V];
        V16 buf[D][NCH];
#pragma unroll
        for (int c = 0; c < NCH; c++)
#pragma unroll
            for (int e = 0; e < V; e++) s[c][e] = 0.;
        auto load = [&](const int r, V16* b) {
            if (r >= len) return;
            const V16* row = reinterpret_cast<const V16*>(P.unit + (size_t)ci[r] * P.pitch);
#pragma unroll
            for (int c = 0; c < NCH; c++) {
                const int x = lane + 32 * c;
                if (x < nvec) b[c] = row[x];
                else b[c] = V16();
            }
        };
#pragma unroll
        for (int d = 0; d < D; d++) load(d, buf[d]);
        double Psum = 0.;
        T mine = NaN;                                        // column base + lane of the current round of 32 ranks
        for (int r0 = 0; r0 < len; r0 += D) {
#pragma unroll
            for (int d = 0; d < D; d++) {
                const int r = r0 + d;
                if (r < len) {
                    double u[NCH][V];
#pragma unroll
                    for (int c = 0; c < NCH; c++) {
                        const T* e = reinterpret_cast<const T*>(&buf[d][c]);
#pragma unroll
                        for (int q = 0; q < V; q++) u[c][q] = (double)e[q];
                    }
                    load(r + D, buf[d]);                     // the next rows go out before this rank's arithmetic
                    double dot = 0.;
#pragma unroll
                    for (int c = 0; c < NCH; c++)
#pragma unroll
                        for (int q = 0; q < V; q++) dot = fma(u[c][q], s[c][q], dot);
                    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
                    Psum += dot;
#pragma unroll
                    for (int c = 0; c < NCH; c++)
#pragma unroll
                        for (int q = 0; q < V; q++) s[c][q] += u[c][q];
                    if (P.cumulative) {
                        const int i = r + 1;
                        const T val = i > 1 ? (T)(1. - 2. * Psum / ((double)i * (double)(i - 1))) : NaN;
                        if (lane == (r & 31)) mine = val;
                        if ((r & 31) == 31 || r == len - 1) { if (lane <= (r & 31)) ild[(r & ~31) + lane] = mine; }
                    }
                }
            }
        }
        if (!P.cumulative && lane == 0)
            *ild = len > 1 ? (T)(1. - 2. * Psum / ((double)len * (double)(len - 1))) : NaN;
    }
}

}  // namespace rmb
