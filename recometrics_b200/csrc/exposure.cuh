// exposure.cuh -- item exposure of the ranked top-K lists: how many evaluated users have each item in their list, and the
// catalogue statistics derived from those counts (coverage, Gini index, Shannon entropy).
//
//   exposure_count_kernel   one batch's ranked lists into a call-lifetime uint32 histogram [n] (+ the counted users in [n])
//   exposure_widen_kernel   the histogram widened to int64 for the caller
//   exposure_stats_host     the statistics, on the host, from the integer counts only: a single-GPU call, a multi-GPU call
//                           and a process-sharded run (counts summed over ranks) give bit-identical statistics
#pragma once
#include <cmath>
#include <cstdint>
#include <limits>
#include <vector>
#include <algorithm>

#include "../../include/recometrics_b200.h"

namespace rmb {

constexpr int EXPOSURE_THREADS = 256;

// Lane = user, loop over ranks.  In a popularity-heavy model the same few items head almost every list: at every rank
// __match_any_sync groups the lanes holding the same item and the group's first lane adds the group's size, so a hot item
// costs one atomic per warp and rank instead of one per user.  `items`: the batch's ranked rows (row pitch C, a multiple of
// 4, 16-byte aligned); `list_len`: each user's list length as user_metrics_kernel decided it (0: the user is not counted).
__global__ void __launch_bounds__(EXPOSURE_THREADS) exposure_count_kernel(const int* __restrict__ items, const int C,
                                                                           const int* __restrict__ list_len, const int nb,
                                                                           unsigned* __restrict__ hist, const int n)
{
    const int lane = threadIdx.x & 31;
    const int u = blockIdx.x * EXPOSURE_THREADS + threadIdx.x;
    const int len = u < nb ? list_len[u] : 0;                  // (lanes past the batch take part in the warp's votes)
    const unsigned counted = __ballot_sync(0xffffffffu, len > 0);
    if (lane == 0 && counted) atomicAdd(&hist[n], (unsigned)__popc(counted));
    const int wlen = (int)__reduce_max_sync(0xffffffffu, (unsigned)len);
    const int4* row = reinterpret_cast<const int4*>(items + (size_t)(u < nb ? u : 0) * C);
    for (int r = 0; r < wlen; r += 4) {
        int4 v = make_int4(-1, -1, -1, -1);
        if (r < len) v = row[r >> 2];
        const int it[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int item = (r + j < len) ? it[j] : -1;
            const unsigned grp = __match_any_sync(0xffffffffu, item);
            if (item >= 0 && lane == __ffs(grp) - 1) atomicAdd(&hist[item], (unsigned)__popc(grp));
        }
    }
}

__global__ void exposure_widen_kernel(const unsigned* __restrict__ hist, const int n, long long* __restrict__ out)
{
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) out[j] = (long long)hist[j];
}

// Statistics of item counts c[0..n) (see DESIGN.md, "Item exposure"): entries S = sum c, items_covered, coverage, the Gini
// index over all n items (unrecommended items count as 0) and the Shannon entropy in bits.  The items are grouped by count
// value, ascending; with f_v items of count v whose first has 1-based rank s_v in ascending order, the Gini numerator
// sum_i (2i - n - 1) c_(i) is sum_v f_v v (2 s_v + f_v - n - 2), exact in 128-bit integers, divided once in double.
// Returns false (and leaves *out alone) for n <= 0, a negative count or a total beyond int64.
inline bool exposure_stats_host(const int64_t* c, const int n, rmb200_exposure_t* out)
{
    if (n <= 0 || !c) return false;
    int64_t vmax = 0, covered = 0;
    __int128 S = 0;
    for (int j = 0; j < n; j++) {
        if (c[j] < 0) return false;
        if (c[j] > vmax) vmax = c[j];
        covered += c[j] > 0;
        S += c[j];
    }
    if (S > (__int128)std::numeric_limits<int64_t>::max()) return false;
    // distinct values ascending with their multiplicities: counts of counts where the largest count is small (a call's
    // counts are at most its users), else a sort of the non-zero counts; both give the same sequence
    std::vector<std::pair<int64_t, int64_t>> groups;            // (v, f_v), v > 0
    if (vmax <= 4 * (int64_t)n + 1024) {
        std::vector<int64_t> f((size_t)vmax + 1, 0);
        for (int j = 0; j < n; j++) f[(size_t)c[j]]++;
        for (int64_t v = 1; v <= vmax; v++) if (f[(size_t)v]) groups.emplace_back(v, f[(size_t)v]);
    } else {
        std::vector<int64_t> s;
        s.reserve((size_t)covered);
        for (int j = 0; j < n; j++) if (c[j] > 0) s.push_back(c[j]);
        std::sort(s.begin(), s.end());
        for (size_t i = 0; i < s.size();) {
            size_t e = i;
            while (e < s.size() && s[e] == s[i]) e++;
            groups.emplace_back(s[i], (int64_t)(e - i));
            i = e;
        }
    }
    out->entries = (int64_t)S;
    out->items_covered = covered;
    out->coverage = (double)covered / (double)n;
    if (S == 0) {
        out->gini = out->entropy_bits = std::numeric_limits<double>::quiet_NaN();
        return true;
    }
    __int128 num = 0;
    int64_t s_v = (int64_t)n - covered + 1;                      // the zeros come first and add nothing
    double vlogv = 0.0;
    for (const auto& g : groups) {
        const int64_t v = g.first, f = g.second;
        num += (__int128)(f * v) * (__int128)(2 * s_v + f - (int64_t)n - 2);
        vlogv += (double)f * (double)v * std::log2((double)v);
        s_v += f;
    }
    out->gini = (double)num / (double)((__int128)n * S);
    const double h = std::log2((double)S) - vlogv / (double)S;
    out->entropy_bits = h > 0.0 ? h : 0.0;
    return true;
}

}  // namespace rmb
