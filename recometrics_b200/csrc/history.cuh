// history.cuh -- per-user Unexpectedness@K and Serendipity@K of the ranked top-K lists: how far each listed item lies from
// the user's own training history (Kaminskas & Bridge 2016; Microsoft Recommenders' user_serendipity with cosine similarity
// over B's rows, relevance = held-out membership).
//
//   history_distance_kernel  one warp per user of a batch, reading the ranked rows and list lengths of the metrics step, the
//                            user's X_train row and X_test row, and the unit-row image of B (beyond.cuh, unit_rows_kernel)
//
// Definitions (user's list j_1..j_L, L = list_len as user_metrics_kernel decides it; H_u = the stored entries of the user's
// X_train row, T_u = |H_u|; u_j = b_j / ||b_j|| as for ILD, a zero row gives u_j = 0):
//   c_u = sum_{t in H_u} u_t (in the row's order)       sim_r = (u_{j_r} . c_u) / T_u       rel_r = [j_r stored in X_test's row]
//   Unexpectedness@i = (1/i) sum_{r<=i} (1 - sim_r)       Serendipity@i = (1/i) sum_{r<=i} rel_r (1 - sim_r)
// A user is defined when L > 0 and T_u > 0; every other user gets the NaN value in both rows.  Entries of the history outside
// [0, n) add nothing to c_u (they still count in T_u).  Every sum is accumulated in double in a fixed order and cast to T once;
// the per-rank dot product is reduced across the warp by the fixed butterfly of beyond_accuracy_kernel.  So column K of a
// cumulative row is bit-identical to the non-cumulative value, and a user's values do not depend on how the users are split
// into batches, shards or devices (a user's X_train row lies wholly in its shard).
#pragma once
#include "beyond.cuh"

namespace rmb {

constexpr int HISTORY_WARPS = 8;           // users (warps) per block of history_distance_kernel

template <typename T>
struct HistoryParams {
    const int* items; int C;               // the batch's ranked rows (row pitch C)
    const int* list_len;                   // [nb]: L of every user of the batch (0: undefined)
    int nb, user0, n, K, cumulative;       // user0: the batch's first user in the shard-local CSR arrays
    const int *trp, *tri;                  // X_train rows (tri null: no entry at all)
    const int *tep, *tei;                  // X_test rows, sorted
    const T* unit; int pitch;              // [n][pitch] unit rows of B
    T *unexp, *seren;                      // the batch's rows (row stride K if cumulative else 1); null: not requested
    T nan_value;
};

// Lane l owns 16-byte chunks l, l + 32, ... (NCH of them) of a unit row and the matching components of c_u, in double.  The
// rows of the history and then of the list form one stream: the loads of the next D rows are issued before a row is summed
// into c_u or dotted with it, so the gather of the first listed rows overlaps the end of the history.  (NCH = 1 asks for two
// blocks per SM: left to itself, ptxas targets 80 registers there and spills.)
template <typename T, int NCH>
__global__ void __launch_bounds__(HISTORY_WARPS * 32, NCH == 1 ? 2 : 1) history_distance_kernel(const __grid_constant__ HistoryParams<T> P)
{
    using V16 = typename Vec16<T>::type;
    constexpr int V = 16 / (int)sizeof(T);
    constexpr int D = NCH >= 4 ? 1 : 4 / NCH;                // rows in flight
    const int lane = threadIdx.x & 31;
    const int ul = blockIdx.x * HISTORY_WARPS + (threadIdx.x >> 5);
    if (ul >= P.nb) return;                                  // the whole warp leaves
    const int u = P.user0 + ul;
    const size_t rs = P.cumulative ? (size_t)P.K : 1;
    const T NaN = P.nan_value;
    T* ue = P.unexp ? P.unexp + (size_t)ul * rs : nullptr;
    T* se = P.seren ? P.seren + (size_t)ul * rs : nullptr;
    const int len = P.list_len[ul];
    const int h0 = P.tri ? P.trp[u] : 0;
    const int nh = P.tri ? P.trp[u + 1] - h0 : 0;            // T_u
    const bool defined = len > 0 && nh > 0;
    // undefined users, and the columns past the list (none under the eligibility rules, which make L = K)
    for (int c = (defined ? len : 0) + lane; c < (int)rs; c += 32) {
        if (ue) ue[c] = NaN;
        if (se) se[c] = NaN;
    }
    if (!defined) return;
    const int* ci = P.items + (size_t)ul * P.C;
    const int* hi = P.tri + h0;
    const int t0 = P.tep[u], npos = P.tep[u + 1] - t0;
    const int* ti = P.tei + t0;
    const int total = nh + len;                              // rows 0..nh-1: the history; nh..total-1: the list

    const int nvec = P.pitch / V;                            // 16-byte chunks per unit row
    double c[NCH][V];
    V16 buf[D][NCH];
#pragma unroll
    for (int q = 0; q < NCH; q++)
#pragma unroll
        for (int e = 0; e < V; e++) c[q][e] = 0.;
    auto load = [&](const int r, V16* b) {
        if (r >= total) return;
        const int j = r < nh ? hi[r] : ci[r - nh];
        const bool ok = (unsigned)j < (unsigned)P.n;
        const V16* row = reinterpret_cast<const V16*>(P.unit + (size_t)(ok ? j : 0) * P.pitch);
#pragma unroll
        for (int q = 0; q < NCH; q++) {
            const int x = lane + 32 * q;
            if (ok && x < nvec) b[q] = row[x];
            else b[q] = V16();
        }
    };
#pragma unroll
    for (int d = 0; d < D; d++) load(d, buf[d]);
    double su = 0., ss = 0.;
    unsigned rel = 0u;                                       // held-out membership of the current round of 32 ranks
    T mine_u = NaN, mine_s = NaN;                            // column base + lane of the current round
    for (int r0 = 0; r0 < total; r0 += D) {
#pragma unroll
        for (int d = 0; d < D; d++) {
            const int r = r0 + d;
            if (r < total) {
                double v[NCH][V];
#pragma unroll
                for (int q = 0; q < NCH; q++) {
                    const T* e = reinterpret_cast<const T*>(&buf[d][q]);
#pragma unroll
                    for (int w = 0; w < V; w++) v[q][w] = (double)e[w];
                }
                load(r + D, buf[d]);                         // the next rows go out before this row's arithmetic
                if (r < nh) {
#pragma unroll
                    for (int q = 0; q < NCH; q++)
#pragma unroll
                        for (int w = 0; w < V; w++) c[q][w] += v[q][w];
                } else {
                    const int k = r - nh;                    // rank, 0-based
                    if ((k & 31) == 0) {                     // one listed id per lane, binary-searched in the sorted test row
                        const int kk = k + lane;
                        bool hit = false;
                        if (kk < len) {
                            const int item = ci[kk];
                            int lo = 0, hb = npos;
                            while (lo < hb) { const int mid = (lo + hb) >> 1; if (ti[mid] < item) lo = mid + 1; else hb = mid; }
                            hit = lo < npos && ti[lo] == item;
                        }
                        rel = __ballot_sync(0xffffffffu, hit);
                    }
                    double dot = 0.;
#pragma unroll
                    for (int q = 0; q < NCH; q++)
#pragma unroll
                        for (int w = 0; w < V; w++) dot = fma(v[q][w], c[q][w], dot);
                    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
                    const double dist = 1. - dot / (double)nh;
                    su += dist;
                    if ((rel >> (k & 31)) & 1u) ss += dist;
                    if (P.cumulative) {
                        const double i = (double)(k + 1);
                        if (lane == (k & 31)) { mine_u = (T)(su / i); mine_s = (T)(ss / i); }
                        if ((k & 31) == 31 || k == len - 1) {
                            if (lane <= (k & 31)) {
                                if (ue) ue[(k & ~31) + lane] = mine_u;
                                if (se) se[(k & ~31) + lane] = mine_s;
                            }
                        }
                    }
                }
            }
        }
    }
    if (!P.cumulative && lane == 0) {
        if (ue) *ue = (T)(su / (double)len);
        if (se) *se = (T)(ss / (double)len);
    }
}

}  // namespace rmb
