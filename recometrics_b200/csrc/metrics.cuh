// metrics.cuh -- per-user metrics from the ranked top-K, the held-out row and the rank buckets.
//
// One warp per user; every accumulator is added up in rank order, in double, with the same
// operations as the reference so that -- given the same ranking -- the results are
// bit-identical:
//   validity of the ranking        /root/reference/src/recometrics.hpp:537-563
//   top-K walk                      :605-708   (hits, AP, DCG, RR; cumulative writes :625-635)
//   post-hoc NaN rules              :750-788
//   ROC-AUC / PR-AUC                :795-865   (from rank counts instead of a sorted walk)
//   NDCG normalisation              :868-961   (incl. the frozen cumulative tail :951-956)
// log2(ix+2) comes from a host table (glibc values) so the discount factors match the host's.
#pragma once
#include "score_select.cuh"

namespace rmb {

template <typename T>
struct MetricsParams {
    int n, K, C, user0, mb, cumulative;
    int want_roc, want_pr, count_ranks;   // count_ranks: the rank-counting pass ran
    int noise;                            // break_ties_with_noise: validity rules of the noise branch (hpp:516-528)
    const int* trp; const int* tep; const int* tei; const T* tev;
    const int* ustatus; const int* uflags;
    const T* cand_score; const int* cand_item; const int* cand_count;
    const unsigned int* auc_cnt; const unsigned long long* umin; const int* pos_perm;
    const double* log2tab;                // [K]: log2(ix + 2)
    T nan_value;
    // outputs, already offset to the batch's first user (row stride: K if cumulative else 1)
    T *p, *tp, *r, *ap, *tap, *ndcg, *hit, *rr, *roc, *pr;
    int* status_out;                      // optional, offset to the batch
    int* topk_items; T* topk_scores;      // optional [mb][K], offset to the batch
    long long* pos_rank;                  // optional [nnz_test] (absolute)
    int* list_len;                        // optional [mb]: length of the user's ranked list, 0 where it is undefined (exposure.cuh, beyond.cuh)
};

constexpr int METRICS_WARPS = 8;           // users (warps) per block of user_metrics_kernel
constexpr unsigned FULL_WARP = 0xffffffffu;

template <typename T>
__device__ __forceinline__ void fill_row(T* out, const size_t ul, const int K, const int cumulative, const T v, const int lane)
{
    if (!out) return;
    if (!cumulative) { if (lane == 0) out[ul] = v; }
    else for (int c = lane; c < K; c += 32) out[ul * (size_t)K + c] = v;
}

template <typename T>
__device__ void all_nan(const MetricsParams<T>& P, const size_t ul, const int lane)
{
    fill_row(P.p, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.tp, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.r, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.ap, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.tap, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.ndcg, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.hit, ul, P.K, P.cumulative, P.nan_value, lane);
    fill_row(P.rr, ul, P.K, P.cumulative, P.nan_value, lane);
    if (lane == 0) {
        if (P.roc) P.roc[ul] = P.nan_value;
        if (P.pr) P.pr[ul] = P.nan_value;
    }
}

__device__ __forceinline__ int warp_sum(int v)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_WARP, v, o);
    return v;
}

template <typename T>
__device__ __forceinline__ T warp_max(T v)      // ordinary '>' (no NaNs reach it)
{
    for (int o = 16; o > 0; o >>= 1) { const T w = __shfl_xor_sync(FULL_WARP, v, o); if (w > v) v = w; }
    return v;
}

// One WARP per user.  Rank ix of the walk and column ix of a cumulative row belong to lane ix % 32: the membership
// tests, the divisions and the row writes run in parallel, while every accumulator (hits, AP, DCG, IDCG) is still
// added up in rank order, in double, term by term -- the reference's sequence of operations, hence its bits.
template <typename T>
__global__ void __launch_bounds__(METRICS_WARPS * 32) user_metrics_kernel(const __grid_constant__ MetricsParams<T> P)
{
    const int lane = threadIdx.x & 31;
    const int uli = blockIdx.x * METRICS_WARPS + (threadIdx.x >> 5);
    if (uli >= P.mb) return;                                  // the whole warp leaves
    const size_t ul = (size_t)uli;
    const int u = P.user0 + uli;
    const int K = P.K, n = P.n;
    const T NaN = P.nan_value;
    const unsigned lanes_le = FULL_WARP >> (31 - lane);

    if (P.topk_items) for (int c = lane; c < K; c += 32) P.topk_items[ul * K + c] = -1;
    if (P.topk_scores) for (int c = lane; c < K; c += 32) P.topk_scores[ul * K + c] = NaN;

    int st = P.ustatus[u];
    if (st != 0) {
        all_nan(P, ul, lane);
        if (P.status_out && lane == 0) P.status_out[uli] = st;
        if (P.list_len && lane == 0) P.list_len[uli] = 0;
        return;
    }
    const int ntrain = P.trp[u + 1] - P.trp[u];
    const int tp0 = P.tep[u];
    const int npos = P.tep[u + 1] - tp0;
    const int cand = n - ntrain;
    const bool only_ndcg = (ntrain + npos) >= n;             // hpp:479-482
    const bool k_leq_n = cand <= K;                          // hpp:483
    const int walk = K < cand ? K : cand;
    const T* cs = P.cand_score + ul * (size_t)P.C;
    const int* ci = P.cand_item + ul * (size_t)P.C;

    // ---- validity of the ranking (hpp:537-563; NaN anywhere => NaN row, hpp:195-197) ----
    {
        bool bad = (P.uflags[u] & 1) != 0 || P.cand_count[uli] < walk;
        if (!bad) {
            const bool partial_path = ((!P.want_roc || only_ndcg) && K < cand);
            const T pred_max = cs[0];
            T pred_min;
            if (partial_path) pred_min = cs[K - 1];
            else if (cand <= K) pred_min = cs[cand - 1];
            else pred_min = NumTraits<T>::from_orderable(P.umin[u]);   // full order: smallest candidate score
            // noise off: the sorted extremes decide (hpp:541-548 / :555-562).  Noise on: the rule is "all candidates equal"
            // (hpp:527), decided before the noise went in: flag 4 from the scoring stage, or -- full order -- the exact extremes
            const bool equal = !P.noise ? (pred_max == pred_min)
                                        : ((P.uflags[u] & 4) != 0 || (!partial_path && cand > K && pred_max == pred_min));
            bad = (pred_max != pred_max) || (pred_min != pred_min) || isinf(pred_max) || isinf(pred_min) || equal;
        }
        if (bad) {
            all_nan(P, ul, lane);
            if (P.status_out && lane == 0) P.status_out[uli] = 3;
            if (P.list_len && lane == 0) P.list_len[uli] = 0;
            return;
        }
    }
    if (P.status_out && lane == 0) P.status_out[uli] = 0;
    if (P.list_len && lane == 0) P.list_len[uli] = walk;
    if (P.topk_items) for (int c = lane; c < walk; c += 32) P.topk_items[ul * K + c] = ci[c];
    if (P.topk_scores) for (int c = lane; c < walk; c += 32) P.topk_scores[ul * K + c] = cs[c];

    const int* ti = P.tei + tp0;
    const T* tv = P.tev ? (P.tev + tp0) : nullptr;
    const size_t rs = P.cumulative ? (size_t)K : 1;          // row stride of the top-K outputs
    T* p_u = P.p ? P.p + ul * rs : nullptr;
    T* tp_u = P.tp ? P.tp + ul * rs : nullptr;
    T* r_u = P.r ? P.r + ul * rs : nullptr;
    T* ap_u = P.ap ? P.ap + ul * rs : nullptr;
    T* tap_u = P.tap ? P.tap + ul * rs : nullptr;
    T* ndcg_u = P.ndcg ? P.ndcg + ul * rs : nullptr;
    T* hit_u = P.hit ? P.hit + ul * rs : nullptr;
    T* rr_u = P.rr ? P.rr + ul * rs : nullptr;

    // ---- top-K walk (hpp:605-708).  Unlike the reference (quirk Q2) Hit@K / RR@K requested on their
    //      own are computed too.  (The early exit of hpp:637-638 can only trigger on the last rank.) ----
    int hits = 0;
    double avg_p = 0, dcg = 0;
    int min_rank = INT_MAX;
    bool did_walk = false;
    const bool calc_top = P.p || P.tp || P.r || P.ap || P.tap || P.ndcg || P.hit || P.rr;
    if (calc_top && (!k_leq_n || P.ap || P.tap || P.rr || P.ndcg)) {
        did_walk = true;
        for (int base = 0; base < walk; base += 32) {
            const int ix = base + lane;
            bool hit = false;
            T val = (T)0;
            if (ix < walk) {
                const int item = ci[ix];
                int lo = 0, hi = npos;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (ti[mid] < item) lo = mid + 1; else hi = mid; }
                if (lo < npos && ti[lo] == item) { hit = true; if (tv) val = tv[lo]; }
            }
            const unsigned mask = __ballot_sync(FULL_WARP, hit);
            const int my_hits = hits + __popc(mask & lanes_le);          // hits up to and including rank ix
            // this rank's terms, computed by its lane ...
            double t_ap = 0., t_dcg = 0.;
            if (hit) {
                t_ap = my_hits / (double)(ix + 1);
                t_dcg = tv ? ((double)val / P.log2tab[ix]) : 0.;
            }
            // ... and added in rank order; a lane keeps the sums as of its own rank
            double my_ap = avg_p, my_dcg = dcg;
            for (unsigned m = mask; m; m &= m - 1) {
                const int b = __ffs(m) - 1;
                avg_p += __shfl_sync(FULL_WARP, t_ap, b);
                dcg += __shfl_sync(FULL_WARP, t_dcg, b);
                if (b <= lane) { my_ap = avg_p; my_dcg = dcg; }
            }
            int my_min_rank = min_rank;
            if (mask) {
                const int first = base + __ffs(mask) - 1;
                if (my_min_rank == INT_MAX && (mask & lanes_le)) my_min_rank = first;
                if (min_rank == INT_MAX) min_rank = first;
            }
            hits += __popc(mask);
            if (P.cumulative && ix < walk) {
                const int tn = (ix + 1) < npos ? (ix + 1) : npos;
                if (p_u) p_u[ix] = (T)(my_hits / (double)(ix + 1));
                if (tp_u) tp_u[ix] = (T)(my_hits / (double)tn);
                if (r_u) r_u[ix] = (T)(my_hits / (double)npos);
                if (ap_u) ap_u[ix] = (T)(my_ap / (double)npos);
                if (tap_u) tap_u[ix] = (T)(my_ap / (double)tn);
                if (ndcg_u) ndcg_u[ix] = (T)my_dcg;
                if (hit_u) hit_u[ix] = (T)(my_hits > 0);
                if (rr_u) rr_u[ix] = (T)(my_hits ? (1. / (double)(my_min_rank + 1)) : 0.);
            }
        }
        if (!P.cumulative && lane == 0) {
            const int tn = K < npos ? K : npos;
            if (p_u) *p_u = (T)((double)hits / (double)K);
            if (tp_u) *tp_u = (T)((double)hits / (double)tn);
            if (r_u) *r_u = (T)((double)hits / (double)npos);
            if (ap_u) *ap_u = (T)(avg_p / (double)npos);
            if (tap_u) *tap_u = (T)(avg_p / (double)tn);
            if (hit_u) *hit_u = (T)(hits > 0);
            if (rr_u) *rr_u = (T)(hits ? (1. / (double)(min_rank + 1)) : 0.);
        }
    }
    __syncwarp();

    // ---- post-hoc NaN rules (hpp:750-788).  Column c of a row is always touched by lane c % 32, scalars by lane 0. ----
    {
        const int cnt = P.cumulative ? K : 1;
        if (k_leq_n) {
            if (!P.cumulative || !did_walk)
                for (int c = lane; c < cnt; c += 32) {
                    if (p_u) p_u[c] = NaN;
                    if (tp_u) tp_u[c] = NaN;
                    if (r_u) r_u[c] = NaN;
                    if (hit_u) hit_u[c] = NaN;
                }
            if (!did_walk)     // outputs the reference leaves untouched here; keep every element defined
                for (int c = lane; c < cnt; c += 32) {
                    if (ap_u) ap_u[c] = NaN;
                    if (tap_u) tap_u[c] = NaN;
                    if (rr_u) rr_u[c] = NaN;
                    if (ndcg_u) ndcg_u[c] = NaN;
                }
        } else if (only_ndcg) {
            for (int c = lane; c < cnt; c += 32) {
                if (p_u) p_u[c] = NaN;
                if (tp_u) tp_u[c] = NaN;
                if (r_u) r_u[c] = NaN;
                if (ap_u) ap_u[c] = NaN;
                if (tap_u) tap_u[c] = NaN;
                if (hit_u) hit_u[c] = NaN;
                if (rr_u) rr_u[c] = NaN;
            }
        }
    }

    // ---- ROC-AUC / PR-AUC (hpp:795-865) from the rank counts ----
    if (P.roc || P.pr || P.pos_rank) {
        if (only_ndcg || !P.count_ranks) {
            if (lane == 0) {
                if (P.roc) P.roc[ul] = NaN;
                if (P.pr) P.pr[ul] = NaN;
            }
        } else {
            // above[j] = number of candidates scoring strictly above the j-th smallest held-out score
            // (counted by score_select_kernel); walk the held-out items from the best down.  Lane l takes the
            // held-out items h = l+1, l+33, ...: the rank a tie chain assigns is a running maximum, the sums follow
            // in order.
            const unsigned int* ab = P.auc_cnt + (size_t)tp0;
            unsigned long long prev_rank = 0, sum_ranks = 0;
            double ap_full = 0;
            for (int hb = 1; hb <= npos; hb += 32) {
                const int h = hb + lane;
                const bool on = h <= npos;
                // rank_h = max(above_h + 1, rank_{h-1} + 1)  <=>  rank_h - h = max over h' <= h of (above_h' + 1 - h')
                long long key = on ? (long long)ab[npos - h] + 1 - (long long)h : LLONG_MIN;
                for (int o = 1; o < 32; o <<= 1) {
                    const long long w = __shfl_up_sync(FULL_WARP, key, o);
                    if (lane >= o && w > key) key = w;
                }
                const long long carry = (long long)prev_rank - (long long)(hb - 1);   // rank_{hb-1} - (hb-1)
                if (hb > 1 && carry > key) key = carry;
                const unsigned long long rank = (unsigned long long)(key + (long long)h);
                const double t_ap = on ? (double)h / (double)rank : 0.;
                if (on && P.pos_rank) P.pos_rank[(size_t)tp0 + P.pos_perm[tp0 + npos - h]] = (long long)rank;
                const int cnt = npos - hb + 1 < 32 ? npos - hb + 1 : 32;
                for (int t = 0; t < cnt; t++) {
                    sum_ranks += __shfl_sync(FULL_WARP, rank, t);
                    ap_full += __shfl_sync(FULL_WARP, t_ap, t);
                }
                prev_rank = __shfl_sync(FULL_WARP, rank, cnt - 1);
            }
            if (lane == 0) {
                const unsigned long long np = (unsigned long long)npos;
                const unsigned long long nneg = (unsigned long long)cand - np;
                if (P.roc)   // hpp:821-822 (long double there; double here, difference < 1e-15)
                    P.roc[ul] = (T)(1. - (double)(sum_ranks - (np * (np + 1)) / 2) / (double)(np * nneg));
                if (P.pr) P.pr[ul] = (T)(ap_full / (double)npos);
            }
        }
    }

    // ---- NDCG normalisation (hpp:868-961) ----
    if (ndcg_u && did_walk) {
        __syncwarp();
        const int L = K < npos ? K : npos;
        // what partial_sort + the vmax/vmin checks (hpp:870-887) decide, from one scan
        bool has_nan = false;
        int n_neg_inf = 0;
        T vmax = -NumTraits<T>::inf();
        for (int j = lane; j < npos; j += 32) {
            const T v = tv[j];
            has_nan |= (v != v);
            n_neg_inf += (v == -NumTraits<T>::inf());
            if (v > vmax) vmax = v;
        }
        has_nan = __any_sync(FULL_WARP, has_nan);
        n_neg_inf = warp_sum(n_neg_inf);
        vmax = warp_max(vmax);
        const bool bad = has_nan || isinf(vmax) || vmax <= 0 || (npos - n_neg_inf) < L;
        if (bad) {
            const int cnt = P.cumulative ? K : 1;
            for (int c = lane; c < cnt; c += 32) ndcg_u[c] = NaN;
            return;
        }
        // ideal DCG: the user's values in descending order.  One round per DISTINCT value: the largest value below
        // the previous round's and how often it occurs (equal values give equal terms, their order is immaterial);
        // its terms val / log2(ix + 2) are computed by the lanes owning those ranks and added in rank order.
        double idcg = 0;
        T prev_v = NumTraits<T>::inf();
        bool first = true, stopped = false;
        int ix = 0;
        while (ix < L) {
            T best = -NumTraits<T>::inf();
            int cnt = 0;
            for (int j = lane; j < npos; j += 32) {
                const T v = tv[j];
                if (first || v < prev_v) {
                    if (v > best) { best = v; cnt = 1; }
                    else if (v == best) cnt++;
                }
            }
            const T wmax = warp_max(best);
            const int total = warp_sum(best == wmax ? cnt : 0);
            if (total <= 0) break;                                           // cannot happen: npos - ix values remain
            const int take = total < L - ix ? total : L - ix;
            const double val = (double)wmax;
            if (!P.cumulative ? (val <= 0) : (val < 0)) { stopped = true; break; }   // hpp:907-910 (== :901-902 when all >= 0), :938
            const int end = ix + take;
            for (int cb = ix & ~31; cb < end; cb += 32) {
                const int r = cb + lane;
                const bool on = r >= ix && r < end;
                const double term = on ? val / P.log2tab[r] : 0.;
                const int t0 = (ix > cb ? ix : cb) - cb, t1 = (end < cb + 32 ? end : cb + 32) - cb;
                double my_idcg = 0.;
                for (int t = t0; t < t1; t++) {
                    idcg += __shfl_sync(FULL_WARP, term, t);
                    if (t == lane) my_idcg = idcg;
                }
                if (P.cumulative && on) ndcg_u[r] = (T)((double)ndcg_u[r] / my_idcg);   // hpp:927, :940
            }
            ix = end;
            prev_v = wmax;
            first = false;
        }
        if (!P.cumulative) {
            if (lane == 0) *ndcg_u = (T)(dcg / idcg);                        // hpp:903, :912
        } else {
            if (stopped) for (int c = ix + lane; c < L; c += 32) ndcg_u[c] = (T)((double)ndcg_u[c] / idcg);   // hpp:946-948
            __syncwarp();
            if (npos < K) {                                                  // hpp:951-956 frozen tail (quirk Q4)
                const int upto = K < cand ? K : cand;
                const T last = ndcg_u[npos - 1];
                __syncwarp();
                for (int c = npos + lane; c < upto; c += 32) ndcg_u[c] = last;
            }
        }
    }
}

// break_ties_with_noise on the FMA path without rank counting: the reference's noise branch turns a user whose candidates
// all score the same into a NaN row (hpp:524-527).  Necessary: the K best (clean) scores are equal -- only for those users
// (rare) one block re-scores every candidate with the tile kernel's fma chain and raises flag 4 when none differs.
template <typename T>
__global__ void all_equal_check_kernel(const T* __restrict__ cand_score, const int* __restrict__ cand_count, const int C,
                                       const int user0, const int K, const int n,
                                       const int* __restrict__ trp, const int* __restrict__ tri, const int* __restrict__ ustatus,
                                       const T* __restrict__ At, const T* __restrict__ Bt, const T* __restrict__ bias, const int p_pad,
                                       int* __restrict__ uflags)
{
    const int ul = blockIdx.x, u = user0 + ul;
    if (ustatus[u] != 0) return;
    const int t0 = trp[u], t1 = trp[u + 1];
    const int cand = n - (t1 - t0), walk = K < cand ? K : cand;
    if (walk <= 0 || cand_count[ul] < walk) return;
    const T ref = cand_score[(size_t)ul * C];
    if (!(ref == cand_score[(size_t)ul * C + walk - 1])) return;
    constexpr int BN = NumTraits<T>::BN;
    const T* a = At + (size_t)(ul / BM) * p_pad * BM + (ul % BM);
    int differs = 0;
    for (int item = threadIdx.x; item < n && !differs; item += blockDim.x) {
        int lo = t0, hi = t1;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (tri[mid] < item) lo = mid + 1; else hi = mid; }
        if (lo < t1 && tri[lo] == item) continue;
        const T* b = Bt + (size_t)(item / BN) * p_pad * BN + (item % BN);
        T acc = (T)0;
        for (int k = 0; k < p_pad; k++) acc = NumTraits<T>::fma(a[(size_t)k * BM], b[(size_t)k * BN], acc);
        if (bias != nullptr) acc += bias[item];
        if (!(acc == ref)) differs = 1;
    }
    if (!__syncthreads_or(differs) && threadIdx.x == 0) atomicOr(&uflags[u], 4);
}

// ---------------------------------------------------------------- per-metric means over users (extension)
// numpy.nanmean of the per-user rows, on the device and in a fixed summation order:
//   metric_partial_kernel  one block per 256 users of a batch and metric (blockIdx.y): sum and count of the non-NaN
//                          entries of every column (W = K if cumulative else 1), users in ascending order
//   metric_final_kernel    one thread per (metric, column): adds the blocks' partials in ascending order, divides
// A table has `slots` metrics: the ten accuracy metrics (the first eight have W columns, ROC/PR-AUC one), or the three of
// beyond.cuh (all W columns), each with partial buffers of its own.
constexpr int MEAN_CHUNK = 256;

template <typename T>
struct MeanParams {
    const T* out[10];        // metric rows of the batch (nullptr: not requested), row stride W (slots >= wide: 1)
    int nb, W;
    int slots, wide;         // metrics in the table; the first `wide` have W columns
    double* part_sum;        // [blocks_total][slots][W]
    int* part_cnt;
    int block0;              // first partial block of this batch
};

template <typename T>
__global__ void metric_partial_kernel(const __grid_constant__ MeanParams<T> P)
{
    const int q = blockIdx.y;
    const T* src = P.out[q];
    const int W = P.W, Wq = q < P.wide ? W : 1;
    const int u0 = blockIdx.x * MEAN_CHUNK;
    const int u1 = min(u0 + MEAN_CHUNK, P.nb);
    double* ps = P.part_sum + ((size_t)(P.block0 + blockIdx.x) * P.slots + q) * W;
    int* pc = P.part_cnt + ((size_t)(P.block0 + blockIdx.x) * P.slots + q) * W;
    if (Wq > 1) {
        // a thread per column walks the chunk's users in order (consecutive threads read consecutive columns)
        for (int c = threadIdx.x; c < W; c += blockDim.x) {
            double s = 0.;
            int cnt = 0;
            if (src)
                for (int u = u0; u < u1; u++) {
                    const double v = (double)src[(size_t)u * Wq + c];
                    if (v == v) { s += v; cnt++; }
                }
            ps[c] = s;
            pc[c] = cnt;
        }
    } else {
        // one value per user: fixed-shape tree over the chunk
        __shared__ double sh_s[MEAN_CHUNK];
        __shared__ int sh_c[MEAN_CHUNK];
        const int u = u0 + threadIdx.x;
        double v = (src && u < u1) ? (double)src[u] : CUDART_NAN;
        sh_s[threadIdx.x] = (v == v) ? v : 0.;
        sh_c[threadIdx.x] = (v == v) ? 1 : 0;
        __syncthreads();
        for (int o = MEAN_CHUNK / 2; o > 0; o >>= 1) {
            if (threadIdx.x < o) { sh_s[threadIdx.x] += sh_s[threadIdx.x + o]; sh_c[threadIdx.x] += sh_c[threadIdx.x + o]; }
            __syncthreads();
        }
        if (threadIdx.x == 0) { ps[0] = sh_s[0]; pc[0] = sh_c[0]; }
        for (int c = 1 + threadIdx.x; c < W; c += blockDim.x) { ps[c] = 0.; pc[c] = 0; }
    }
}

__global__ void metric_final_kernel(const double* __restrict__ part_sum, const int* __restrict__ part_cnt, const int blocks,
                                    const int slots, const int W, double* __restrict__ means, long long* __restrict__ counts)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;     // (metric, column)
    const int cells = slots * W;
    if (i >= cells) return;
    double s = 0.;
    long long c = 0;
    const double* ps = part_sum + i;
    const int* pc = part_cnt + i;
    for (int b = 0; b < blocks; b++, ps += cells, pc += cells) { s += *ps; c += *pc; }
    if (means) means[i] = c > 0 ? s / (double)c : CUDART_NAN;
    if (counts) counts[i] = c;
}

}  // namespace rmb
