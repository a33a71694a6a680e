/* TEST INFRASTRUCTURE -- not part of the product; see recometrics_oracle.c.
 *
 * Type-generic body, included twice (REAL = float, REAL = double).
 * Every block cites the reference lines it restates (paths under /root/reference).
 */

/* src/recometrics.hpp:84-112  dot1(): fused-multiply-add reduction that the
 * compiler vectorises through "omp simd reduction".  Compiled with the same
 * flags as oracle/_ref (Makefile) so the lane split and rounding are the same. */
static inline REAL FN(dot1)(const REAL *restrict x, const REAL *restrict y, const int n)
{
    REAL res = 0;
    #pragma omp simd reduction(+:res)
    for (int32_t ix = 0; ix < n; ix++) res = FMA(x[ix], y[ix], res);
    return res;
}

/* order used for ranking: score descending (src/recometrics.hpp:538-540, :552-554 use a
 * strict '>' comparator, leaving ties to libstdc++); the oracle pins ties by ascending
 * item id so that its output is a deterministic function of the scores. */
static inline int FN(goes_before)(const REAL *pred, int32_t i, int32_t j)
{
    if (pred[i] > pred[j]) return 1;
    if (pred[i] < pred[j]) return 0;
    return i < j;
}

static void FN(merge_sort)(int32_t *ind, int32_t *tmp, int32_t len, const REAL *pred)
{
    if (len < 2) return;
    if (len <= 8) { /* insertion sort */
        for (int32_t a = 1; a < len; a++) {
            int32_t v = ind[a], b = a;
            while (b > 0 && FN(goes_before)(pred, v, ind[b-1])) { ind[b] = ind[b-1]; b--; }
            ind[b] = v;
        }
        return;
    }
    int32_t half = len / 2;
    FN(merge_sort)(ind, tmp, half, pred);
    FN(merge_sort)(ind + half, tmp, len - half, pred);
    int32_t a = 0, b = half, o = 0;
    while (a < half && b < len)
        tmp[o++] = FN(goes_before)(pred, ind[b], ind[a]) ? ind[b++] : ind[a++];
    while (a < half) tmp[o++] = ind[a++];
    while (b < len) tmp[o++] = ind[b++];
    memcpy(ind, tmp, (size_t)len * sizeof(int32_t));
}

typedef struct {
    REAL *p, *tp, *r, *ap, *tap, *ndcg, *hit, *rr, *roc, *pr;
} FN(outs_t);

/* src/recometrics.hpp:450-476  "set_as_NAN" block */
static void FN(fill_nan)(const FN(outs_t) *o, int32_t user, int32_t K, int cumulative)
{
    REAL *top[8] = {o->p, o->tp, o->r, o->ap, o->tap, o->ndcg, o->hit, o->rr};
    for (int q = 0; q < 8; q++) {
        if (!top[q]) continue;
        if (!cumulative) top[q][user] = (REAL)NAN;
        else for (int32_t c = 0; c < K; c++) top[q][(size_t)user*(size_t)K + c] = (REAL)NAN;
    }
    if (o->roc) o->roc[user] = (REAL)NAN;
    if (o->pr) o->pr[user] = (REAL)NAN;
}

/* src/recometrics.hpp:531-534  per-user tie-breaking noise:
 *     std::mt19937 rng_user(seed + (uint64_t)user);
 *     std::uniform_real_distribution<real_t> runif((real_t)(-1e-12), (real_t)1e-12);
 *     for (ix < move_to) pred[ind[ix]] += runif(rng_user);
 * restated from the published algorithms: MT19937 (Matsumoto & Nishimura 1998; the parameters of
 * std::mt19937, seeded with value mod 2^32) and libstdc++ 13's uniform_real_distribution =
 * generate_canonical<real_t, digits>(rng) * (b - a) + a, where generate_canonical draws
 * ceil(digits / 32) words (1 for float, 2 for double), sums them as real_t(word) * 2^(32 i), divides by
 * 2^(32 m) and replaces a result >= 1 by nextafter(1, 0).  Pinned against the compiled reference by the
 * noise cases of tests/golden (tie-heavy inputs whose ranking is decided by the noise alone). */
#ifndef RMO_MT_DEFINED
#define RMO_MT_DEFINED
typedef struct { uint32_t x[624]; int pos; } rmo_mt_t;
static void rmo_mt_seed(rmo_mt_t *g, uint64_t value)
{
    g->x[0] = (uint32_t)(value & 0xffffffffu);
    for (int i = 1; i < 624; i++) g->x[i] = 1812433253u * (g->x[i-1] ^ (g->x[i-1] >> 30)) + (uint32_t)i;
    g->pos = 624;
}
static uint32_t rmo_mt_next(rmo_mt_t *g)
{
    if (g->pos >= 624) {
        for (int k = 0; k < 624; k++) {
            const uint32_t y = (g->x[k] & 0x80000000u) | (g->x[(k + 1) % 624] & 0x7fffffffu);
            g->x[k] = g->x[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        g->pos = 0;
    }
    uint32_t z = g->x[g->pos++];
    z ^= (z >> 11);
    z ^= (z << 7) & 0x9d2c5680u;
    z ^= (z << 15) & 0xefc60000u;
    z ^= (z >> 18);
    return z;
}
#endif

static inline REAL FN(runif)(rmo_mt_t *g)
{
    REAL sum, tmp;
    if (sizeof(REAL) == 4) {
        sum = (REAL)rmo_mt_next(g);
        tmp = (REAL)4294967296.0;
    } else {
        sum = (REAL)rmo_mt_next(g);
        sum += (REAL)rmo_mt_next(g) * (REAL)4294967296.0;
        tmp = (REAL)4294967296.0 * (REAL)4294967296.0;
    }
    REAL ret = sum / tmp;
    if (ret >= (REAL)1) ret = (sizeof(REAL) == 4) ? (REAL)nextafterf(1.0f, 0.0f) : (REAL)nextafter(1.0, 0.0);
    const REAL a = (REAL)(-1e-12), b = (REAL)1e-12;
    return FMA(ret, b - a, a);      /* the reference's C++ build contracts (u * (b - a)) + a into one fma */
}

/* One user of the loop at src/recometrics.hpp:437-962.
 * scratch: pred[n], ind[n], tmp[n], isnew mask[n] */
static int32_t FN(one_user)(
    int32_t user,
    const REAL *restrict A, size_t lda, const REAL *restrict B, size_t ldb,
    int32_t n, int32_t k,
    const int32_t *restrict trp, const int32_t *restrict tri,
    const int32_t *restrict tep, const int32_t *restrict tei, const REAL *restrict tev,
    int32_t K, int cumulative, const FN(outs_t) *o,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int fix_quirks, int noise, uint64_t seed,
    REAL *pred, int32_t *ind, int32_t *tmp, unsigned char *mask,
    int32_t *topk_items, REAL *topk_scores, int64_t *pos_rank, int32_t *tie_flag)
{
    const int32_t ntrain = trp[user+1] - trp[user];
    const int32_t npos_i = tep[user+1] - tep[user];
    const int want_auc = (o->roc || o->pr);

    /* :439-448 eligibility */
    if (npos_i <= 0 ||
        ((ntrain + npos_i) >= n && !o->ndcg) ||
        (n - ntrain) < min_items_pool ||
        (!consider_cold_start && ntrain == 0) ||
        npos_i < min_pos_test)
    {
        FN(fill_nan)(o, user, K, cumulative);
        return 1;
    }

    /* :479-486 */
    const int only_ndcg = (ntrain + npos_i) >= n;
    const int k_leq_n = (n - ntrain) <= K;
    if (k_leq_n && !o->roc && !o->pr && !o->ap && !o->tap && !o->rr) {
        FN(fill_nan)(o, user, K, cumulative);
        return 2;
    }

    /* :491-497 candidate ids = every item outside the (sorted, duplicate-free) train row, ascending */
    memset(mask, 0, (size_t)n);
    for (int32_t ix = trp[user]; ix < trp[user+1]; ix++) mask[tri[ix]] = 1;
    int32_t cand = 0;
    for (int32_t j = 0; j < n; j++) if (!mask[j]) ind[cand++] = j;
    /* with duplicate-free rows cand == n - ntrain == move_to (:493-495) */

    /* :499-512 scoring */
    const REAL *Au = A + (size_t)user * lda;
    int has_nan = 0;
    for (int32_t ix = 0; ix < cand; ix++) {
        REAL s = FN(dot1)(Au, B + (size_t)ind[ix] * ldb, k);
        pred[ind[ix]] = s;
        has_nan |= isnan(s);
    }
    /* Documented rule (:195-197): "one or more of the predicted scores evaluates to NAN" => NaN row.
     * The reference only enforces it when break_ties_with_noise (:517-518); with noise off a NaN
     * inside the comparator is unspecified behaviour, so the oracle (and the product) pin it to
     * the documented rule. */
    if (has_nan) { FN(fill_nan)(o, user, K, cumulative); return 3; }

    if (noise) {
        /* :516-534 validity of the noise branch (every candidate: NaN above, all equal, infinite extremes), then the noise */
        REAL pred_max = pred[ind[0]], pred_min = pred[ind[0]];
        for (int32_t ix = 1; ix < cand; ix++) {
            if (pred_max < pred[ind[ix]]) pred_max = pred[ind[ix]];
            if (pred_min > pred[ind[ix]]) pred_min = pred[ind[ix]];
        }
        if (pred_max == pred_min || isinf(pred_max) || isinf(pred_min)) { FN(fill_nan)(o, user, K, cumulative); return 3; }
        rmo_mt_t g;
        rmo_mt_seed(&g, seed + (uint64_t)user);
        for (int32_t ix = 0; ix < cand; ix++) pred[ind[ix]] += FN(runif)(&g);
    }

    /* :537-563 ranking + validity.  The oracle always produces the full order; which pair of
     * scores is checked depends on the branch the reference takes. */
    FN(merge_sort)(ind, tmp, cand, pred);
    const int partial_path = ((!o->roc || only_ndcg) && K < cand);
    if (!noise) {          /* :541-548, :555-562: only the noise-off branch looks at the sorted extremes */
        REAL pred_max = pred[ind[0]];
        REAL pred_min = partial_path ? pred[ind[K-1]] : pred[ind[cand-1]];
        if (isnan(pred_max) || isnan(pred_min) || isinf(pred_max) || isinf(pred_min) ||
            pred_max == pred_min)
        {
            FN(fill_nan)(o, user, K, cumulative);
            return 3;
        }
    }

    /* extras the reference API never returns (SURVEY 8(c)) */
    const int32_t walk = K < cand ? K : cand;
    if (topk_items)  for (int32_t ix = 0; ix < walk; ix++) topk_items[(size_t)user*K + ix] = ind[ix];
    if (topk_scores) for (int32_t ix = 0; ix < walk; ix++) topk_scores[(size_t)user*K + ix] = pred[ind[ix]];

    /* :565-573 test mask (the oracle uses it for every membership test) */
    memset(mask, 0, (size_t)n);
    for (int32_t ix = tep[user]; ix < tep[user+1]; ix++) mask[tei[ix]] = 1;

    /* Exact score ties whose order the reference leaves to libstdc++ (quirk Q8): flag the users for
     * which the tie order can change an output, so that comparisons against the reference can
     * set them aside.  bit0: tie between neighbours inside ranks [1, K+1] where one is a held-out
     * item and the other is not (or any tie across the K/K+1 boundary);
     * bit1: same, anywhere in the full order (matters for ROC/PR-AUC only). */
    if (tie_flag) {
        int32_t f = 0;
        for (int32_t ix = 0; ix + 1 < cand; ix++) {
            if (pred[ind[ix]] == pred[ind[ix+1]]) {
                const int differ = mask[ind[ix]] != mask[ind[ix+1]];
                if (ix < walk && (differ || ix == walk - 1)) f |= 1;
                if (differ) f |= 2;
            }
        }
        *tie_flag = f;
    }

    const int32_t *user_istart = tei + tep[user];
    const int32_t *user_iend = tei + tep[user+1];
    const REAL *user_v = tev ? (tev + tep[user]) : NULL;
    const uint64_t npos = (uint64_t)npos_i;
    const uint64_t nneg = (uint64_t)cand - npos;               /* :594-595 */
    const size_t st = (size_t)user * (size_t)K;

    REAL *p_u = o->p, *tp_u = o->tp, *r_u = o->r, *ap_u = o->ap, *tap_u = o->tap,
         *ndcg_u = o->ndcg, *hit_u = o->hit, *rr_u = o->rr;
    if (cumulative) {                                          /* :575-586 */
        if (p_u) p_u += st;  if (tp_u) tp_u += st;  if (r_u) r_u += st;  if (ap_u) ap_u += st;
        if (tap_u) tap_u += st;  if (ndcg_u) ndcg_u += st;  if (hit_u) hit_u += st;  if (rr_u) rr_u += st;
    }

    int did_short_loop = 0;
    int32_t hits = 0;
    double avg_p = 0, dcg = 0;
    int32_t min_rank = INT32_MAX;

    /* :420 calc_top_metrics leaves hit/rr out, so a hit/rr-only request never runs the walk
     * and the reference returns uninitialised memory (SURVEY quirk Q2).  fix_quirks computes them. */
    int calc_top = (o->p || o->tp || o->r || o->ap || o->tap || o->ndcg);
    if (fix_quirks) calc_top = calc_top || o->hit || o->rr;

    /* :605-748 top-K walk */
    if (calc_top && (!k_leq_n || o->ap || o->tap || o->rr || o->ndcg))
    {
        did_short_loop = 1;
        for (int32_t ix = 0; ix < walk; ix++)
        {
            const int32_t item = ind[ix];
            if (mask[item]) {
                /* :615-621 position inside the (sorted) test row gives the value */
                const int32_t *res = user_istart;
                { int32_t lo = 0, hi = (int32_t)(user_iend - user_istart);
                  while (lo < hi) { int32_t mid = lo + (hi - lo)/2; if (user_istart[mid] < item) lo = mid+1; else hi = mid; }
                  res = user_istart + lo; }
                hits++;
                avg_p += hits / (double)(ix+1);
                dcg += user_v ? ((double)user_v[res - user_istart] / log2((double)(ix+2))) : 0.;   /* :620 */
                if (ix < min_rank) min_rank = ix;
            }
            if (cumulative) {                                   /* :625-635 */
                const int32_t tn = (ix+1) < (int32_t)npos ? (ix+1) : (int32_t)npos;
                if (p_u) p_u[ix] = (REAL)(hits / (double)(ix+1));
                if (tp_u) tp_u[ix] = (REAL)(hits / (double)tn);
                if (r_u) r_u[ix] = (REAL)(hits / (double)npos);
                if (ap_u) ap_u[ix] = (REAL)(avg_p / (double)npos);
                if (tap_u) tap_u[ix] = (REAL)(avg_p / (double)tn);
                if (ndcg_u) ndcg_u[ix] = (REAL)dcg;
                if (hit_u) hit_u[ix] = (REAL)(hits > 0);
                if (rr_u) rr_u[ix] = (REAL)(hits ? (1. / (double)(min_rank+1)) : 0.);
            }
            if (!cumulative && hits >= cand) break;            /* :637-638 */
        }
        if (!cumulative) {                                      /* :699-708 */
            const int32_t tn = K < (int32_t)npos ? K : (int32_t)npos;
            if (o->p) o->p[user] = (REAL)((double)hits / (double)K);
            if (o->tp) o->tp[user] = (REAL)((double)hits / (double)tn);
            if (o->r) o->r[user] = (REAL)((double)hits / (double)npos);
            if (o->ap) o->ap[user] = (REAL)(avg_p / (double)npos);
            if (o->tap) o->tap[user] = (REAL)(avg_p / (double)tn);
            if (o->hit) o->hit[user] = (REAL)(hits > 0);
            if (o->rr) o->rr[user] = (REAL)(hits ? (1. / (double)(min_rank+1)) : 0.);
        }
        /* :710-747 (K > move_to) cannot happen: eligibility forces cand >= max(min_items_pool,K,2) */
    }

    /* :750-788 post-hoc NaN rules */
    if (k_leq_n) {
        if (!cumulative) {
            if (o->p) o->p[user] = (REAL)NAN;
            if (o->tp) o->tp[user] = (REAL)NAN;
            if (o->r) o->r[user] = (REAL)NAN;
            if (o->hit) o->hit[user] = (REAL)NAN;
        } else if (!did_short_loop) {
            for (int32_t c = 0; c < K; c++) {
                if (p_u) p_u[c] = (REAL)NAN;
                if (tp_u) tp_u[c] = (REAL)NAN;
                if (r_u) r_u[c] = (REAL)NAN;
                if (hit_u) hit_u[c] = (REAL)NAN;
            }
        }
    } else if (only_ndcg) {
        if (!cumulative) {
            if (o->p) o->p[user] = (REAL)NAN;   if (o->tp) o->tp[user] = (REAL)NAN;
            if (o->r) o->r[user] = (REAL)NAN;   if (o->ap) o->ap[user] = (REAL)NAN;
            if (o->tap) o->tap[user] = (REAL)NAN; if (o->hit) o->hit[user] = (REAL)NAN;
            if (o->rr) o->rr[user] = (REAL)NAN;
        } else {
            for (int32_t c = 0; c < K; c++) {
                if (p_u) p_u[c] = (REAL)NAN;   if (tp_u) tp_u[c] = (REAL)NAN;
                if (r_u) r_u[c] = (REAL)NAN;   if (ap_u) ap_u[c] = (REAL)NAN;
                if (tap_u) tap_u[c] = (REAL)NAN; if (hit_u) hit_u[c] = (REAL)NAN;
                if (rr_u) rr_u[c] = (REAL)NAN;
            }
        }
    }

    /* :795-865 AUC walks.  The reference walks the FULL order when roc_auc is requested; with
     * pr_auc alone it walks a partially sorted list (SURVEY quirk Q3) -- not restatable, the oracle
     * always walks the full order (== the reference whenever roc_auc is also requested). */
    if (want_auc || pos_rank) {
        if (only_ndcg) {
            if (o->roc) o->roc[user] = (REAL)NAN;
            if (o->pr) o->pr[user] = (REAL)NAN;
        } else {
            uint64_t sum_ranks_pos = 0;
            int32_t h = 0;
            double ap_full = 0;
            for (int32_t ix = 0; ix < cand; ix++) {
                if (mask[ind[ix]]) {
                    sum_ranks_pos += (uint64_t)(ix+1);
                    h++;
                    ap_full += (double)h / (double)(ix+1);
                    if (pos_rank) {
                        int32_t lo = 0, hi = (int32_t)npos;
                        while (lo < hi) { int32_t mid = lo + (hi - lo)/2; if (user_istart[mid] < ind[ix]) lo = mid+1; else hi = mid; }
                        pos_rank[tep[user] + lo] = (int64_t)(ix+1);
                    }
                    if (h == (int32_t)npos) break;
                }
            }
            if (o->roc)                                         /* :821-822 */
                o->roc[user] = (REAL)(1. - (long double)(sum_ranks_pos - (npos * (npos + 1)) / 2)
                                            / (long double)(npos * nneg));
            if (o->pr) o->pr[user] = (REAL)(ap_full / (double)npos);   /* :823 */
        }
    }

    /* :868-961 NDCG normalisation */
    if (o->ndcg)
    {
        const int32_t L = K < (int32_t)npos ? K : (int32_t)npos;
        /* order of the user's test values, descending (:870-873); ties by position */
        for (int32_t ix = 0; ix < (int32_t)npos; ix++) ind[ix] = ix;
        FN(merge_sort)(ind, tmp, (int32_t)npos, user_v);

        const REAL vmax = user_v[ind[0]];
        const REAL vmin = user_v[ind[L-1]];
        /* A NaN gain makes NDCG NaN wherever it sits (quirk Q9): the reference checks only the two values partial_sort
         * leaves at ranks 0 and L-1, and where a NaN lands under its '>' comparator is unspecified. */
        int nan_gain = 0;
        for (int32_t ix = 0; ix < (int32_t)npos; ix++) nan_gain |= isnan(user_v[ix]);
        if (nan_gain || isnan(vmax) || isinf(vmax) || isnan(vmin) || isinf(vmin) || vmax <= 0) {   /* :875-887 */
            if (!cumulative) o->ndcg[user] = (REAL)NAN;
            else for (int32_t c = 0; c < K; c++) ndcg_u[c] = (REAL)NAN;
            return 0;
        }
        double idcg = 0, val = 0;
        const REAL last_val = vmin;
        if (!cumulative) {
            if (last_val >= 0) {                                /* :900-904 */
                for (int32_t ix = 0; ix < L; ix++) idcg += (double)user_v[ind[ix]] / log2((double)(ix+2));
            } else {                                            /* :906-913 */
                for (int32_t ix = 0; ix < L; ix++) {
                    val = user_v[ind[ix]];
                    if (val <= 0) break;
                    idcg += val / log2((double)(ix+2));
                }
            }
            o->ndcg[user] = (REAL)(dcg / idcg);
        } else {
            if (last_val >= 0) {                                /* :922-929 */
                for (int32_t ix = 0; ix < L; ix++) {
                    idcg += (double)user_v[ind[ix]] / log2((double)(ix+2));
                    ndcg_u[ix] = (REAL)((double)ndcg_u[ix] / idcg);
                }
            } else {                                            /* :931-949 (vmin is finite here) */
                int32_t ix;
                for (ix = 0; ix < L; ix++) {
                    val = user_v[ind[ix]];
                    if (val < 0) break;
                    idcg += val / log2((double)(ix+2));
                    ndcg_u[ix] = (REAL)((double)ndcg_u[ix] / idcg);
                }
                for (; ix < L; ix++) ndcg_u[ix] = (REAL)((double)ndcg_u[ix] / idcg);
            }
            if (npos < (uint64_t)K) {                           /* :951-956 frozen tail (quirk Q4) */
                const int32_t upto = K < cand ? K : cand;
                for (int32_t c = (int32_t)npos; c < upto; c++) ndcg_u[c] = ndcg_u[npos-1];
            }
        }
    }
    return 0;
}

/* Whole call: src/recometrics.hpp:359-965 (OpenMP over users :428-437). */
int FN(rmo_calc_metrics)(
    const REAL *A, size_t lda, const REAL *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_p, const int32_t *Xtrain_i,
    const int32_t *Xtest_p, const int32_t *Xtest_i, const REAL *Xtest_v,
    int32_t k_metrics, int cumulative,
    REAL *p_at_k, REAL *tp_at_k, REAL *r_at_k, REAL *ap_at_k, REAL *tap_at_k,
    REAL *ndcg_at_k, REAL *hit_at_k, REAL *rr_at_k, REAL *roc_auc, REAL *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, int fix_quirks, int break_ties_with_noise, uint64_t seed,
    int32_t *status, int32_t *topk_items, REAL *topk_scores, int64_t *pos_rank, int32_t *tie_flags)
{
    if (nthreads < 1) nthreads = 1;
#ifndef _OPENMP
    nthreads = 1;
#endif
    /* :391-393 (note std::min on min_pos_test: quirk Q1) */
    if (min_items_pool < k_metrics) min_items_pool = k_metrics;
    if (min_items_pool < 2) min_items_pool = 2;
    if (min_pos_test > 1) min_pos_test = 1;

    FN(outs_t) o = {p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k, ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc};
    const size_t nn = (size_t)n;
    REAL *pred = (REAL*)malloc(nn * (size_t)nthreads * sizeof(REAL));
    int32_t *ind = (int32_t*)malloc(nn * (size_t)nthreads * sizeof(int32_t));
    int32_t *tmp = (int32_t*)malloc(nn * (size_t)nthreads * sizeof(int32_t));
    unsigned char *mask = (unsigned char*)malloc(nn * (size_t)nthreads);
    if (!pred || !ind || !tmp || !mask) { free(pred); free(ind); free(tmp); free(mask); return 1; }

    if (topk_items) for (size_t q = 0; q < (size_t)m * (size_t)k_metrics; q++) topk_items[q] = -1;
    if (topk_scores) for (size_t q = 0; q < (size_t)m * (size_t)k_metrics; q++) topk_scores[q] = (REAL)NAN;
    if (pos_rank) for (int32_t q = 0; q < Xtest_p[m]; q++) pos_rank[q] = 0;
    if (tie_flags) for (int32_t q = 0; q < m; q++) tie_flags[q] = 0;

    #pragma omp parallel for schedule(dynamic) num_threads(nthreads)
    for (int32_t user = 0; user < m; user++)
    {
#ifdef _OPENMP
        const size_t t = (size_t)omp_get_thread_num();
#else
        const size_t t = 0;
#endif
        int32_t s = FN(one_user)(user, A, lda, B, ldb, n, k, Xtrain_p, Xtrain_i, Xtest_p, Xtest_i, Xtest_v,
                                 k_metrics, cumulative, &o, consider_cold_start, min_items_pool, min_pos_test,
                                 fix_quirks, break_ties_with_noise, seed,
                                 pred + t*nn, ind + t*nn, tmp + t*nn, mask + t*nn,
                                 topk_items, topk_scores, pos_rank, tie_flags ? tie_flags + user : NULL);
        if (status) status[user] = s;
    }
    free(pred); free(ind); free(tmp); free(mask);
    return 0;
}
