/* recometrics_b200.h -- C-ABI of librecometrics_b200.so
 *
 * B200-native (sm_100a) implementation of the per-user evaluation path of david-cortes/recometrics.
 * The entry points below are what the reference's own bindings bind for that path:
 *
 *   reference interface (replaced)                                         this library
 *   ---------------------------------------------------------------------  ---------------------------
 *   calc_metrics_float   src/recometrics_signatures.hpp:73-98              rmb200_calc_metrics_f32
 *     (defined src/recometrics_instantiated.cpp:94-143,
 *      called from recometrics/wrapper.pyx:381-403)
 *   calc_metrics_double  src/recometrics_signatures.hpp:48-72              rmb200_calc_metrics_f64
 *     (defined src/recometrics_instantiated.cpp:43-92,
 *      called from recometrics/wrapper.pyx:282-304)
 *   calc_metrics<real_t> src/recometrics.hpp:359-385                       both of the above
 *     (called directly from src/Rwrapper.cpp:250-274)                      (via include/recometrics_b200_shim.hpp)
 *   get_has_openmp       src/recometrics_signatures.hpp:46                 rmb200_device_count() > 0
 *   std::runtime_error on SIGINT, src/recometrics.hpp:167-173, :964        RMB200_ERR_INTERRUPTED
 *
 * Parameter order, types and meaning of the first 30 arguments are those of the reference
 * (bool -> int so that the boundary is plain C).  All pointers are HOST pointers owned by the
 * caller unless rmb200_extra_t::inputs_on_device says otherwise; outputs may be uninitialised on
 * entry and EVERY element of every non-NULL output is written (NaN rows included), as the
 * reference does (np.empty outputs, recometrics/wrapper.pyx:270-280).  A NULL output pointer means
 * "metric not requested" (wrapper.pyx:208-224).  Data problems of single users never raise:
 * they give NaN rows (src/recometrics.hpp:193-209).
 *
 * There is no CPU fallback: without a CUDA device every compute entry returns RMB200_ERR_NO_DEVICE.
 */
#ifndef RECOMETRICS_B200_H
#define RECOMETRICS_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__) || defined(__clang__)
#   define RMB200_API __attribute__((visibility("default")))
#else
#   define RMB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define RMB200_VERSION 100 /* 0.1.0 */

enum rmb200_status {
    RMB200_OK = 0,
    RMB200_ERR_BAD_ARG = 1,      /* inconsistent sizes / NULL where data is required          */
    RMB200_ERR_NO_DEVICE = 2,    /* no usable CUDA device (no CPU fallback exists)            */
    RMB200_ERR_CUDA = 3,         /* a CUDA call failed; see rmb200_last_error()               */
    RMB200_ERR_OOM = 4,          /* device or host allocation failed (reference: bad_alloc)   */
    RMB200_ERR_INTERRUPTED = 5,  /* SIGINT arrived during the call (reference: runtime_error) */
    RMB200_ERR_UNSUPPORTED = 6,  /* valid request outside what this build implements          */
    RMB200_ERR_RUNTIME = 7       /* the input is one the reference answers with std::runtime_error (splitters);   */
                                 /* rmb200_last_error() holds the reference's message                              */
};

/* Largest k_metrics the fused top-K selection kernels handle.  Larger values (the reference's only bound is k_metrics <= n,
 * src/recometrics.hpp:391) are computed as well, on the full-order path: every candidate scored and sorted in HBM. */
#define RMB200_MAX_K 384

/* Per-call timing breakdown (milliseconds, CUDA events on the call's stream). */
typedef struct rmb200_timing {
    double total_ms;        /* whole call, host clock                                           */
    double h2d_ms;          /* host->device staging (0 when inputs_on_device)                   */
    double prep_ms;         /* layout kernels: factor transposes, held-out item scores, sorting  */
    double score_select_ms; /* the fused score + exclude + top-K (+rank counting) kernel        */
    double metrics_ms;      /* per-user metrics kernel                                          */
    double d2h_ms;          /* device->host result copies                                       */
    int64_t kernel_launches;/* kernels of this library launched by the call                     */
    int64_t h2d_bytes, d2h_bytes;
    int64_t scoring_path;   /* which scoring kernel ran: 1 = FMA tiles, 2 = tensor-core filter + exact re-score, 3 = full order */
    int64_t filter_fallback_batches; /* user batches the tensor-core filter handed back to the FMA path         */
    double dominant_kernel_ms; /* the scoring kernel alone (filter_select_kernel / score_select_kernel), all batches */
    int64_t filter_retry_rows; /* users whose sampled threshold guess failed its check (their CTA walked the catalogue twice) */
    int64_t filter_fallback_users;   /* users the tensor-core filter handed back to the FMA path (only they are re-run)          */
    double filter_err_ratio_max;     /* extra.filter_stats: largest |approximate - exact| / error bound over all re-scored       */
                                     /* candidates of the call (the bound holds iff this is <= 1)                                 */
    int64_t noise_handback_users;    /* break_ties_with_noise with ROC/PR-AUC: users for whom the noise decides a rank (another candidate  */
                                     /* within its reach of a held-out item) -- re-ranked on the full-order path with their noise          */
    int64_t devices_used;            /* GPUs the call ran on (1 unless rmb200_extra_t::devices / RMB200_DEVICES spread it); on a  */
                                     /* multi-GPU call the *_ms fields are the maximum over the devices, counters are sums        */
} rmb200_timing_t;

/* Optional extension block (pass NULL for reference behaviour).  Zero-initialise, then set
 * struct_size = sizeof(rmb200_extra_t). */
typedef struct rmb200_extra {
    int32_t struct_size;
    int32_t device;             /* CUDA device ordinal; -1 = env RMB200_DEVICE or 0                    */
    int32_t user_begin;         /* evaluate only users [user_begin, user_end) -- the unit by which a   */
    int32_t user_end;           /* job is sharded over GPUs/processes; 0,0 = all m users; user_end < 0  */
                                /* = an empty block (nothing is evaluated or written).  Arrays keep     */
                                /* their full-size indexing: row u of every output is written at u.    */
    int32_t inputs_on_device;   /* 1: A, B, item_biases, the CSR arrays AND all outputs are device     */
                                /* pointers on `device` (HBM-resident call, no host copies)            */
    int32_t strict_min_pos_test;/* 1: honour min_pos_test as documented; 0 (default): reproduce the    */
                                /* reference, which clamps it to <= 1 (src/recometrics.hpp:393)        */
    int32_t *topk_items;        /* optional out [m * k_metrics]: ranked item ids, -1 where undefined   */
    void    *topk_scores;       /* optional out [m * k_metrics] (float or double): their scores        */
    int64_t *pos_rank;          /* optional out [nnz_test]: 1-based rank of every held-out item among  */
                                /* the user's candidates (0 where not computed); forces rank counting  */
    int32_t *status;            /* optional out [m]: 0 computed, 1 not eligible (hpp:439-448),         */
                                /* 2 NaN by the cand<=K rule (hpp:485-486), 3 NaN by score validity     */
    rmb200_timing_t *timing;    /* optional out                                                        */
    int32_t scoring_path;       /* 0 = automatic; 1 = FP32/FP64 FMA tiles for every score; 2 = tensor-core     */
                                /* (fp16 tcgen05) candidate filter + exact FMA re-scoring of the survivors:    */
                                /* same top-K, same scores; not available with ROC/PR-AUC (rank counting);     */
                                /* 3 = full order: every candidate scored, given its tie-breaking noise and    */
                                /* sorted in HBM (what the reference does literally; any k_metrics <= n; slow). */
                                /* Env RMB200_PATH=fma|tensor|full overrides 0.                                */
    int32_t skip_row_copy;      /* 1 (host-pointer calls): the per-user rows of every requested metric are computed  */
                                /* in device memory but NOT copied back -- the non-NULL output pointers only say    */
                                /* which metrics are wanted and are left untouched; use with metric_means           */
    double  *metric_means;      /* optional out [10 * W], W = cumulative ? k_metrics : 1: mean over the users of   */
                                /* this call ([user_begin, user_end)) of every requested metric, NaN rows left out */
                                /* (numpy.nanmean of the per-user output -- the step that follows the call in the   */
                                /* reference's examples, examples/recometrics_example.ipynb cell 15); row q of the  */
                                /* table = metric q in the order of the signature (p, tp, r, ap, tap, ndcg, hit,    */
                                /* rr, roc_auc, pr_auc; the last two use column 0).  Computed on the device from    */
                                /* the metric rows in double, in a fixed order (results are reproducible); NaN for */
                                /* metrics that were not requested or have no valid user.  Host pointer, or device */
                                /* pointer when inputs_on_device.                                                   */
    int64_t *metric_counts;     /* optional out [10 * W]: users that entered each mean                              */
    int32_t has_nan_bits;       /* 1: every "NaN" the call writes into the metric outputs is the bit pattern nan_bits (low 32 bits   */
    int32_t filter_stats;       /*    for float calls) instead of a plain quiet NaN -- R's NA_REAL, src/recometrics.hpp:75-80.      */
    uint64_t nan_bits;          /* filter_stats = 1: fill timing.filter_err_ratio_max (costs a little in the exact stage)           */
    const int32_t *devices;     /* optional [n_devices] (host-pointer calls): CUDA device ordinals to spread the users of this ONE   */
    int32_t n_devices;          /* call over -- the reference's call uses every core (src/recometrics.hpp:428-437), this uses every   */
    int32_t reserved0;          /* listed GPU: contiguous user blocks, one host thread and stream set per GPU, item factors uploaded */
                                /* once and copied GPU-to-GPU, result rows written at the shard offsets.  n_devices = 0: `device`    */
                                /* alone, unless env RMB200_DEVICES ("all" or "0,1,2,...") names several.                            */
} rmb200_extra_t;

/* Drop-in for calc_metrics_float (src/recometrics_signatures.hpp:73-98).  Returns rmb200_status. */
RMB200_API int rmb200_calc_metrics_f32(
    const float *A, size_t lda, const float *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const float *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float *p_at_k, float *tp_at_k, float *r_at_k, float *ap_at_k, float *tap_at_k,
    float *ndcg_at_k, float *hit_at_k, float *rr_at_k, float *roc_auc, float *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed);

/* Drop-in for calc_metrics_double (src/recometrics_signatures.hpp:48-72). */
RMB200_API int rmb200_calc_metrics_f64(
    const double *A, size_t lda, const double *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const double *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double *p_at_k, double *tp_at_k, double *r_at_k, double *ap_at_k, double *tap_at_k,
    double *ndcg_at_k, double *hit_at_k, double *rr_at_k, double *roc_auc, double *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed);

/* Same call with two additions: item_biases[n] taken as a separate vector and added to the score
 * inside the scoring kernel (replaces the np.c_[A,1] / np.c_[B,bias] copies of
 * recometrics/__init__.py:548-551; NULL = none), and the extension block above. */
RMB200_API int rmb200_calc_metrics_ex_f32(
    const float *A, size_t lda, const float *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const float *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float *p_at_k, float *tp_at_k, float *r_at_k, float *ap_at_k, float *tap_at_k,
    float *ndcg_at_k, float *hit_at_k, float *rr_at_k, float *roc_auc, float *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const float *item_biases, const rmb200_extra_t *extra);

RMB200_API int rmb200_calc_metrics_ex_f64(
    const double *A, size_t lda, const double *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const double *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double *p_at_k, double *tp_at_k, double *r_at_k, double *ap_at_k, double *tap_at_k,
    double *ndcg_at_k, double *hit_at_k, double *rr_at_k, double *roc_auc, double *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const double *item_biases, const rmb200_extra_t *extra);

/* Item exposure of the ranked top-K lists of one call (zero-initialise, then set struct_size = sizeof(rmb200_exposure_t)).
 * Counted are the users of the call ([user_begin, user_end), every device of a multi-GPU call) whose ranked list is defined
 * (status 0: exactly the users whose topk_items row the call writes); each adds its min(k_metrics, candidates) listed items.
 * item_counts[j] = how many counted users have item j in their list = numpy.bincount(topk_items[topk_items >= 0], minlength=n).
 * The statistics depend only on the integer counts and are computed by rmb200_exposure_stats, on the host:
 *   coverage = items_covered / n;  gini = sum_i (2i - n - 1) c_(i) / (n * entries) over ALL n items, c ascending (RecBole's
 *   GiniIndex: one item holding everything gives (n - 1) / n, uniform exposure 0);  entropy_bits = -sum_{c_j > 0} p_j log2 p_j,
 *   p_j = c_j / entries.  With entries = 0: coverage 0, gini and entropy_bits NaN.  Statistics at k_metrics only (also
 *   when cumulative). */
typedef struct rmb200_exposure {
    int32_t struct_size;          /* = sizeof(rmb200_exposure_t)                                                          */
    int32_t reserved0;            /* padding                                                                              */
    int64_t *item_counts;         /* optional out [n]; a device pointer when extra->inputs_on_device                     */
    int64_t users, entries, items_covered;     /* out: counted users, listed entries (sum of item_counts), items with a count > 0 */
    double  coverage, gini, entropy_bits;      /* out                                                                     */
} rmb200_exposure_t;

/* rmb200_calc_metrics_ex_f32 / _f64 plus the item exposure of the call's ranked lists; exposure == NULL is exactly the _ex
 * call.  Requesting it counts as an output (a call with only `exposure` computes the ranked lists).  An interrupted call writes
 * nothing into `exposure`; an empty user block gives zero counts and the statistics of no entry. */
RMB200_API int rmb200_calc_metrics_exposure_f32(
    const float *A, size_t lda, const float *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const float *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float *p_at_k, float *tp_at_k, float *r_at_k, float *ap_at_k, float *tap_at_k,
    float *ndcg_at_k, float *hit_at_k, float *rr_at_k, float *roc_auc, float *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const float *item_biases, const rmb200_extra_t *extra, rmb200_exposure_t *exposure);

RMB200_API int rmb200_calc_metrics_exposure_f64(
    const double *A, size_t lda, const double *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const double *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double *p_at_k, double *tp_at_k, double *r_at_k, double *ap_at_k, double *tap_at_k,
    double *ndcg_at_k, double *hit_at_k, double *rr_at_k, double *roc_auc, double *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const double *item_biases, const rmb200_extra_t *extra, rmb200_exposure_t *exposure);

/* Host only, needs no GPU: entries, items_covered, coverage, gini and entropy_bits of `out` from counts[n] -- the function the
 * library itself uses after every call, so that counts summed over shards give the statistics of the whole run.  users and
 * item_counts are left alone.  RMB200_ERR_BAD_ARG for n <= 0, a negative count, a total beyond int64 or a wrong struct_size. */
RMB200_API int rmb200_exposure_stats(const int64_t *counts, int32_t n, rmb200_exposure_t *out);
RMB200_API int rmb200_sizeof_exposure(void);

/* Per-user beyond-accuracy metrics of the ranked top-K lists (zero-initialise, then set struct_size = sizeof(rmb200_beyond_t)).
 * A user's list is j_1..j_L with L = min(k_metrics, candidates) (the eligibility rules make it k_metrics); the user is defined
 * when L > 0 -- exactly the users whose topk_items row the call writes.  Every other user gets the NaN value (nan_bits is
 * honoured) in all three outputs.  pop_j = item_popularity[j] (e.g. rmb200_item_popularity over the first m rows of X_train),
 * U = popularity_users (e.g. m).  Column i of a cumulative row (i = L otherwise):
 *   Novelty@i = (1/i) sum_{r<=i} -log2((pop_{j_r} + 1) / (U + 1))            AvgPop@i = (1/i) sum_{r<=i} pop_{j_r}
 *   ILD@i     = 1 - 2 P_i / (i (i - 1)): the mean pairwise cosine distance of the first i items, over the unit rows
 *               u_r = b_{j_r} / ||b_{j_r}|| of B (item factors only, no bias; a zero row gives u_r = 0, distance 1), with
 *               P_r = P_{r-1} + u_r . (u_1 + ... + u_{r-1}).  ILD@1 is NaN.
 * Sums are accumulated in double in rank order and cast once: column k_metrics of a cumulative row is bit-identical to the
 * non-cumulative value, and a user's values do not depend on user_range, the batch size or the devices.  ILD needs
 * k <= 1024 (float) / 512 (double) factors (RMB200_ERR_UNSUPPORTED beyond).  RMB200_ERR_BAD_ARG, before any work: a wrong
 * struct_size; Novelty or AvgPop without item_popularity; popularity_users < 1; a count outside [0, popularity_users]. */
typedef struct rmb200_beyond {
    int32_t struct_size;          /* = sizeof(rmb200_beyond_t)                                                            */
    int32_t reserved0;            /* padding                                                                              */
    const int64_t *item_popularity;    /* [n]; needed for Novelty / AvgPop; a device pointer when extra->inputs_on_device */
    int64_t popularity_users;     /* U                                                                                    */
    void *novelty, *avg_popularity, *ild;   /* optional out: [m] or [m * k_metrics] (cumulative) of T, rows written at       */
                                  /* [user_begin, user_end); NULL = not requested; device pointers when inputs_on_device   */
    double  *means;               /* optional out [3 * W], W = cumulative ? k_metrics : 1: numpy.nanmean of every requested */
                                  /* row over the call's users (Novelty, AvgPop, ILD); NaN for a metric not requested      */
    int64_t *counts;              /* optional out [3 * W]: users that entered each mean                                     */
} rmb200_beyond_t;

/* rmb200_calc_metrics_exposure_f32 / _f64 plus the beyond-accuracy metrics; beyond == NULL is exactly the exposure call.
 * Requesting one of the three rows counts as an output.  An interrupted call writes no means. */
RMB200_API int rmb200_calc_metrics_beyond_f32(
    const float *A, size_t lda, const float *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const float *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float *p_at_k, float *tp_at_k, float *r_at_k, float *ap_at_k, float *tap_at_k,
    float *ndcg_at_k, float *hit_at_k, float *rr_at_k, float *roc_auc, float *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const float *item_biases, const rmb200_extra_t *extra, rmb200_exposure_t *exposure, rmb200_beyond_t *beyond);

RMB200_API int rmb200_calc_metrics_beyond_f64(
    const double *A, size_t lda, const double *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const double *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double *p_at_k, double *tp_at_k, double *r_at_k, double *ap_at_k, double *tap_at_k,
    double *ndcg_at_k, double *hit_at_k, double *rr_at_k, double *roc_auc, double *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const double *item_biases, const rmb200_extra_t *extra, rmb200_exposure_t *exposure, rmb200_beyond_t *beyond);

RMB200_API int rmb200_sizeof_beyond(void);

/* Per-user unexpectedness and serendipity of the ranked top-K lists against each user's training history (zero-initialise,
 * then set struct_size = sizeof(rmb200_serendipity_t)).  A user's list is j_1..j_L as for rmb200_beyond_t; H_u is the set of
 * stored entries of the user's X_train row (values are ignored: the entries the candidate exclusion removes) and
 * T_u = |H_u|.  u_j = b_j / ||b_j|| are ILD's unit rows of B (item factors only, no bias; a zero row gives u_j = 0).
 *   c_u   = sum_{t in H_u} u_t, summed in the row's order;   sim_r = (u_{j_r} . c_u) / T_u, the mean cosine similarity of the
 *           r-th listed item to the history;   rel_r = 1 when j_r is stored in the user's X_test row (any value), else 0 --
 *           the membership P@K and Hit@K count.  Column i of a cumulative row (i = L otherwise):
 *   Unexpectedness@i = (1/i) sum_{r<=i} (1 - sim_r)          Serendipity@i = (1/i) sum_{r<=i} rel_r (1 - sim_r)
 * (Serendipity is Microsoft Recommenders' user_serendipity with cosine similarity over B's rows and held-out membership as the
 * relevance; Unexpectedness is its relevance-free form.)  A user is defined when L > 0 and T_u > 0; every other user --
 * including cold-start users, who have a list but no history, and every user of a call without X_train entries -- gets the
 * NaN value (nan_bits is honoured) in both outputs.  Sums are accumulated in double in a fixed order and cast once: column
 * k_metrics of a cumulative row is bit-identical to the non-cumulative value, and a user's values do not depend on
 * user_range, the batch size or the devices.  Needs k <= 1024 (float) / 512 (double) factors (RMB200_ERR_UNSUPPORTED
 * beyond).  RMB200_ERR_BAD_ARG, before any work: a wrong struct_size. */
typedef struct rmb200_serendipity {
    int32_t struct_size;          /* = sizeof(rmb200_serendipity_t)                                                       */
    int32_t reserved0;            /* padding                                                                              */
    void *unexpectedness, *serendipity;   /* optional out: [m] or [m * k_metrics] (cumulative) of T, rows written at         */
                                  /* [user_begin, user_end); NULL = not requested; device pointers when inputs_on_device   */
    double  *means;               /* optional out [2 * W], W = cumulative ? k_metrics : 1: numpy.nanmean of every requested */
                                  /* row over the call's users (Unexpectedness, Serendipity); NaN for a row not requested  */
    int64_t *counts;              /* optional out [2 * W]: users that entered each mean                                     */
} rmb200_serendipity_t;

/* rmb200_calc_metrics_beyond_f32 / _f64 plus unexpectedness and serendipity; serendipity == NULL is exactly the beyond call.
 * Requesting one of the two rows counts as an output.  An interrupted call writes no means. */
RMB200_API int rmb200_calc_metrics_serendipity_f32(
    const float *A, size_t lda, const float *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const float *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float *p_at_k, float *tp_at_k, float *r_at_k, float *ap_at_k, float *tap_at_k,
    float *ndcg_at_k, float *hit_at_k, float *rr_at_k, float *roc_auc, float *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const float *item_biases, const rmb200_extra_t *extra, rmb200_exposure_t *exposure, rmb200_beyond_t *beyond,
    rmb200_serendipity_t *serendipity);

RMB200_API int rmb200_calc_metrics_serendipity_f64(
    const double *A, size_t lda, const double *B, size_t ldb,
    int32_t m, int32_t n, int32_t k,
    const int32_t *Xtrain_csr_p, const int32_t *Xtrain_csr_i,
    const int32_t *Xtest_csr_p, const int32_t *Xtest_csr_i, const double *Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double *p_at_k, double *tp_at_k, double *r_at_k, double *ap_at_k, double *tap_at_k,
    double *ndcg_at_k, double *hit_at_k, double *rr_at_k, double *roc_auc, double *pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test,
    int32_t nthreads, uint64_t seed,
    const double *item_biases, const rmb200_extra_t *extra, rmb200_exposure_t *exposure, rmb200_beyond_t *beyond,
    rmb200_serendipity_t *serendipity);

RMB200_API int rmb200_sizeof_serendipity(void);

/* Item popularity on the GPU: counts[j] = number of entries of item j in rows [row_begin, row_end) of a CSR matrix
 * (numpy.bincount of those rows' indices, minlength n).  indptr / indices / counts are device pointers on `device` when
 * inputs_on_device, else host pointers (the indices go up through the library's upload pipeline).  device < 0: env
 * RMB200_DEVICE or the current device. */
RMB200_API int rmb200_item_popularity(const int32_t *indptr, const int32_t *indices, int32_t row_begin, int32_t row_end,
    int32_t n, int32_t device, int32_t inputs_on_device, int64_t *counts);

/* Number of usable CUDA devices (0 = the library cannot compute). */
RMB200_API int rmb200_device_count(void);
/* RMB200_VERSION of the loaded library. */
RMB200_API int rmb200_version(void);
/* sizeof(rmb200_extra_t) / sizeof(rmb200_timing_t) as compiled into the library (bindings check their mirrors against it). */
RMB200_API int rmb200_sizeof_extra(void);
RMB200_API int rmb200_sizeof_timing(void);
/* Message of the last failing call on this thread ("" if none).  Never NULL. */
RMB200_API const char *rmb200_last_error(void);
/* Ask a running call to stop at the next user-batch boundary (what SIGINT does). */
RMB200_API void rmb200_request_interrupt(void);
/* Device scratch (operand images, candidate buffers) is cached between calls; this returns it to the driver.
 * RMB200_NO_POOL=1 in the environment disables the cache. */
RMB200_API void rmb200_release_workspace(void);
/* Measured FP32 / FP64 FMA throughput of `device` in TFLOP/s (register-resident FMA chains on all
 * SMs; the roofline denominator for the scoring kernel).  dtype_bytes = 4 or 8.  <0 on error. */
RMB200_API double rmb200_measure_fma_peak(int device, int dtype_bytes, double *elapsed_ms);

/* ---------------------------------------------------------------------------------------------------------------------
 * Train/test splitters -- the step BEFORE the evaluation path (SURVEY.md section 8, row f-4).
 *
 *   reference interface (replaced)                                                    this library
 *   --------------------------------------------------------------------------------  --------------------------------
 *   split_data_selected_users_float/_double  src/recometrics_signatures.hpp:100-130   rmb200_split_selected_users_f32/_f64
 *     (template src/recometrics.hpp:1015-1106; declared recometrics/wrapper.pyx:64-77, :147-160; called :541, :580)
 *   split_data_separate_users_float/_double  src/recometrics_signatures.hpp:132-178   rmb200_split_separate_users_f32/_f64
 *     (template src/recometrics.hpp:1201-1322; wrapper.pyx:79-100, :162-183; called :647, :732)
 *   split_data_joined_users_float/_double    src/recometrics_signatures.hpp:180-221   rmb200_split_joined_users_f32/_f64
 *     (template src/recometrics.hpp:1439-1505; wrapper.pyx:102-120, :185-203; called :677, :762)
 *
 * Same arguments in the same order as the reference; the reference's std::vector outputs become one rmb200_split_t of
 * library-owned host arrays, released with rmb200_split_free().  include/recometrics_b200_shim.hpp defines the reference's
 * functions (and the templates Rwrapper.cpp instantiates) on top.  test_fraction is a double for both value types, as in the
 * reference's templates; its *_float linkage functions declare it `const float` (src/recometrics_signatures.hpp:127, :174,
 * :217), i.e. round it to float first -- a binding that mirrors them passes (double)(float)fraction, as the shim's do.
 *
 * Division of work.  WHICH entries of a user are held out is decided by ONE sequential std::mt19937 stream that the
 * reference consumes user after user through std::shuffle (src/recometrics.hpp:1055-1060, :1223-1226): that replay is
 * sequential by the definition of the output and runs on the host (while X is on its way to the GPU), producing one byte
 * per entry.  Everything that touches the matrix itself -- ordering each row's entries by item id where the input is not
 * sorted, the stable partition of every row into its training and held-out part, the gather of the selected / remaining
 * users' rows and of the values -- runs on the GPU.  Results are entry-for-entry those of the reference built with the same
 * libstdc++.  No CPU fallback: without a CUDA device the calls return RMB200_ERR_NO_DEVICE.
 * Errors the reference throws as std::runtime_error come back as RMB200_ERR_RUNTIME with its message.
 * ------------------------------------------------------------------------------------------------------------------- */
typedef struct rmb200_csr_t {
    int32_t rows, cols;
    int64_t nnz;
    int32_t *indptr;            /* [rows + 1]; NULL when the matrix is not part of this split (or the reference leaves it empty) */
    int32_t *indices;           /* [nnz] */
    void *values;               /* [nnz] float or double */
} rmb200_csr_t;

typedef struct rmb200_split_t {
    rmb200_csr_t train, test, rem;   /* rem: separate users only */
    int32_t *users_test;        /* [n_users_test] rows of X taken as test users, ascending (NULL for selected_users) */
    int32_t n_users_test;
    int32_t value_bytes;        /* 4 or 8 */
    int32_t rows_sorted_on_device;   /* 1: some split row came with unsorted item ids and was ordered on the GPU */
    int32_t device;
    double total_ms, plan_ms, h2d_ms, kernel_ms, d2h_ms;   /* plan_ms: the sequential mt19937 replay on the host (overlaps h2d_ms) */
    int64_t kernel_launches, h2d_bytes, d2h_bytes;
    void *owner;                /* internal */
} rmb200_split_t;

RMB200_API int rmb200_split_selected_users_f32(const int32_t *X_csr_p, const int32_t *X_csr_i, const float *X_csr,
    int32_t m, int32_t n, double test_fraction, uint64_t seed, int32_t device, rmb200_split_t *out);
RMB200_API int rmb200_split_selected_users_f64(const int32_t *X_csr_p, const int32_t *X_csr_i, const double *X_csr,
    int32_t m, int32_t n, double test_fraction, uint64_t seed, int32_t device, rmb200_split_t *out);
RMB200_API int rmb200_split_separate_users_f32(const int32_t *X_csr_p, const int32_t *X_csr_i, const float *X_csr,
    int32_t m, int32_t n, int32_t n_users_test, double test_fraction, int consider_cold_start,
    int32_t min_items_pool, int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t *out);
RMB200_API int rmb200_split_separate_users_f64(const int32_t *X_csr_p, const int32_t *X_csr_i, const double *X_csr,
    int32_t m, int32_t n, int32_t n_users_test, double test_fraction, int consider_cold_start,
    int32_t min_items_pool, int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t *out);
RMB200_API int rmb200_split_joined_users_f32(const int32_t *X_csr_p, const int32_t *X_csr_i, const float *X_csr,
    int32_t m, int32_t n, int32_t n_users_test, double test_fraction, int consider_cold_start,
    int32_t min_items_pool, int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t *out);
RMB200_API int rmb200_split_joined_users_f64(const int32_t *X_csr_p, const int32_t *X_csr_i, const double *X_csr,
    int32_t m, int32_t n, int32_t n_users_test, double test_fraction, int consider_cold_start,
    int32_t min_items_pool, int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t *out);
/* The host half of the splitters on its own: the replay of the reference's mt19937 stream, with no matrix touched and no
 * GPU needed -- NOT a CPU path to a split (it returns no matrices), but the part of the result that can be checked on any
 * machine.  sample_users = 0: every row is split (selected_users); 1: the user sample of separate / joined users is drawn
 * first and written to users_test[<= m] / *n_users_out.  held[<= nnz] receives one byte per entry of the split rows, in row
 * order (1 = held out), *n_entries_out their number. */
RMB200_API int rmb200_split_plan(const int32_t *X_csr_p, int32_t m, int32_t n, int32_t sample_users, int32_t n_users_test,
    double test_fraction, int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, uint64_t seed,
    int32_t *users_test, int32_t *n_users_out, uint8_t *held, int64_t *n_entries_out);
/* Release the arrays of a split (safe on a zeroed or already released struct). */
RMB200_API void rmb200_split_free(rmb200_split_t *split);
RMB200_API int rmb200_sizeof_split(void);

#ifdef __cplusplus
}
#endif
#endif /* RECOMETRICS_B200_H */
