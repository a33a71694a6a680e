// api.cu -- C-ABI of librecometrics_b200.so and the host orchestration of one call.
//
// Stands where /root/reference/src/recometrics_instantiated.cpp:43-143 stands in the reference: the
// non-template entry points its bindings call (calc_metrics_float / calc_metrics_double), here
// driving the GPU instead of an OpenMP loop.  The host prologue mirrors
// /root/reference/src/recometrics.hpp:387-393 (clamps) and :426 / :488 / :964 (SIGINT latch).
#include "../../include/recometrics_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cfloat>
#include <cmath>
#include <csignal>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "metrics.cuh"
#include "prep.cuh"
#include "score_select.cuh"
#include "filter_select.cuh"
#include "exposure.cuh"
#include "beyond.cuh"
#include "full_order.h"
#include "runtime.h"

namespace {

using rmb::DevBuf;
using rmb::set_err;
using rmb::upload_rows;

std::atomic<int> g_interrupt{0};

extern "C" void rmb200_sigint_handler(int) { g_interrupt.store(1); }

// /root/reference/src/recometrics.hpp:126-174 (SignalSwitcher): swap the SIGINT handler for the
// duration of the call, poll the latch between user batches, restore + re-raise afterwards.
struct SignalLatch {
    void (*old_handler)(int) = SIG_DFL;
    bool active = false;
    explicit SignalLatch(bool engage = true)
    {
        if (!engage) return;
        g_interrupt.store(0);
        old_handler = std::signal(SIGINT, rmb200_sigint_handler);
        active = (old_handler != SIG_ERR);
    }
    void restore()
    {
        if (active) { std::signal(SIGINT, old_handler); active = false; }
    }
    ~SignalLatch() { restore(); }
};

inline int round_up(int x, int q) { return (x + q - 1) / q * q; }

struct PhaseTimer {
    cudaStream_t st;
    cudaEvent_t a = nullptr, b = nullptr;
    explicit PhaseTimer(cudaStream_t s) : st(s) { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~PhaseTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    void start() { cudaEventRecord(a, st); }
    void stop(double& acc)
    {
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        acc += ms;
    }
};

__global__ void rebase_indptr_kernel(const int* __restrict__ src, const int lo, int* __restrict__ dst, const int cnt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cnt) dst[i] = src[i] - lo;
}

// One call spread over several GPUs (rmb200_extra_t::devices / RMB200_DEVICES): every device runs run_call() on its own
// contiguous block of users from its own host thread.  The only thing the devices share is the item-factor matrix: device
// g uploads the g-th slice of its rows over its own PCIe link and fetches the other slices from its peers' memory
// (NVLink), instead of G uploads of the whole matrix.  The threads meet twice: slices uploaded / slices fetched.
struct MultiCtx {
    int G = 0;
    std::mutex mu;
    std::condition_variable cv;
    int arrived[2] = {0, 0};
    int departed = 0;
    bool failed = false;
    void* Bptr[rmb::MAX_DEVICES] = {};
    int Bdev[rmb::MAX_DEVICES] = {};
    // false: a peer failed (the caller gives up as well)
    bool meet(int phase)
    {
        std::unique_lock<std::mutex> lk(mu);
        arrived[phase]++;
        cv.notify_all();
        cv.wait(lk, [&] { return arrived[phase] + departed >= G; });
        return !failed;
    }
    void depart(bool fail)          // the device's thread is done (a thread that fails early stands in for its later meetings)
    {
        std::lock_guard<std::mutex> lk(mu);
        departed++;
        if (fail) failed = true;
        cv.notify_all();
    }
};

template <typename T>
struct CallArgs {
    MultiCtx* mc = nullptr; int mc_rank = 0;
    const T* A; size_t lda; const T* B; size_t ldb;
    int m, n, k;
    const int32_t *trp, *tri, *tep, *tei; const T* tev;
    int K, cumulative, noise;
    T* out[10];   // p tp r ap tap ndcg hit rr roc pr
    int consider_cold_start, min_items_pool, min_pos_test;
    uint64_t seed;
    const T* bias;
    const rmb200_extra_t* ex;
    rmb200_exposure_t* expo = nullptr;   // item exposure of the ranked lists (exposure.cuh); null: not requested
    rmb200_beyond_t* bey = nullptr;      // Novelty / AvgPop / ILD of the ranked lists (beyond.cuh); null: not requested
};

template <typename T, int C, bool AUC>
cudaError_t launch_score_select_inst(const rmb::ScoreSelectParams<T>& P, int n_rows, int slices, cudaStream_t st)
{
    auto kern = rmb::score_select_kernel<T, C, AUC>;
    const size_t smem = rmb::score_select_smem_bytes<T, AUC>();
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<dim3((n_rows + rmb::BM - 1) / rmb::BM, slices), AUC ? rmb::AUC_THREADS : rmb::NTHREADS, smem, st>>>(P);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_score_select(const rmb::ScoreSelectParams<T>& P, int C, bool auc, int n_rows, int slices, cudaStream_t st)
{
    if (C == 256) return auc ? launch_score_select_inst<T, 256, true>(P, n_rows, slices, st)
                             : launch_score_select_inst<T, 256, false>(P, n_rows, slices, st);
    if (C == 512) return auc ? launch_score_select_inst<T, 512, true>(P, n_rows, slices, st)
                             : launch_score_select_inst<T, 512, false>(P, n_rows, slices, st);
    return auc ? launch_score_select_inst<T, 1024, true>(P, n_rows, slices, st)
               : launch_score_select_inst<T, 1024, false>(P, n_rows, slices, st);
}

template <int C>
cudaError_t launch_filter_inst(const rmb::FilterParams& P, int n_user_tiles, cudaStream_t st)
{
    const size_t smem = rmb::filter_smem_bytes(P.KB, P.stages);
    auto kern = rmb::filter_select_kernel<C>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<n_user_tiles, rmb::F_THREADS, smem, st>>>(P);
    return cudaGetLastError();
}

inline cudaError_t launch_filter_select(const rmb::FilterParams& P, int C, int n_user_tiles, cudaStream_t st)
{
    if (C == 256) return launch_filter_inst<256>(P, n_user_tiles, st);
    if (C == 512) return launch_filter_inst<512>(P, n_user_tiles, st);
    return launch_filter_inst<1024>(P, n_user_tiles, st);
}

struct NoiseArgs { int on; unsigned long long seed_user0; const int* trp; const int* tri; int n; };

template <typename T, int C>
cudaError_t launch_exact_topk_inst(const uint2* capx, T* cs, int* ci, int* cc, int nb, int user0, const T* At, int p_pad, int p,
                                   const T* Brow, size_t ldb, const T* bias, int* uflags, int K, const NoiseArgs& nz,
                                   const rmb::FilterErrStat& es, cudaStream_t st)
{
    const int blocks = (nb + rmb::EXACT_WARPS - 1) / rmb::EXACT_WARPS;
    const size_t staging = (rmb::exact_topk_smem_bytes(p_pad, sizeof(T)) + 15) & ~size_t(15);
    const size_t mt_bytes = nz.on ? (size_t)rmb::EXACT_WARPS * rmb::MT_N * sizeof(unsigned) : 0;   // generator states (tie_noise.cuh)
    if (staging + mt_bytes <= 100 * 1024) {       // two blocks per SM
        // 16-byte copies when every factor row starts on a 16-byte boundary and is a multiple of 16 bytes long
        constexpr int V = 16 / (int)sizeof(T);
        const bool vec = (p % V == 0) && (ldb % V == 0) && ((reinterpret_cast<uintptr_t>(Brow) & 15) == 0);
        auto kern = vec ? rmb::exact_topk_kernel<T, C, 2> : rmb::exact_topk_kernel<T, C, 1>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(staging + mt_bytes));
        if (e != cudaSuccess) return e;
        kern<<<blocks, rmb::EXACT_WARPS * 32, staging + mt_bytes, st>>>(capx, cs, ci, cc, nb, user0, At, p_pad, p, Brow, ldb, bias, uflags, K,
                                                                        nz.on, nz.seed_user0, staging, nz.trp, nz.tri, nz.n, es);
    } else {
        rmb::exact_topk_kernel<T, C, 0><<<blocks, rmb::EXACT_WARPS * 32, mt_bytes, st>>>(capx, cs, ci, cc, nb, user0, At, p_pad, p, Brow, ldb, bias, uflags, K,
                                                                                             nz.on, nz.seed_user0, (size_t)0, nz.trp, nz.tri, nz.n, es);
    }
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_exact_topk(const uint2* capx, T* cs, int* ci, int* cc, int C, int nb, int user0, const T* At, int p_pad, int p,
                              const T* Brow, size_t ldb, const T* bias, int* uflags, int K, const NoiseArgs& nz,
                              const rmb::FilterErrStat& es, cudaStream_t st)
{
    if (C == 256) return launch_exact_topk_inst<T, 256>(capx, cs, ci, cc, nb, user0, At, p_pad, p, Brow, ldb, bias, uflags, K, nz, es, st);
    if (C == 512) return launch_exact_topk_inst<T, 512>(capx, cs, ci, cc, nb, user0, At, p_pad, p, Brow, ldb, bias, uflags, K, nz, es, st);
    return launch_exact_topk_inst<T, 1024>(capx, cs, ci, cc, nb, user0, At, p_pad, p, Brow, ldb, bias, uflags, K, nz, es, st);
}

// order the <= K survivors of every user (warp per user, bitonic network sized to K)
template <typename T>
cudaError_t launch_rank_topk(T* cs, int* ci, const int* cc, int C, int nb, int K, cudaStream_t st)
{
    const int blocks = (nb + 7) / 8;
    if (K <= 32) rmb::rank_topk_kernel<T, 1><<<blocks, 256, 0, st>>>(cs, ci, cc, C, nb);
    else if (K <= 64) rmb::rank_topk_kernel<T, 2><<<blocks, 256, 0, st>>>(cs, ci, cc, C, nb);
    else if (K <= 128) rmb::rank_topk_kernel<T, 4><<<blocks, 256, 0, st>>>(cs, ci, cc, C, nb);
    else if (K <= 256) rmb::rank_topk_kernel<T, 8><<<blocks, 256, 0, st>>>(cs, ci, cc, C, nb);
    else rmb::rank_topk_kernel<T, 16><<<blocks, 256, 0, st>>>(cs, ci, cc, C, nb);
    return cudaGetLastError();
}


// The user factors are uploaded one user batch ahead, on a stream of their own, into two alternating staging buffers:
// the upload of batch b+1 runs while the scoring kernel of batch b does.  ready[s]: the upload into buffer s has landed;
// freed[s]: the kernels that read buffer s have run.
struct PrefetchStream {
    cudaStream_t s = nullptr;
    cudaEvent_t ready[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr};
    cudaEvent_t test_rows = nullptr;                 // the held-out CSR arrays (read first by the metrics kernel) have landed
    bool freed_valid[2] = {false, false}, test_rows_pending = false;
    cudaError_t init()
    {
        cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        for (int i = 0; i < 2 && e == cudaSuccess; i++) {
            e = cudaEventCreateWithFlags(&ready[i], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&freed[i], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&test_rows, cudaEventDisableTiming);
        return e;
    }
    ~PrefetchStream()
    {
        if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }     // nothing may still be writing the staging buffers
        for (int i = 0; i < 2; i++) { if (ready[i]) cudaEventDestroy(ready[i]); if (freed[i]) cudaEventDestroy(freed[i]); }
        if (test_rows) cudaEventDestroy(test_rows);
    }
};

// The metric rows of a user batch go back to the host on a stream of their own, out of two alternating sets of staging
// buffers: the copy of batch b runs while batch b+1 is scored (cumulative rows are m x K values per metric: 400 MB at cfg5).
// ready[s]: the kernels writing set s have run; copied[s]: its copies have landed (the set may be written again).
struct ResultStream {
    cudaStream_t s = nullptr;
    cudaEvent_t ready[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    bool copied_valid[2] = {false, false};
    cudaError_t init()
    {
        cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        for (int i = 0; i < 2 && e == cudaSuccess; i++) {
            e = cudaEventCreateWithFlags(&ready[i], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming);
        }
        return e;
    }
    ~ResultStream()
    {
        if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }       // nothing may still be reading the staging buffers
        for (int i = 0; i < 2; i++) { if (ready[i]) cudaEventDestroy(ready[i]); if (copied[i]) cudaEventDestroy(copied[i]); }
    }
};

inline const rmb200_extra_t* ex_or_default(const rmb200_extra_t* ex)
{
    static const rmb200_extra_t dflt = []() {
        rmb200_extra_t e;
        std::memset(&e, 0, sizeof(e));
        e.struct_size = (int32_t)sizeof(e);
        e.device = -1;
        return e;
    }();
    return ex ? ex : &dflt;
}

// The users [*ub, *ue) of a call: rmb200_extra_t::user_begin / user_end; 0, 0 = all m users, user_end < 0 = none.
int user_range(const rmb200_extra_t* ex, int m, int* ub, int* ue)
{
    *ub = 0; *ue = ex->user_end < 0 ? 0 : m;                             // user_end < 0: explicit empty block
    if (ex->user_end >= 0 && (ex->user_begin != 0 || ex->user_end != 0)) { *ub = ex->user_begin; *ue = ex->user_end; }
    if (*ub < 0 || *ue > m || *ub > *ue) { set_err("bad argument", "user range outside [0, m]"); return RMB200_ERR_BAD_ARG; }
    return RMB200_OK;
}

// The statistics of item counts (exposure.cuh) into *out: what every call that asks for them and rmb200_exposure_stats do
int exposure_stats(const int64_t* counts, int n, rmb200_exposure_t* out)
{
    if (!rmb::exposure_stats_host(counts, n, out)) { set_err("bad argument", "item counts: n <= 0, a negative count or a total beyond int64"); return RMB200_ERR_BAD_ARG; }
    return RMB200_OK;
}

// The exposure of a call that evaluates nobody (an empty user block): zero counts, no user
int exposure_of_nobody(rmb200_exposure_t* expo, int n, bool counts_on_device)
{
    std::vector<int64_t> zero((size_t)n, 0);
    if (expo->item_counts) {
        if (counts_on_device) CK(cudaMemset(expo->item_counts, 0, (size_t)n * sizeof(int64_t)));
        else std::memset(expo->item_counts, 0, (size_t)n * sizeof(int64_t));
    }
    expo->users = 0;
    return exposure_stats(zero.data(), n, expo);
}

// One per-user output of a call: the caller's rows (host or device; null: not requested) at row_bytes per user; a host
// output is written into one of two result sets and copied out behind its batch (Call::send_results)
struct RowOut {
    void* base = nullptr;
    size_t row_bytes = 0;
    bool skippable = false;                     // left on the device by rmb200_extra_t::skip_row_copy (metric and beyond rows)
    DevBuf staged[2];
    void set(void* p, size_t bytes, bool skip) { base = p; row_bytes = bytes; skippable = skip; }
};

// One [slots][W] table of means / counts over the users of a call (the first `wide` slots have W columns, the others one):
// slot q reduces row output first_row + q into the caller's means / counts (host or device; both null: not requested)
struct MeanTable {
    int slots = 0, wide = 0, first_row = 0;
    double* means = nullptr; long long* counts = nullptr;
    DevBuf part_sum, part_cnt;                  // per 256 users of every batch (metric_partial_kernel), added up in order at the end
    DevBuf d_means, d_counts;                   // the final values of host outputs
    bool on() const { return means || counts; }
    void set(int s, int w, int row0, double* m, int64_t* c) { slots = s; wide = w; first_row = row0; means = m; counts = reinterpret_cast<long long*>(c); }
};

// One evaluation call on one device.  plan() makes every decision that needs only the arguments and the device; the resident
// steps (csr_slices .. batch_buffers) put on the device what every batch reads; run_batch() evaluates one batch of UB users.
// All of it runs on the legacy default stream `st`, but the uploads of host inputs (PrefetchStream) and result copies (ResultStream).
template <typename T>
struct Call {
    static constexpr int BN = rmb::NumTraits<T>::BN;
    // filter counters (d_overflow): [0] users handed back to the FMA path, [1] users that took the retry pass, [6] length of the hand-back list
    static constexpr int OVERFLOW_INTS = 7;
    struct Batch {   // users [b0, b0 + nb) of the call; slot: staging buffer of their factors (host inputs) and result set (host outputs)
        int b0, nb, nb_pad, slot; bool prefetched = false;
        const T* Asrc = nullptr; size_t Ald = 0;     // the batch's user factors, row-major on the device
    };
    const CallArgs<T>& a;
    const rmb200_extra_t* ex;
    const bool on_dev, nested;                  // nested: one device's share of a multi-GPU call (run_multi)
    const int dev, ub, mr, K;                   // mr users from ub ("shard"); device-side rows are shard-local
    cudaStream_t st = nullptr;                  // legacy default stream: ordered after the caller's default-stream work
    PhaseTimer pt{st}, pk{st};                  // phases; the dominant scoring kernel alone
    rmb200_timing_t tm;
    // the row outputs, in the order their copies leave: the 10 metrics (MetricsParams order), status, top-K items and scores,
    // Novelty / AvgPop / ILD
    static constexpr int RO_STATUS = 10, RO_TOPK_ITEMS = 11, RO_TOPK_SCORES = 12, RO_BEYOND = 13, ROW_OUTS = 16;
    // ---- the plan ----
    int mip = 0, mpt = 0, C = 0, p_pad = 0, n_pad = 0, n_pad128 = 0, KB = 0, f_stages = 0, nsm = 148, UB = 0, fma_slices = 1, mean_W = 1;
    size_t rs = 1;
    T nan_value = std::numeric_limits<T>::quiet_NaN();
    bool want_roc = false, want_pr = false, count_ranks = false, want_filter_stats = false, want_exposure = false;
    bool want_pop = false, want_ild = false, want_beyond = false;   // beyond.cuh
    int unit_pitch = 0, unit_nch = 0;           // ILD: row pitch of the unit-row image (elements), 16-byte chunks per lane
    RowOut row_outs[ROW_OUTS];
    MeanTable mean_tables[2];                   // the 10 metrics {10, 8}; Novelty / AvgPop / ILD {3, 3}
    bool use_full = false, use_tensor = false, fma_counts_first = false, noise_handback = false;
    int f_sample_tiles = 0, f_sample_stride = 1, f_sample_rank = 0;
    int fo_chunk = 0; size_t fo_bytes = 0;
    // ---- resident state ----
    int lo_hi[4] = {0, 0, 0, 0};                // trp[ub], trp[ue], tep[ub], tep[ue]
    size_t nnz_tr = 0, nnz_te = 0;
    const int *trp_d = nullptr, *tep_d = nullptr, *tri_d = nullptr, *tei_d = nullptr;
    const T *tev_d = nullptr, *bias_d = nullptr, *Bsrc = nullptr; size_t Bld = 0;    // Bsrc: item factors, row-major on the device
    long long* pos_rank_d = nullptr;
    bool have_Bt = false; int mean_block0 = 0;
    DevBuf d_trp, d_tri, d_tep, d_tei, d_tev, d_Arow[2];
    DevBuf d_Bt, d_bias, d_Brow, d_Bb, d_maxbn, d_chunkn;
    DevBuf d_status, d_flags, d_umin, d_pos_raw, d_pos_sorted, d_pos_perm, d_pos_item, d_auc, d_log2, d_pos_rank;
    DevBuf d_fo, d_near, d_nz_mark, d_nz_list, d_nz_cnt, d_At_nz;
    DevBuf d_At, d_cs, d_ci, d_cc, d_Ab, d_anorm;
    DevBuf d_capx, d_overflow, d_fb_list, d_At_fb;
    DevBuf d_expo_hist, d_list_len, d_expo_counts;
    DevBuf d_pop, d_poptab, d_pop_bad, d_unit;
    const long long* pop_d = nullptr;           // the caller's popularity counts on the device
    PrefetchStream pf;                          // (declared after the buffers they fill or read: destroyed, i.e. drained, before them)
    ResultStream rsx;
    Call(const CallArgs<T>& args, int device, int user_begin, int users) : a(args), ex(args.ex), on_dev(args.ex->inputs_on_device != 0),
        nested(args.mc != nullptr), dev(device), ub(user_begin), mr(users), K(args.K) { std::memset(&tm, 0, sizeof(tm)); }
    int plan()
    {
        using namespace rmb;
        // hpp:391-393
        mip = a.min_items_pool < K ? K : a.min_items_pool;
        if (mip < 2) mip = 2;
        mpt = a.min_pos_test;
        if (!ex->strict_min_pos_test) mpt = mpt < 1 ? mpt : 1;   // std::min(min_pos_test, 1): quirk Q1
        // what a "NaN" written into the outputs looks like: a quiet NaN, or the caller's bit pattern (R: NA_REAL, hpp:75-80)
        if (ex->has_nan_bits) {
            if (sizeof(T) == 8) { const uint64_t b = ex->nan_bits; std::memcpy(&nan_value, &b, 8); }
            else { const uint32_t b = (uint32_t)ex->nan_bits; std::memcpy(&nan_value, &b, 4); }
            if (nan_value == nan_value) { set_err("bad argument", "rmb200_extra_t::nan_bits is not a NaN"); return RMB200_ERR_BAD_ARG; }
        }
        // candidate buffer: K kept + 128 appended per tile + head-room between two cuts (the tensor-core filter keeps
        // the slack band below the K-th best as well: about 2.5 K entries on Gaussian scores, so it gets more room)
        C = (K <= 64) ? 256 : (K <= 192 ? 512 : 1024);
        want_roc = a.out[8] != nullptr; want_pr = a.out[9] != nullptr;
        count_ranks = want_roc || want_pr || ex->pos_rank;
        want_filter_stats = ex->filter_stats != 0;
        want_exposure = a.expo != nullptr;
        rs = a.cumulative ? (size_t)K : 1;
        mean_W = a.cumulative ? K : 1;
        for (int q = 0; q < 10; q++) row_outs[q].set(a.out[q], (q < 8 ? rs : 1) * sizeof(T), true);
        row_outs[RO_STATUS].set(ex->status, sizeof(int), false);
        row_outs[RO_TOPK_ITEMS].set(ex->topk_items, (size_t)K * sizeof(int), false);
        row_outs[RO_TOPK_SCORES].set(ex->topk_scores, (size_t)K * sizeof(T), false);
        mean_tables[0].set(10, 8, 0, ex->metric_means, ex->metric_counts);
        if (a.bey) {
            void* const bey[3] = {a.bey->novelty, a.bey->avg_popularity, a.bey->ild};
            for (int q = 0; q < 3; q++) row_outs[RO_BEYOND + q].set(bey[q], rs * sizeof(T), true);
            want_pop = bey[0] || bey[1];
            want_ild = bey[2] != nullptr;
            want_beyond = want_pop || want_ild;
            if (want_beyond) mean_tables[1].set(3, 3, RO_BEYOND, a.bey->means, a.bey->counts);
        }
        if (want_ild) {            // lane l of beyond_accuracy_kernel holds 16-byte chunks l, l + 32, ... of a unit row: 1, 2, 4 or 8
            constexpr int V = 16 / (int)sizeof(T);
            unit_pitch = round_up(a.k, V);
            const int chunks = unit_pitch / V;
            unit_nch = chunks <= 32 ? 1 : chunks <= 64 ? 2 : chunks <= 128 ? 4 : chunks <= 256 ? 8 : 0;
            if (!unit_nch) { set_err("unsupported", "ILD needs k <= 1024 (float) / 512 (double) factors"); return RMB200_ERR_UNSUPPORTED; }
        }
        p_pad = round_up(a.k, KPAD);
        n_pad = round_up(a.n, BN);
        // ---- which scoring path: tensor-core filter + exact re-scoring (top-K only), or FMA tiles ----
        int path_req = ex->scoring_path;                                 // 0 auto, 1 fma, 2 tensor
        if (path_req == 0) if (const char* env = std::getenv("RMB200_PATH")) {
            if (!std::strcmp(env, "fma")) path_req = 1; else if (!std::strcmp(env, "tensor")) path_req = 2; else if (!std::strcmp(env, "full")) path_req = 3;
        }
        // k_metrics beyond what the selection kernels' candidate buffers hold: the full-order path (full_order.cu)
        use_full = path_req == 3 || K > RMB200_MAX_K;
        if (use_full && (ex->scoring_path == 1 || ex->scoring_path == 2)) { set_err("unsupported", "scoring_path fma / tensor need k_metrics <= RMB200_MAX_K (384)"); return RMB200_ERR_UNSUPPORTED; }
        if (use_full) path_req = 3;                                      // (an RMB200_PATH preference does not apply)
        KB = round_up(a.k + (a.bias ? 1 : 0), 16);                       // fp16 factors per row (bias = one more factor)
        // A tile + ring stages + barriers + row state within the 227 KB a CTA can have
        const long long tile = (long long)KB * 256, budget = 227 * 1024 - (long long)filter_smem_fixed_bytes();
        f_stages = (int)(budget / tile) - 1;
        if (f_stages > F_MAX_STAGES) f_stages = F_MAX_STAGES;
        // With rank counting (ROC/PR-AUC) every score has to be exact: the FMA tiles do everything.  Exception: with the
        // reference's tie-breaking noise the ranked top-K comes from the tensor path as well (its exact stage is where the
        // noise is applied, tie_noise.cuh), after the FMA pass has counted the ranks.
        const bool tensor_shape_ok = f_stages >= 2 && K <= 256 && !use_full;
        const bool tensor_ok = tensor_shape_ok && (!count_ranks || a.noise);
        if (path_req == 2 && !tensor_ok) { set_err("unsupported", "scoring_path=tensor needs no ROC/PR-AUC (rank counting), k <= ~400 and k_metrics <= 256"); return RMB200_ERR_UNSUPPORTED; }
        use_tensor = tensor_ok && path_req != 1;
        // break_ties_with_noise (the reference's default) where the tensor path's exact stage cannot apply it -- shapes only the FMA
        // tiles handle (k_metrics 257..384, more than ~400 factors) or an RMB200_PATH=fma preference: the full-order path, which
        // adds every candidate's draw before sorting.  Only an explicit scoring_path = 1 keeps the FMA tiles (noise-free order).
        if (a.noise && !use_tensor && !use_full && ex->scoring_path != 1) use_full = true;
        fma_counts_first = use_tensor && count_ranks;
        // ... and inside the rank counts (ROC/PR-AUC with the noise): the FMA tiles count on the noise-free scores and report, per
        // held-out item, the candidates within the noise's reach; users for whom the noise decides a rank are handed to the full-order path
        noise_handback = a.noise && count_ranks && !use_full;
        tm.scoring_path = use_full ? 3 : (use_tensor ? 2 : 1);
        if (use_tensor) C = (K <= 32) ? 256 : (K <= 128 ? 512 : 1024);
        if (use_full) C = round_up(K < a.n ? K : a.n, 32);              // row pitch of the ranked lists
        n_pad128 = round_up(a.n, 128);
        // ---- user batches ----
        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
        const int wave_users = nsm * BM;                       // one CTA (128 users) per SM
        UB = 8 * wave_users;                                   // users per batch: 8 full waves ...
        // ... 4 when the filter's item image is much larger than the L2 (256 MB at 1M items x 128 factors): the CTAs of a longer
        // launch drift further apart and re-stream the item tiles from HBM (cfg4: 3.16 M users/s at 4 waves, 3.10 at 8, 2.96 at
        // 16, 2.76 with all 1M users in one launch; smaller catalogues prefer 8; profiles/r02_batch_size.txt)
        if (use_tensor && (size_t)n_pad128 * KB * sizeof(__half) > (size_t)160 << 20) UB = 4 * wave_users;
        if (const char* env = std::getenv("RMB200_BATCH_USERS")) { const int v = std::atoi(env); if (v > 0) UB = round_up(v, BM); }
        if (use_full) {
            // ranked lists (K entries per user) and cumulative rows (K columns per metric) of a batch within ~2 GB
            const long long per_user = (long long)C * (long long)(sizeof(T) + 4) + (a.cumulative ? 8ll * K * (long long)sizeof(T) : 0);
            long long cap = (2ll << 30) / (per_user > 0 ? per_user : 1);
            cap = cap / BM * BM;
            if (cap < BM) cap = BM;
            if (UB > cap) UB = (int)cap;
        }
        if (UB > round_up(mr, BM)) UB = round_up(mr, BM);
        if (use_full) full_order_plan(a.n, (int)sizeof(T), UB, &fo_chunk, &fo_bytes);
        // sampled threshold guess of the filter (filter_select.cuh, pass 0): every stride-th item tile, about 7/K of the
        // catalogue (1/16 .. 1/8); the guess is the r-th best of the sample with r = the smallest rank for which
        // P(Poisson(K * sample / n) >= r) <= 1e-6, i.e. fewer than K items of the whole catalogue reach it about once
        // in a million users (those users' CTAs walk the catalogue a second time; results never depend on the guess)
        if (use_tensor) {
            const int NT = (a.n + 127) / 128;
            if (NT >= 512) {                                                  // (64K items and up)
                double frac = 7.0 / K;
                if (frac < 1.0 / 16) frac = 1.0 / 16;
                if (frac > 1.0 / 8) frac = 1.0 / 8;
                const int stride = (int)(1.0 / frac);
                const int ns = NT / stride;                                  // tiles 0, stride, ..., (ns-1)*stride: all full tiles
                const double lam = (double)K * ((double)ns * 128.0) / (double)a.n;
                double term = std::exp(-lam), cdf = 0.0;                     // P(X <= r-1), X ~ Poisson(lam)
                int r = 0;
                while (r < 4096) { cdf += term; r++; term *= lam / r; if (1.0 - cdf <= 1e-6) break; }
                if (const char* env = std::getenv("RMB200_SAMPLE_RANK")) { const int v = std::atoi(env); if (v >= 1) r = v; }
                // (the guess is the r-th largest of up to min(C / 4, 128) group maxima of the sample, filter_select.cuh)
                const int groups = (C / 4 < 128 ? C / 4 : 128) < ns ? (C / 4 < 128 ? C / 4 : 128) : ns;
                if (ns >= 8 && 2 * r <= groups) { f_sample_tiles = ns; f_sample_stride = stride; f_sample_rank = r; }
            }
        }
        // A call with fewer user tiles than SMs (small m) cuts the catalogue into item ranges on the FMA tiles: one CTA per (user tile,
        // range), every range keeping its own best K, joined afterwards (merge_slices_kernel); rank counts are added atomically.
        if (!use_full) {
            const int tiles = UB / BM, NT_all = (a.n + BN - 1) / BN;
            int sl = tiles > 0 ? nsm / tiles : 1;
            if (sl > NT_all / 8) sl = NT_all / 8;                       // (at least eight item tiles per range)
            if (sl > C / K) sl = C / K;                                 // the joined heads fit one row ...
            if (sl > 512 / K) sl = 512 / K;                             // ... and the final sort
            if (sl > 1) fma_slices = sl;
        }
        return RMB200_OK;
    }
    // CSR slices of users [ub, ue), index pointers re-based to the slice
    int csr_slices()
    {
        const int* ends[4] = {a.trp + ub, a.trp + ub + mr, a.tep + ub, a.tep + ub + mr};
        for (int i = 0; i < 4; i++)
            if (on_dev) CK(cudaMemcpy(&lo_hi[i], ends[i], sizeof(int), cudaMemcpyDeviceToHost)); else lo_hi[i] = *ends[i];
        if (lo_hi[1] < lo_hi[0] || lo_hi[3] < lo_hi[2]) { set_err("bad argument", "CSR index pointers decrease"); return RMB200_ERR_BAD_ARG; }
        nnz_tr = (size_t)(lo_hi[1] - lo_hi[0]);
        nnz_te = (size_t)(lo_hi[3] - lo_hi[2]);
        if ((nnz_tr && !a.tri) || (nnz_te && !a.tei)) { set_err("bad argument", "CSR indices missing"); return RMB200_ERR_BAD_ARG; }
        if (!on_dev) CK(pf.init());
        CK(d_trp.alloc((size_t)(mr + 1) * sizeof(int)));
        CK(d_tep.alloc((size_t)(mr + 1) * sizeof(int)));
        pt.start();
        if (!on_dev) {
            std::vector<int> tmp1((size_t)mr + 1), tmp2((size_t)mr + 1);
            for (int i = 0; i <= mr; i++) { tmp1[i] = a.trp[ub + i] - lo_hi[0]; tmp2[i] = a.tep[ub + i] - lo_hi[2]; }
            CK(cudaMemcpyAsync(d_trp.p, tmp1.data(), tmp1.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(d_tep.p, tmp2.data(), tmp2.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            CK(d_tri.alloc(nnz_tr * sizeof(int)));
            CK(d_tei.alloc(nnz_te * sizeof(int)));
            if (nnz_tr) CK(upload_rows(d_tri.p, a.tri + lo_hi[0], nnz_tr * sizeof(int), nnz_tr * sizeof(int), 1, st));
            // the held-out rows are not needed before the first batch's metrics (rank counting: its first scoring step): they
            // go up on the prefetch stream, behind the item factors on the link instead of in front of them
            if (nnz_te) CK(upload_rows(d_tei.p, a.tei + lo_hi[2], nnz_te * sizeof(int), nnz_te * sizeof(int), 1, pf.s));
            if (a.tev) {
                CK(d_tev.alloc(nnz_te * sizeof(T)));
                if (nnz_te) CK(upload_rows(d_tev.p, a.tev + lo_hi[2], nnz_te * sizeof(T), nnz_te * sizeof(T), 1, pf.s));
                tev_d = d_tev.as<T>();
            }
            CK(cudaEventRecord(pf.test_rows, pf.s));
            pf.test_rows_pending = true;
            CK(cudaStreamSynchronize(st));   // tmp1/tmp2 go out of scope
            tri_d = d_tri.as<int>(); tei_d = d_tei.as<int>();
            tm.h2d_bytes += (int64_t)(2 * (size_t)(mr + 1) * sizeof(int) + (nnz_tr + nnz_te) * sizeof(int) + (a.tev ? nnz_te * sizeof(T) : 0));
            pt.stop(tm.h2d_ms);
        } else {
            rebase_indptr_kernel<<<(mr + 1 + 255) / 256, 256, 0, st>>>(a.trp + ub, lo_hi[0], d_trp.as<int>(), mr + 1);
            rebase_indptr_kernel<<<(mr + 1 + 255) / 256, 256, 0, st>>>(a.tep + ub, lo_hi[2], d_tep.as<int>(), mr + 1);
            TRY(launched(2));
            tri_d = a.tri ? a.tri + lo_hi[0] : nullptr;
            tei_d = a.tei ? a.tei + lo_hi[2] : nullptr;
            tev_d = a.tev ? a.tev + lo_hi[2] : nullptr;
            pt.stop(tm.prep_ms);
        }
        trp_d = d_trp.as<int>(); tep_d = d_tep.as<int>();
        return RMB200_OK;
    }
    // item factors: row-major on the device, then the operand image of the FMA path where it scores
    int item_factors()
    {
        if (!on_dev) {
            CK(d_Brow.alloc((size_t)a.n * a.k * sizeof(T)));
            pt.start();
            TRY(upload_item_rows());
            pt.stop(tm.h2d_ms);
            Bsrc = d_Brow.as<T>(); Bld = (size_t)a.k;
        } else { Bsrc = a.B; Bld = a.ldb; }
        if (want_ild) TRY(unit_rows());                 // (from the complete rows: after the peer fetch, before d_Brow goes)
        if (!use_tensor || fma_counts_first) TRY(ensure_Bt());
        if (!use_tensor) { d_Brow.release(); if (!on_dev) Bsrc = nullptr; }     // the FMA path reads only the tiled copy
        return RMB200_OK;
    }
    // ILD: the unit-row image of B, once per call
    int unit_rows()
    {
        CK(d_unit.alloc((size_t)a.n * unit_pitch * sizeof(T)));
        pt.start();
        constexpr int WARPS = 8;
        rmb::unit_rows_kernel<T><<<(a.n + WARPS - 1) / WARPS, WARPS * 32, 0, st>>>(Bsrc, Bld, a.n, a.k, d_unit.as<T>(), unit_pitch);
        TRY(launched());
        pt.stop(tm.prep_ms);
        return RMB200_OK;
    }
    // Novelty / AvgPop: the caller's popularity counts on the device, checked against [0, U] there, and the per-item table
    int popularity_table()
    {
        if (!want_pop) return RMB200_OK;
        pop_d = reinterpret_cast<const long long*>(a.bey->item_popularity);
        if (!on_dev) {
            CK(d_pop.alloc((size_t)a.n * sizeof(long long)));
            pt.start();
            CK(cudaMemcpyAsync(d_pop.p, a.bey->item_popularity, (size_t)a.n * sizeof(long long), cudaMemcpyHostToDevice, st));
            tm.h2d_bytes += (int64_t)a.n * (int64_t)sizeof(long long);
            pt.stop(tm.h2d_ms);
            pop_d = d_pop.as<long long>();
        }
        CK(d_poptab.alloc((size_t)a.n * sizeof(double2)));
        CK(d_pop_bad.alloc(sizeof(int)));
        pt.start();
        CK(cudaMemsetAsync(d_pop_bad.p, 0, sizeof(int), st));
        rmb::popularity_table_kernel<<<(a.n + 255) / 256 < 4 * nsm ? (a.n + 255) / 256 : 4 * nsm, 256, 0, st>>>(
            pop_d, a.n, (long long)a.bey->popularity_users, d_poptab.as<double2>(), d_pop_bad.as<int>());
        TRY(launched());
        int bad = 0;
        CK(cudaMemcpyAsync(&bad, d_pop_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        pt.stop(tm.prep_ms);   // (synchronises)
        if (bad) { set_err("bad argument", "item_popularity: a count outside [0, popularity_users]"); return RMB200_ERR_BAD_ARG; }
        return RMB200_OK;
    }
    long long item_slice(int h) const { return (long long)a.n * h / (nested ? a.mc->G : 1); }
    // the host's item factors into d_Brow; one device of a multi-GPU call uploads its slice of the rows and fetches the other
    // slices from the peers' copies (see MultiCtx)
    int upload_item_rows()
    {
        const int g = a.mc_rank;
        const size_t row_bytes = (size_t)a.k * sizeof(T);
        unsigned char* base = static_cast<unsigned char*>(d_Brow.p);
        if (item_slice(g + 1) > item_slice(g))
            CK(upload_rows(base + (size_t)item_slice(g) * row_bytes, a.B + (size_t)item_slice(g) * a.ldb, a.ldb * sizeof(T), row_bytes,
                           (size_t)(item_slice(g + 1) - item_slice(g)), st));
        tm.h2d_bytes += (int64_t)(item_slice(g + 1) - item_slice(g)) * (int64_t)row_bytes;
        if (!nested) return RMB200_OK;
        MultiCtx& mc = *a.mc;
        CK(cudaStreamSynchronize(st));
        mc.Bptr[g] = d_Brow.p; mc.Bdev[g] = dev;
        if (!mc.meet(0)) { set_err("multi-GPU call", "another device failed"); return RMB200_ERR_CUDA; }
        for (int h = 1; h < mc.G; h++) {
            const int src = (g + h) % mc.G;
            const size_t off = (size_t)item_slice(src) * row_bytes, bytes = (size_t)(item_slice(src + 1) - item_slice(src)) * row_bytes;
            if (bytes) CK(cudaMemcpyPeerAsync(base + off, dev, static_cast<unsigned char*>(mc.Bptr[src]) + off, mc.Bdev[src], bytes, st));
        }
        CK(cudaStreamSynchronize(st));
        if (!mc.meet(1)) { set_err("multi-GPU call", "another device failed"); return RMB200_ERR_CUDA; }   // nobody frees its copy before everybody has fetched
        return RMB200_OK;
    }
    // operand image of the FMA path (the tensor path needs it only for a hand-back)
    int ensure_Bt()
    {
        if (have_Bt) return RMB200_OK;
        CK(d_Bt.alloc((size_t)p_pad * n_pad * sizeof(T)));
        pt.start();
        dim3 grid(n_pad / 32, (p_pad + 31) / 32), block(32, 8);
        rmb::pack_tiles_kernel<T, BN><<<grid, block, 0, st>>>(Bsrc, Bld, a.n, a.k, d_Bt.as<T>(), n_pad, p_pad);
        TRY(launched());
        pt.stop(tm.prep_ms);   // (synchronises)
        have_Bt = true;
        return RMB200_OK;
    }
    int item_bias()
    {
        if (!a.bias) return RMB200_OK;
        CK(d_bias.alloc((size_t)n_pad * sizeof(T)));
        DevBuf d_braw;
        const T* bsrc = a.bias;
        if (!on_dev) {
            CK(d_braw.alloc((size_t)a.n * sizeof(T)));
            pt.start();
            CK(cudaMemcpyAsync(d_braw.p, a.bias, (size_t)a.n * sizeof(T), cudaMemcpyHostToDevice, st));
            tm.h2d_bytes += (int64_t)a.n * (int64_t)sizeof(T);
            pt.stop(tm.h2d_ms);
            bsrc = d_braw.as<T>();
        }
        pt.start();
        rmb::pad_copy_kernel<T><<<(n_pad + 255) / 256, 256, 0, st>>>(bsrc, a.n, d_bias.as<T>(), n_pad);
        TRY(launched());
        pt.stop(tm.prep_ms);
        bias_d = d_bias.as<T>();
        return RMB200_OK;
    }
    // the tensor path's fp16 item image and the norms its error bound uses
    int item_image()
    {
        using namespace rmb;
        if (!use_tensor) return RMB200_OK;
        CK(d_Bb.alloc((size_t)n_pad128 * KB * sizeof(__half)));
        CK(d_maxbn.alloc(4 * sizeof(unsigned)));                    // [0] max_j ||b_j||, [1] largest observed error / bound ratio (statistic)
        CK(d_chunkn.alloc((size_t)(n_pad128 / 32) * sizeof(float)));
        pt.start();
        CK(cudaMemsetAsync(d_maxbn.p, 0, 4 * sizeof(unsigned), st));
        CK(cudaMemsetAsync(d_chunkn.p, 0, (size_t)(n_pad128 / 32) * sizeof(float), st));
        const long long total = (long long)n_pad128 * (KB / 8);
        row_norm_kernel<T><<<(a.n + NORM_ROWS_PER_BLOCK - 1) / NORM_ROWS_PER_BLOCK, 256, 0, st>>>(Bsrc, Bld, a.n, a.k, bias_d, 0, nullptr,
                                                                                              d_maxbn.as<unsigned>(), d_chunkn.as<float>());
        CK(cudaGetLastError());
        pack_f16_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(Bsrc, Bld, a.n, a.k, bias_d, 0, nullptr, d_maxbn.as<unsigned>(),
                                                                            d_Bb.as<__half>(), n_pad128, KB);
        TRY(launched(2));
        pt.stop(tm.prep_ms);
        return RMB200_OK;
    }
    int user_state()
    {
        using namespace rmb;
        CK(d_status.alloc((size_t)mr * sizeof(int)));
        CK(d_flags.alloc((size_t)mr * sizeof(int)));
        if (count_ranks) {
            CK(d_umin.alloc((size_t)mr * sizeof(unsigned long long)));
            CK(d_pos_raw.alloc(nnz_te * sizeof(T)));
            CK(d_pos_sorted.alloc(nnz_te * sizeof(T)));
            CK(d_pos_perm.alloc(nnz_te * sizeof(int)));
            CK(d_pos_item.alloc(nnz_te * sizeof(int)));
            CK(d_auc.alloc(nnz_te * sizeof(unsigned int)));
            CK(cudaMemsetAsync(d_auc.p, 0, nnz_te * sizeof(unsigned int) + (nnz_te ? 0 : 16), st));
            CK(cudaMemsetAsync(d_pos_sorted.p, 0, nnz_te * sizeof(T) + (nnz_te ? 0 : 16), st));
            CK(cudaMemsetAsync(d_pos_perm.p, 0, nnz_te * sizeof(int) + (nnz_te ? 0 : 16), st));
            CK(cudaMemsetAsync(d_pos_item.p, 0, nnz_te * sizeof(int) + (nnz_te ? 0 : 16), st));
        }
        if (ex->pos_rank) {
            if (on_dev) pos_rank_d = reinterpret_cast<long long*>(ex->pos_rank) + lo_hi[2];
            else { CK(d_pos_rank.alloc(nnz_te * sizeof(long long))); pos_rank_d = d_pos_rank.as<long long>(); }
            CK(cudaMemsetAsync(pos_rank_d, 0, nnz_te * sizeof(long long), st));
        }
        std::vector<double> l2((size_t)K);
        for (int i = 0; i < K; i++) l2[i] = std::log2((double)(i + 2));   // hpp:620 std::log2(ix+2)
        CK(d_log2.alloc((size_t)K * sizeof(double)));
        CK(cudaMemcpy(d_log2.p, l2.data(), (size_t)K * sizeof(double), cudaMemcpyHostToDevice));
        pt.start();
        StatusParams sp;
        sp.trp = trp_d; sp.tep = tep_d; sp.n = a.n; sp.K = K; sp.user_begin = 0; sp.user_end = mr;
        sp.has_ndcg = a.out[5] != nullptr;
        sp.has_rescue = (a.out[8] || a.out[9] || a.out[3] || a.out[4] || a.out[7]) ? 1 : 0;   // hpp:485
        sp.consider_cold_start = a.consider_cold_start; sp.min_items_pool = mip; sp.min_pos_test = mpt;
        sp.ustatus = d_status.as<int>(); sp.uflags = d_flags.as<int>();
        sp.umin = count_ranks ? d_umin.as<unsigned long long>() : nullptr;
        user_status_kernel<<<(mr + 255) / 256, 256, 0, st>>>(sp);
        TRY(launched());
        pt.stop(tm.prep_ms);
        return RMB200_OK;
    }
    // buffers of one batch (two sets of the staging buffers for host inputs and outputs); the first batch's users go up
    int batch_buffers()
    {
        if (use_full) CK(d_fo.alloc(fo_bytes));
        if (noise_handback) {
            CK(d_near.alloc(nnz_te * sizeof(unsigned)));
            CK(cudaMemsetAsync(d_near.p, 0, nnz_te * sizeof(unsigned) + (nnz_te ? 0 : 16), st));
            CK(d_nz_mark.alloc((size_t)UB * sizeof(int)));
            CK(d_nz_list.alloc((size_t)UB * sizeof(int)));
            CK(d_nz_cnt.alloc(16));
        }
        if (!on_dev) CK(rsx.init());
        CK(d_At.alloc((size_t)p_pad * UB * sizeof(T)));
        if (use_tensor) {
            CK(d_Ab.alloc((size_t)UB * KB * sizeof(__half)));
            CK(d_anorm.alloc((size_t)UB * sizeof(float)));
            CK(d_capx.alloc((size_t)UB * C * sizeof(uint2)));
            CK(d_overflow.alloc(OVERFLOW_INTS * sizeof(int)));
            CK(d_fb_list.alloc((size_t)UB * sizeof(int)));
        }
        if (!on_dev) {
            CK(d_Arow[0].alloc((size_t)UB * a.k * sizeof(T)));
            if (UB < mr) CK(d_Arow[1].alloc((size_t)UB * a.k * sizeof(T)));
            TRY(upload_users(0, 0));
        }
        CK(d_cs.alloc((size_t)UB * fma_slices * C * sizeof(T)));
        CK(d_ci.alloc((size_t)UB * fma_slices * C * sizeof(int)));
        CK(d_cc.alloc((size_t)UB * fma_slices * sizeof(int)));
        for (int set = 0; !on_dev && set < (UB < mr ? 2 : 1); set++)
            for (RowOut& r : row_outs)
                if (r.base) CK(r.staged[set].alloc((size_t)UB * r.row_bytes));
        int mean_blocks_total = 0;
        for (int b0 = 0; b0 < mr; b0 += UB) mean_blocks_total += (((mr - b0) < UB ? (mr - b0) : UB) + rmb::MEAN_CHUNK - 1) / rmb::MEAN_CHUNK;
        for (MeanTable& t : mean_tables) {
            if (!t.on()) continue;
            CK(t.part_sum.alloc((size_t)mean_blocks_total * t.slots * mean_W * sizeof(double)));
            CK(t.part_cnt.alloc((size_t)mean_blocks_total * t.slots * mean_W * sizeof(int)));
        }
        // item exposure: one uint32 count per item for the whole call (at most mr users each), [n] = users counted
        if (want_exposure) {
            CK(d_expo_hist.alloc(((size_t)a.n + 1) * sizeof(unsigned)));
            CK(cudaMemsetAsync(d_expo_hist.p, 0, ((size_t)a.n + 1) * sizeof(unsigned), st));
        }
        if (want_exposure || want_beyond) CK(d_list_len.alloc((size_t)UB * sizeof(int)));
        return RMB200_OK;
    }
    // upload of users [b0, b0 + UB) into staging buffer `slot`, on the prefetch stream
    int upload_users(int b0, int slot)
    {
        const int nb = (mr - b0) < UB ? (mr - b0) : UB;
        if (pf.freed_valid[slot]) CK(cudaStreamWaitEvent(pf.s, pf.freed[slot], 0));
        CK(upload_rows(d_Arow[slot].p, a.A + (size_t)(ub + b0) * a.lda, a.lda * sizeof(T), (size_t)a.k * sizeof(T), (size_t)nb, pf.s));
        tm.h2d_bytes += (int64_t)nb * a.k * (int64_t)sizeof(T);
        CK(cudaEventRecord(pf.ready[slot], pf.s));
        return RMB200_OK;
    }
    // the kernels reading the staged rows are queued: mark the buffer; once the scoring kernel is queued as well, the
    // next batch's rows go up into the other buffer (pageable sources keep this thread busy copying meanwhile)
    int staged_rows_consumed(const Batch& b)
    {
        if (!on_dev) { CK(cudaEventRecord(pf.freed[b.slot], st)); pf.freed_valid[b.slot] = true; }
        return RMB200_OK;
    }
    int prefetch_next_users(Batch& b)
    {
        if (on_dev || b.prefetched || b.b0 + UB >= mr) return RMB200_OK;
        b.prefetched = true;
        return upload_users(b.b0 + UB, b.slot ^ 1);
    }
    int launched(int n = 1) { CK(cudaGetLastError()); tm.kernel_launches += n; return RMB200_OK; }   // the kernels just queued
    int wait_test_rows() { if (pf.test_rows_pending) { CK(cudaStreamWaitEvent(st, pf.test_rows, 0)); pf.test_rows_pending = false; } return RMB200_OK; }
    int run_batch(int b0)
    {
        const int nb = (mr - b0) < UB ? (mr - b0) : UB;
        Batch b{b0, nb, round_up(nb, rmb::BM), (b0 / UB) & 1};
        TRY(stage_users(b));
        TRY(score(b));
        TRY(rank_fixups(b));
        pt.stop(tm.score_select_ms);                       // (the span score() opened)
        float ms = 0;                                      // (every path's dominant kernel is wrapped in pk)
        cudaEventElapsedTime(&ms, pk.a, pk.b);
        tm.dominant_kernel_ms += ms;
        TRY(metrics(b));
        return send_results(b);
    }
    // user factors of the batch -> k-major; with rank counting, the held-out items' scores, sorted per user
    int stage_users(Batch& b)
    {
        using namespace rmb;
        if (!on_dev) {
            pt.start();
            CK(cudaStreamWaitEvent(st, pf.ready[b.slot], 0));     // uploaded one batch ahead: only what is still exposed is timed
            b.Asrc = static_cast<const T*>(d_Arow[b.slot].p); b.Ald = (size_t)a.k;
            pt.stop(tm.h2d_ms);
        } else { b.Asrc = a.A + (size_t)(ub + b.b0) * a.lda; b.Ald = a.lda; }
        pt.start();
        dim3 grid(b.nb_pad / 32, (p_pad + 31) / 32), block(32, 8);
        pack_tiles_kernel<T, BM><<<grid, block, 0, st>>>(b.Asrc, b.Ald, b.nb, a.k, d_At.as<T>(), b.nb_pad, p_pad);
        TRY(launched());
        if (!use_tensor) TRY(staged_rows_consumed(b));
        if (count_ranks && !use_full) {
            TRY(wait_test_rows());
            const int blocks = (b.nb + 7) / 8 < 8 * nsm ? (b.nb + 7) / 8 : 8 * nsm;
            score_entries_kernel<T, BM><<<blocks, 256, 0, st>>>(d_At.as<T>(), d_Bt.as<T>(), bias_d, p_pad, b.b0, b.nb,
                                                             tep_d, tei_d, d_status.as<int>(), d_pos_raw.as<T>());
            CK(cudaGetLastError());
            sort_positives_kernel<T><<<blocks, 256, 0, st>>>(b.b0, b.nb, tep_d, tei_d, d_status.as<int>(), d_pos_raw.as<T>(),
                                                              d_pos_sorted.as<T>(), d_pos_perm.as<int>(), d_pos_item.as<int>());
            TRY(launched(2));
        }
        pt.stop(tm.prep_ms);
        return RMB200_OK;
    }
    // the batch's candidates on its path; opens the scoring span (run_batch closes it)
    int score(Batch& b)
    {
        if (fma_counts_first) {            // rank counts (and the smallest candidate score) from the FMA tiles; its top-K is replaced below
            pt.start();
            TRY(run_fma(b, d_At.as<T>(), b.nb, nullptr, count_ranks, true));
            TRY(prefetch_next_users(b));
            pt.stop(tm.score_select_ms);
        }
        if (use_tensor) return score_tensor(b);
        pt.start();
        if (!use_full) TRY(run_fma(b, d_At.as<T>(), b.nb, nullptr, count_ranks, true));
        else {    // every candidate scored, (noise,) sorted: ranked top-K, smallest candidate score and held-out ranks off the sorted lists
            TRY(wait_test_rows());
            TRY(run_full_order(b, d_At.as<T>(), b.nb, nullptr, fo_chunk, fo_bytes, true));
        }
        return prefetch_next_users(b);
    }
    // fused score / exclude / select (/ rank counting) on the FMA pipe: the whole batch, or (umap) the listed users only
    int run_fma(Batch& b, const T* At_ptr, int n_rows, const int* umap, bool with_counts, bool timed)
    {
        using namespace rmb;
        ScoreSelectParams<T> sp = ScoreSelectParams<T>();       // (every field defined: optional ones stay null)
        sp.At = At_ptr; sp.Bt = d_Bt.as<T>(); sp.bias = bias_d;
        sp.p_pad = p_pad; sp.n = a.n; sp.mb = n_rows; sp.user0 = b.b0;
        sp.trp = trp_d; sp.tri = tri_d; sp.tep = tep_d; sp.ustatus = d_status.as<int>();
        sp.cand_score = d_cs.as<T>(); sp.cand_item = d_ci.as<int>(); sp.cand_count = d_cc.as<int>();
        sp.uflags = d_flags.as<int>(); sp.K = K;
        sp.pos_sorted = with_counts ? d_pos_sorted.as<T>() : nullptr;
        sp.auc_cnt = with_counts ? d_auc.as<unsigned int>() : nullptr;
        sp.pos_item = with_counts ? d_pos_item.as<int>() : nullptr;
        sp.auc_near = (with_counts && noise_handback) ? d_near.as<unsigned>() : nullptr;
        sp.umin = with_counts ? d_umin.as<unsigned long long>() : nullptr;
        sp.umap = umap;
        const int slices = (umap == nullptr && !use_tensor) ? fma_slices : 1;
        sp.slice_rows = slices > 1 ? UB : 0;
        if (timed) cudaEventRecord(pk.a, st);
        CK(launch_score_select<T>(sp, C, with_counts, n_rows, slices, st));
        if (timed) cudaEventRecord(pk.b, st);
        tm.kernel_launches++;
        if (slices > 1) { merge_slices_kernel<T><<<(n_rows + 7) / 8, 256, 0, st>>>(d_cs.as<T>(), d_ci.as<int>(), d_cc.as<int>(), C, n_rows, slices, UB); TRY(launched()); }
        return RMB200_OK;
    }
    // the full-order path over n_users rows of At (umap: their batch-local users), with scratch of full_order_plan()
    int run_full_order(Batch& b, const T* At, int n_users, const int* umap, int chunk, size_t bytes, bool timed)
    {
        rmb::FullOrderArgs<T> fo;
        fo.At = At; fo.Bt = d_Bt.as<T>(); fo.bias = bias_d; fo.p_pad = p_pad; fo.n = a.n; fo.K = K; fo.C = C;
        fo.user0 = b.b0; fo.nb = n_users; fo.umap = umap;
        fo.trp = trp_d; fo.tri = tri_d; fo.tep = tep_d; fo.tei = tei_d; fo.ustatus = d_status.as<int>(); fo.uflags = d_flags.as<int>();
        fo.cand_score = d_cs.as<T>(); fo.cand_item = d_ci.as<int>(); fo.cand_count = d_cc.as<int>();
        fo.umin = count_ranks ? d_umin.as<unsigned long long>() : nullptr;
        fo.auc_cnt = count_ranks ? d_auc.as<unsigned int>() : nullptr;
        fo.pos_perm = count_ranks ? d_pos_perm.as<int>() : nullptr;
        fo.noise = a.noise; fo.seed_user0 = (unsigned long long)a.seed + (unsigned long long)(ub + b.b0);
        fo.scratch = d_fo.p; fo.scratch_bytes = bytes; fo.chunk_users = chunk;
        if (timed) cudaEventRecord(pk.a, st);
        long long nl = 0;
        CK(rmb::full_order_run<T>(fo, st, &nl));
        if (timed) cudaEventRecord(pk.b, st);
        tm.kernel_launches += nl;
        return RMB200_OK;
    }
    // Re-scores n listed users of the batch on their own: their staged rows gathered into `tile`, then the full-order path, or
    // (on_fma) the FMA tiles over the list.  With `flags`, the list and its length (*list_len) are collected from them first.
    int hand_back(Batch& b, DevBuf& tile, int* list, int n, const int* flags, int* list_len, bool on_fma)
    {
        using namespace rmb;
        TRY(ensure_Bt());
        const int n_pad_u = round_up(n, BM);
        CK(tile.alloc((size_t)p_pad * n_pad_u * sizeof(T)));
        if (flags) { collect_flagged_kernel<<<1, 1024, 0, st>>>(flags, b.nb, list, list_len); TRY(launched()); }
        dim3 grid(n_pad_u / 32, (p_pad + 31) / 32), block(32, 8);
        pack_tiles_gather_kernel<T, BM><<<grid, block, 0, st>>>(b.Asrc, b.Ald, list, n, a.k, tile.as<T>(), n_pad_u, p_pad);
        TRY(launched());
        TRY(staged_rows_consumed(b));      // (the gather read the staged rows once more)
        if (on_fma) return run_fma(b, tile.as<T>(), n, list, false, false);
        int chunk = 0; size_t bytes = 0;
        full_order_plan(a.n, (int)sizeof(T), n, &chunk, &bytes);
        CK(d_fo.alloc(bytes));
        if (count_ranks) TRY(wait_test_rows());
        return run_full_order(b, tile.as<T>(), n, list, chunk, bytes, false);
    }
    // norms + fp16 operand image of the batch's users, then the tensor-core filter and the exact re-scoring
    int score_tensor(Batch& b)
    {
        using namespace rmb;
        pt.start();
        const long long total = (long long)b.nb_pad * (KB / 8);
        row_norm_kernel<T><<<(b.nb + NORM_ROWS_PER_BLOCK - 1) / NORM_ROWS_PER_BLOCK, 256, 0, st>>>(b.Asrc, b.Ald, b.nb, a.k, (const T*)nullptr, a.bias ? 1 : 0,
                                                                                                 d_anorm.as<float>(), nullptr, nullptr);
        CK(cudaGetLastError());
        pack_f16_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(b.Asrc, b.Ald, b.nb, a.k, (const T*)nullptr, a.bias ? 1 : 0,
                                                                            d_anorm.as<float>(), nullptr, d_Ab.as<__half>(), b.nb_pad, KB);
        TRY(launched(2));
        CK(cudaMemsetAsync(d_overflow.p, 0, OVERFLOW_INTS * sizeof(int), st));
        pt.stop(tm.prep_ms);
        pt.start();
        const FilterErrCoef ec = filter_err_coefs(KB);
        FilterParams fp;
        fp.Ab = d_Ab.as<__half>(); fp.Bb = d_Bb.as<__half>(); fp.KB = KB; fp.stages = f_stages;
        fp.c_rel = ec.c_rel; fp.c_abs = ec.c_abs; fp.c_const = ec.c_const;
        fp.n = a.n; fp.mb = b.nb; fp.user0 = b.b0;
        fp.anorm = d_anorm.as<float>(); fp.maxbn = d_maxbn.as<unsigned>(); fp.chunk_norm = d_chunkn.as<float>();
        fp.trp = trp_d; fp.tri = tri_d; fp.ustatus = d_status.as<int>();
        fp.cand = d_capx.as<uint2>(); fp.cand_count = d_cc.as<int>();
        fp.overflow = d_overflow.as<int>(); fp.uflags = d_flags.as<int>(); fp.K = K;
        fp.sample_tiles = f_sample_tiles; fp.sample_stride = f_sample_stride; fp.sample_rank = f_sample_rank;
        fp.retries = d_overflow.as<int>() + 1;
        fp.noise_band = a.noise ? 2.02e-12f : 0.f;
        fp.score_max = sizeof(T) == 4 ? 0.5f * FLT_MAX : HUGE_VALF;
        cudaEventRecord(pk.a, st);
        CK(launch_filter_select(fp, C, b.nb_pad / BM, st));
        cudaEventRecord(pk.b, st);
        tm.kernel_launches++;
        // the exact stage reads the staged user factors (through d_At) and the filter is queued: the next batch's rows can go up
        TRY(staged_rows_consumed(b));
        TRY(prefetch_next_users(b));
        NoiseArgs nz;
        nz.on = a.noise; nz.seed_user0 = (unsigned long long)a.seed + (unsigned long long)(ub + b.b0); nz.trp = trp_d; nz.tri = tri_d; nz.n = a.n;
        FilterErrStat es;
        es.anorm = d_anorm.as<float>(); es.maxbn = d_maxbn.as<unsigned>(); es.chunk_norm = d_chunkn.as<float>();
        es.c_rel = ec.c_rel; es.c_abs = ec.c_abs; es.c_const = ec.c_const;
        es.max_ratio_bits = want_filter_stats ? d_maxbn.as<unsigned>() + 1 : nullptr;
        CK(launch_exact_topk<T>(d_capx.as<uint2>(), d_cs.as<T>(), d_ci.as<int>(), d_cc.as<int>(), C, b.nb, b.b0, d_At.as<T>(), p_pad, a.k,
                                Bsrc, Bld, bias_d, d_flags.as<int>(), K, nz, es, st));
        tm.kernel_launches++;
        int over_retry[OVERFLOW_INTS] = {0};
        CK(cudaMemcpyAsync(over_retry, d_overflow.p, OVERFLOW_INTS * sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const int n_over = over_retry[0];
        tm.filter_retry_rows += over_retry[1];
        if (n_over == 0) return RMB200_OK;
        // some users' kept band did not fit their candidate buffer (near-constant scores) or their factors cannot be scaled
        // into fp16 range: THOSE users are re-run on the FMA tiles (same results), everybody else keeps the filter's result
        tm.filter_fallback_batches++;
        tm.filter_fallback_users += n_over;
        pt.stop(tm.score_select_ms);
        TRY(ensure_Bt());
        pt.start();
        // a few users of a large catalogue go to the full-order path (every candidate scored by item-parallel blocks, one
        // segmented sort) -- on the FMA tiles ONE CTA walked the whole catalogue for them (78 ms at 1M items for a
        // single user, profiles/r02v: two of four ranks of a strong-scaling run ran at half speed for it).  Under the noise
        // every hand-back goes there: the FMA tiles neither add the noise nor check the noise branch's validity rule
        // (any infinite candidate => NaN row), which is what a user with a -inf score below its top K needs.
        const bool on_fma = !a.noise && (n_over > 2048 || a.n < 32768);
        return hand_back(b, d_At_fb, d_fb_list.as<int>(), n_over, d_cc.as<int>(), d_overflow.as<int>() + 6, on_fma);
    }
    // the selected candidates ranked; the noise hand-back; the all-equal check of the FMA tiles under the noise
    int rank_fixups(Batch& b)
    {
        using namespace rmb;
        if (!use_full) { CK(launch_rank_topk<T>(d_cs.as<T>(), d_ci.as<int>(), d_cc.as<int>(), C, b.nb, use_tensor ? K : K * fma_slices, st)); tm.kernel_launches++; }
        if (noise_handback) {
            // users for whom the tie-breaking noise decides a rank: their ranked top-K and ranks from the full-order path
            mark_noise_users_kernel<<<(b.nb + 255) / 256, 256, 0, st>>>(tep_d, d_near.as<unsigned>(), d_status.as<int>(), b.b0, b.nb, d_nz_mark.as<int>());
            CK(cudaGetLastError());
            CK(cudaMemsetAsync(d_nz_cnt.p, 0, 16, st));
            collect_flagged_kernel<<<1, 1024, 0, st>>>(d_nz_mark.as<int>(), b.nb, d_nz_list.as<int>(), d_nz_cnt.as<int>());
            TRY(launched(2));
            int n_nz = 0;
            CK(cudaMemcpyAsync(&n_nz, d_nz_cnt.p, sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (n_nz > 0) {
                tm.noise_handback_users += n_nz;
                TRY(hand_back(b, d_At_nz, d_nz_list.as<int>(), n_nz, nullptr, nullptr, false));
            }
        }
        if (a.noise && !use_tensor && !use_full && !count_ranks) {
            all_equal_check_kernel<T><<<b.nb, 128, 0, st>>>(d_cs.as<T>(), d_cc.as<int>(), C, b.b0, K, a.n, trp_d, tri_d, d_status.as<int>(),
                                                             d_At.as<T>(), d_Bt.as<T>(), bias_d, p_pad, d_flags.as<int>());
            TRY(launched());
        }
        return RMB200_OK;
    }
    // where batch b writes row output i: the caller's rows on device-resident calls, else the batch's result set
    template <typename U> U* rows_of(int i, const Batch& b) const
    {
        const RowOut& r = row_outs[i];
        if (!r.base) return nullptr;
        if (!on_dev) return static_cast<U*>(r.staged[b.slot].p);
        return reinterpret_cast<U*>(static_cast<unsigned char*>(r.base) + (size_t)(ub + b.b0) * r.row_bytes);
    }
    // per-user metrics (and the partial sums of their means) into the caller's rows, or into the batch's result set
    int metrics(Batch& b)
    {
        using namespace rmb;
        pt.start();
        MetricsParams<T> mp;
        mp.n = a.n; mp.K = K; mp.C = C; mp.user0 = b.b0; mp.mb = b.nb; mp.cumulative = a.cumulative;
        mp.want_roc = want_roc; mp.want_pr = want_pr; mp.count_ranks = count_ranks; mp.noise = a.noise;
        mp.trp = trp_d; mp.tep = tep_d; mp.tei = tei_d; mp.tev = tev_d;
        mp.ustatus = d_status.as<int>(); mp.uflags = d_flags.as<int>();
        mp.cand_score = d_cs.as<T>(); mp.cand_item = d_ci.as<int>(); mp.cand_count = d_cc.as<int>();
        mp.auc_cnt = d_auc.as<unsigned int>(); mp.umin = d_umin.as<unsigned long long>();
        mp.pos_perm = d_pos_perm.as<int>(); mp.log2tab = d_log2.as<double>();
        mp.nan_value = nan_value;
        if (!on_dev && rsx.copied_valid[b.slot]) CK(cudaStreamWaitEvent(st, rsx.copied[b.slot], 0));      // the set's previous rows have left
        mp.p = rows_of<T>(0, b); mp.tp = rows_of<T>(1, b); mp.r = rows_of<T>(2, b); mp.ap = rows_of<T>(3, b); mp.tap = rows_of<T>(4, b);
        mp.ndcg = rows_of<T>(5, b); mp.hit = rows_of<T>(6, b); mp.rr = rows_of<T>(7, b); mp.roc = rows_of<T>(8, b); mp.pr = rows_of<T>(9, b);
        mp.status_out = rows_of<int>(RO_STATUS, b);
        mp.topk_items = rows_of<int>(RO_TOPK_ITEMS, b);
        mp.topk_scores = rows_of<T>(RO_TOPK_SCORES, b);
        mp.pos_rank = pos_rank_d;
        mp.list_len = (want_exposure || want_beyond) ? d_list_len.as<int>() : nullptr;
        TRY(wait_test_rows());
        user_metrics_kernel<T><<<(b.nb + METRICS_WARPS - 1) / METRICS_WARPS, METRICS_WARPS * 32, 0, st>>>(mp);
        TRY(launched());
        if (want_exposure) {
            exposure_count_kernel<<<(b.nb + EXPOSURE_THREADS - 1) / EXPOSURE_THREADS, EXPOSURE_THREADS, 0, st>>>(
                d_ci.as<int>(), C, d_list_len.as<int>(), b.nb, d_expo_hist.as<unsigned>(), a.n);
            TRY(launched());
        }
        if (want_beyond) {
            BeyondParams<T> bp;
            bp.items = d_ci.as<int>(); bp.C = C; bp.list_len = d_list_len.as<int>(); bp.nb = b.nb; bp.K = K; bp.cumulative = a.cumulative;
            bp.pop = want_pop ? d_poptab.as<double2>() : nullptr;
            bp.unit = want_ild ? d_unit.as<T>() : nullptr; bp.pitch = unit_pitch;
            bp.nov = rows_of<T>(RO_BEYOND, b); bp.avgpop = rows_of<T>(RO_BEYOND + 1, b); bp.ild = rows_of<T>(RO_BEYOND + 2, b);
            bp.nan_value = nan_value;
            TRY(launch_beyond(bp));
        }
        const int mblocks = (b.nb + MEAN_CHUNK - 1) / MEAN_CHUNK;
        for (const MeanTable& t : mean_tables) {
            if (!t.on()) continue;
            MeanParams<T> qp;
            for (int q = 0; q < 10; q++) qp.out[q] = q < t.slots ? rows_of<T>(t.first_row + q, b) : nullptr;
            qp.nb = b.nb; qp.W = mean_W; qp.slots = t.slots; qp.wide = t.wide;
            qp.part_sum = t.part_sum.as<double>(); qp.part_cnt = t.part_cnt.as<int>(); qp.block0 = mean_block0;
            metric_partial_kernel<T><<<dim3(mblocks, t.slots), MEAN_CHUNK, 0, st>>>(qp);
            TRY(launched());
        }
        mean_block0 += mblocks;
        pt.stop(tm.metrics_ms);
        return RMB200_OK;
    }
    int launch_beyond(const rmb::BeyondParams<T>& bp)
    {
        using namespace rmb;
        const int blocks = (bp.nb + BEYOND_WARPS - 1) / BEYOND_WARPS, threads = BEYOND_WARPS * 32;
        if (unit_nch <= 1) beyond_accuracy_kernel<T, 1><<<blocks, threads, 0, st>>>(bp);      // (also: no ILD)
        else if (unit_nch == 2) beyond_accuracy_kernel<T, 2><<<blocks, threads, 0, st>>>(bp);
        else if (unit_nch == 4) beyond_accuracy_kernel<T, 4><<<blocks, threads, 0, st>>>(bp);
        else beyond_accuracy_kernel<T, 8><<<blocks, threads, 0, st>>>(bp);
        return launched();
    }
    // results of the batch -> caller's arrays at the shard's row offset (no gather collective: every shard writes its own
    // disjoint rows)
    int send_results(const Batch& b)
    {
        if (on_dev) return RMB200_OK;
        const size_t row = (size_t)(ub + b.b0), nb = (size_t)b.nb;
        CK(cudaEventRecord(rsx.ready[b.slot], st));
        CK(cudaStreamWaitEvent(rsx.s, rsx.ready[b.slot], 0));
        for (const RowOut& r : row_outs) {
            if (!r.base || (r.skippable && ex->skip_row_copy)) continue;
            const size_t bytes = nb * r.row_bytes;
            CK(cudaMemcpyAsync(static_cast<unsigned char*>(r.base) + row * r.row_bytes, r.staged[b.slot].p, bytes, cudaMemcpyDeviceToHost, rsx.s));
            tm.d2h_bytes += (int64_t)bytes;
        }
        CK(cudaEventRecord(rsx.copied[b.slot], rsx.s));
        rsx.copied_valid[b.slot] = true;
        return RMB200_OK;
    }
    // ---- after the last batch: what is still in flight, held-out ranks, metric means, the filter's error statistic ----
    int finish()
    {
        if (!on_dev) {                                        // what is still exposed of the result copies
            const auto t_d = std::chrono::steady_clock::now();
            CK(cudaStreamSynchronize(rsx.s));
            tm.d2h_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_d).count();
        }
        if (!on_dev && ex->pos_rank && !g_interrupt.load()) {
            pt.start();
            CK(cudaMemcpyAsync(ex->pos_rank + lo_hi[2], pos_rank_d, nnz_te * sizeof(long long), cudaMemcpyDeviceToHost, st));
            tm.d2h_bytes += (int64_t)(nnz_te * sizeof(long long));
            pt.stop(tm.d2h_ms);
        }
        for (MeanTable& t : mean_tables)
            if (t.on() && !g_interrupt.load()) TRY(means_out(t));
        if (want_exposure && !g_interrupt.load()) TRY(exposure_out());
        if (use_tensor && want_filter_stats) {
            float ratio = 0.f;
            CK(cudaMemcpyAsync(&ratio, d_maxbn.as<unsigned>() + 1, sizeof(float), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            tm.filter_err_ratio_max = (double)ratio;
        }
        CK(cudaStreamSynchronize(st));
        return RMB200_OK;
    }
    // a table's means / counts from its partial sums, into the caller's memory (device-resident calls) or copied out
    int means_out(MeanTable& t)
    {
        const size_t cells = (size_t)t.slots * mean_W;
        double* means_d = t.means; long long* counts_d = t.counts;
        if (!on_dev) {
            if (t.means) { CK(t.d_means.alloc(cells * sizeof(double))); means_d = t.d_means.as<double>(); }
            if (t.counts) { CK(t.d_counts.alloc(cells * sizeof(long long))); counts_d = t.d_counts.as<long long>(); }
        }
        pt.start();
        rmb::metric_final_kernel<<<(int)((cells + 127) / 128), 128, 0, st>>>(t.part_sum.as<double>(), t.part_cnt.as<int>(), mean_block0, t.slots, mean_W, means_d, counts_d);
        TRY(launched());
        pt.stop(tm.metrics_ms);
        if (!on_dev) {
            if (t.means) { CK(cudaMemcpyAsync(t.means, means_d, cells * sizeof(double), cudaMemcpyDeviceToHost, st)); tm.d2h_bytes += (int64_t)(cells * sizeof(double)); }
            if (t.counts) { CK(cudaMemcpyAsync(t.counts, counts_d, cells * sizeof(long long), cudaMemcpyDeviceToHost, st)); tm.d2h_bytes += (int64_t)(cells * sizeof(long long)); }
        }
        return RMB200_OK;
    }
    // the call's item counts, widened to int64, into the caller's array (device-resident calls: on the device, then a copy for
    // the statistics) or an internal one; the statistics from them on the host
    int exposure_out()
    {
        int64_t* dst_d = on_dev ? a.expo->item_counts : nullptr;
        if (!dst_d) { CK(d_expo_counts.alloc((size_t)a.n * sizeof(int64_t))); dst_d = d_expo_counts.as<int64_t>(); }
        pt.start();
        rmb::exposure_widen_kernel<<<(a.n + 255) / 256 < 4 * nsm ? (a.n + 255) / 256 : 4 * nsm, 256, 0, st>>>(
            d_expo_hist.as<unsigned>(), a.n, reinterpret_cast<long long*>(dst_d));
        TRY(launched());
        pt.stop(tm.metrics_ms);
        std::vector<int64_t> own;
        int64_t* dst_h = on_dev ? nullptr : a.expo->item_counts;
        if (!dst_h) { own.resize((size_t)a.n); dst_h = own.data(); }
        unsigned users = 0;
        pt.start();
        CK(cudaMemcpyAsync(dst_h, dst_d, (size_t)a.n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&users, d_expo_hist.as<unsigned>() + a.n, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        tm.d2h_bytes += (int64_t)a.n * (int64_t)sizeof(int64_t) + (int64_t)sizeof(unsigned);
        pt.stop(tm.d2h_ms);   // (synchronises)
        a.expo->users = (int64_t)users;
        return exposure_stats(dst_h, a.n, a.expo);
    }
};

// The device a call asks for: `device`, else env RMB200_DEVICE, else (-1) the calling thread's current device
int requested_device(int device)
{
    const char* env = std::getenv("RMB200_DEVICE");
    return device >= 0 ? device : (env ? std::atoi(env) : -1);
}

template <typename T>
int run_call(const CallArgs<T>& a)
{
    const auto t_begin = std::chrono::steady_clock::now();
    const rmb200_extra_t* ex = a.ex;
    // ---- argument checks (shape errors are the binding's job in the reference,
    //      recometrics/wrapper.pyx:261-268; here they become RMB200_ERR_BAD_ARG) ----
    if (a.m <= 0 || a.n <= 0 || a.k <= 0 || a.K <= 0) { set_err("bad argument", "m, n, k and k_metrics must be positive"); return RMB200_ERR_BAD_ARG; }
    if (!a.A || !a.B || !a.trp || !a.tep) { set_err("bad argument", "A, B, Xtrain_csr_p and Xtest_csr_p are required"); return RMB200_ERR_BAD_ARG; }
    if (a.lda < (size_t)a.k || a.ldb < (size_t)a.k) { set_err("bad argument", "lda/ldb smaller than k"); return RMB200_ERR_BAD_ARG; }
    if (a.out[5] && !a.tev) { set_err("bad argument", "NDCG requested but Xtest_csr (values) is NULL"); return RMB200_ERR_BAD_ARG; }
    if (ex->struct_size != (int32_t)sizeof(rmb200_extra_t)) { set_err("bad argument", "rmb200_extra_t::struct_size mismatch"); return RMB200_ERR_BAD_ARG; }
    if (a.bey && (a.bey->novelty || a.bey->avg_popularity)) {
        const int64_t U = a.bey->popularity_users;
        if (!a.bey->item_popularity) { set_err("bad argument", "Novelty / AvgPop requested but item_popularity is NULL"); return RMB200_ERR_BAD_ARG; }
        if (U < 1) { set_err("bad argument", "popularity_users must be >= 1"); return RMB200_ERR_BAD_ARG; }
        if (!ex->inputs_on_device)            // (device-resident counts are checked on the device, before the first batch)
            for (int j = 0; j < a.n; j++)
                if (a.bey->item_popularity[j] < 0 || a.bey->item_popularity[j] > U) { set_err("bad argument", "item_popularity: a count outside [0, popularity_users]"); return RMB200_ERR_BAD_ARG; }
    }
    bool any_out = ex->metric_means || ex->metric_counts || ex->topk_items || ex->topk_scores || ex->pos_rank || ex->status || a.expo;
    if (a.bey) any_out |= a.bey->novelty || a.bey->avg_popularity || a.bey->ild;
    for (int q = 0; q < 10; q++) any_out |= (a.out[q] != nullptr);
    if (!any_out) return RMB200_OK;
    int ub = 0, ue = 0;
    TRY(user_range(ex, a.m, &ub, &ue));
    if (ue == ub && !a.expo) return RMB200_OK;

    int dev = 0;
    TRY(rmb::use_device(requested_device(ex->device), &dev));
    if (ue == ub) return exposure_of_nobody(a.expo, a.n, ex->inputs_on_device != 0);

    const bool nested = a.mc != nullptr;                   // run_multi() holds the mutex and the latch
    std::unique_lock<std::mutex> lock(rmb::g_call_mutex, std::defer_lock);
    if (!nested) lock.lock();
    SignalLatch latch(!nested);
    Call<T> c(a, dev, ub, ue - ub);
    TRY(c.plan());
    TRY(c.csr_slices());
    TRY(c.item_factors());
    TRY(c.item_bias());
    TRY(c.popularity_table());
    TRY(c.item_image());
    TRY(c.user_state());
    TRY(c.batch_buffers());
    for (int b0 = 0; b0 < c.mr; b0 += c.UB) {
        if (g_interrupt.load()) break;                     // hpp:488-489
        TRY(c.run_batch(b0));
    }
    TRY(c.finish());
    c.tm.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    c.tm.devices_used = 1;
    if (ex->timing) *ex->timing = c.tm;

    if (g_interrupt.load()) {   // hpp:167-173: restore the handler, re-raise, report
        latch.restore();
        if (!nested) std::raise(SIGINT);
        set_err("interrupted", "procedure was interrupted");
        return RMB200_ERR_INTERRUPTED;
    }
    return RMB200_OK;
}

// Which GPUs the call runs on: rmb200_extra_t::devices, else (no explicit `device`) env RMB200_DEVICES = "all" | "0,1,2,...".
// An empty list = the single-device rules of run_call().
int resolve_devices(const rmb200_extra_t* ex, std::vector<int>& devs)
{
    devs.clear();
    if (ex && ex->struct_size != (int32_t)sizeof(rmb200_extra_t)) return RMB200_OK;      // (run_call reports it)
    if (ex && ex->n_devices > 0) {
        if (!ex->devices) { set_err("bad argument", "n_devices > 0 but devices is NULL"); return RMB200_ERR_BAD_ARG; }
        devs.assign(ex->devices, ex->devices + ex->n_devices);
    } else if (!(ex && ex->device >= 0) && !(ex && ex->inputs_on_device)) {
        const char* env = std::getenv("RMB200_DEVICES");
        if (!env || !env[0]) return RMB200_OK;
        if (!std::strcmp(env, "all")) {
            const int ndev = rmb200_device_count();
            for (int d = 0; d < ndev && d < rmb::MAX_DEVICES; d++) devs.push_back(d);
        } else {
            for (const char* c = env; *c;) {
                char* end = nullptr;
                const long v = std::strtol(c, &end, 10);
                if (end == c) { set_err("bad argument", "RMB200_DEVICES is neither \"all\" nor a comma-separated list of ordinals"); return RMB200_ERR_BAD_ARG; }
                devs.push_back((int)v);
                c = (*end == ',') ? end + 1 : end;
                if (*end && *end != ',') { set_err("bad argument", "RMB200_DEVICES is neither \"all\" nor a comma-separated list of ordinals"); return RMB200_ERR_BAD_ARG; }
            }
        }
    }
    if (devs.empty()) return RMB200_OK;
    if ((int)devs.size() > rmb::MAX_DEVICES) { set_err("bad argument", "more than 16 devices"); return RMB200_ERR_BAD_ARG; }
    int ndev = rmb200_device_count();
    if (ndev == 0) return rmb::use_device(-1, &ndev);      // (RMB200_ERR_NO_DEVICE, as for every call without a device)
    for (size_t i = 0; i < devs.size(); i++) {
        if (devs[i] < 0 || devs[i] >= ndev) { set_err("bad argument", "device ordinal out of range"); return RMB200_ERR_BAD_ARG; }
        for (size_t j = 0; j < i; j++)
            if (devs[j] == devs[i]) { set_err("bad argument", "a device is listed twice"); return RMB200_ERR_BAD_ARG; }
    }
    if (devs.size() > 1 && ex && ex->inputs_on_device) { set_err("unsupported", "a multi-GPU call takes host pointers (device-resident inputs live on one GPU)"); return RMB200_ERR_UNSUPPORTED; }
    return RMB200_OK;
}

// One means / counts table of a multi-GPU call (the caller's; both null: not requested): every device reduces its users into
// a table of its own, the call's means are the devices' means weighted by their user counts
struct DeviceMeans {
    double* means; int64_t* counts; size_t cells;
    std::vector<std::vector<double>> dev_means;
    std::vector<std::vector<long long>> dev_counts;
    DeviceMeans(double* m, int64_t* c, size_t n, int G) : means(m), counts(c), cells(n),
        dev_means(m || c ? G : 0, std::vector<double>(n, 0.0)), dev_counts(m || c ? G : 0, std::vector<long long>(n, 0)) {}
    void attach(int g, double*& m, int64_t*& c)          // device g's call reduces into its own table
    {
        if (dev_means.empty()) return;
        m = dev_means[g].data(); c = reinterpret_cast<int64_t*>(dev_counts[g].data());
    }
    void merge() const
    {
        for (size_t i = 0; !dev_means.empty() && i < cells; i++) {
            double s = 0.0; long long cnt = 0;
            for (size_t g = 0; g < dev_means.size(); g++)
                if (dev_counts[g][i] > 0) { s += dev_means[g][i] * (double)dev_counts[g][i]; cnt += dev_counts[g][i]; }
            if (means) means[i] = cnt ? s / (double)cnt : std::numeric_limits<double>::quiet_NaN();
            if (counts) counts[i] = cnt;
        }
    }
};

// /root/reference/src/recometrics.hpp:428-437: the reference's one call spreads the users over every core
// (`#pragma omp parallel for schedule(dynamic) num_threads(nthreads)`); this spreads them over every listed GPU.
template <typename T>
int run_multi(const CallArgs<T>& a0, const std::vector<int>& devs_in)
{
    const auto t_begin = std::chrono::steady_clock::now();
    const rmb200_extra_t* ex = ex_or_default(a0.ex);
    if (a0.m <= 0) { set_err("bad argument", "m, n, k and k_metrics must be positive"); return RMB200_ERR_BAD_ARG; }
    int ub = 0, ue = 0;
    TRY(user_range(ex, a0.m, &ub, &ue));
    // contiguous blocks in units of one CTA's 128 users; devices left without a unit sit the call out
    const int units = (ue - ub + rmb::BM - 1) / rmb::BM;
    std::vector<int> devs, lo, hi;
    {
        const int G0 = (int)devs_in.size();
        for (int g = 0; g < G0; g++) {
            const int u0 = (int)((long long)units * g / G0), u1 = (int)((long long)units * (g + 1) / G0);
            if (u1 <= u0) continue;
            devs.push_back(devs_in[g]);
            lo.push_back(ub + u0 * rmb::BM);
            hi.push_back(std::min(ue, ub + u1 * rmb::BM));
        }
    }
    const int G = (int)devs.size();
    if (G == 0) return a0.expo ? exposure_of_nobody(a0.expo, a0.n, false) : RMB200_OK;

    std::unique_lock<std::mutex> lock(rmb::g_call_mutex);
    SignalLatch latch;
    MultiCtx mc;
    mc.G = G;
    const size_t W = (size_t)(a0.cumulative && a0.K > 0 ? a0.K : 1);
    DeviceMeans metric_means(ex->metric_means, ex->metric_counts, 10 * W, G);
    DeviceMeans beyond_means(a0.bey ? a0.bey->means : nullptr, a0.bey ? a0.bey->counts : nullptr, 3 * W, G);
    std::vector<rmb200_extra_t> exs((size_t)G, *ex);
    std::vector<rmb200_timing_t> tms((size_t)G);
    std::vector<rmb200_exposure_t> expos((size_t)G);
    std::vector<std::vector<int64_t>> item_counts(a0.expo ? (size_t)G : 0);
    std::vector<rmb200_beyond_t> beys((size_t)G);
    std::vector<int> rcs((size_t)G, RMB200_OK);
    std::vector<std::string> errs((size_t)G);
    std::vector<std::thread> workers;
    for (int g = 0; g < G; g++) {
        std::memset(&tms[g], 0, sizeof(rmb200_timing_t));
        rmb200_extra_t& e = exs[g];
        e.device = devs[g]; e.devices = nullptr; e.n_devices = 0;
        e.user_begin = lo[g]; e.user_end = hi[g];
        e.timing = &tms[g];
        metric_means.attach(g, e.metric_means, e.metric_counts);
        if (a0.expo) {
            item_counts[g].assign((size_t)a0.n, 0);
            std::memset(&expos[g], 0, sizeof(rmb200_exposure_t));
            expos[g].struct_size = (int32_t)sizeof(rmb200_exposure_t);
            expos[g].item_counts = item_counts[g].data();
        }
        if (a0.bey) {           // rows straight into the caller's arrays (every device writes its own); means per device
            beys[g] = *a0.bey;
            beyond_means.attach(g, beys[g].means, beys[g].counts);
        }
        workers.emplace_back([&, g]() {
            rmb::g_err.clear();
            rmb::g_upload_share = G;
            const int rc = rmb::guard([&] {
                // peers' memory directly over NVLink where the hardware allows it (else the copies are staged by the driver)
                if (cudaSetDevice(devs[g]) == cudaSuccess)
                    for (int h = 0; h < G; h++) {
                        int can = 0;
                        if (h != g && cudaDeviceCanAccessPeer(&can, devs[g], devs[h]) == cudaSuccess && can) cudaDeviceEnablePeerAccess(devs[h], 0);
                        cudaGetLastError();
                    }
                CallArgs<T> a = a0;
                a.ex = &exs[g]; a.mc = &mc; a.mc_rank = g;
                if (a0.expo) a.expo = &expos[g];
                if (a0.bey) a.bey = &beys[g];
                return run_call<T>(a);
            });
            rcs[g] = rc; errs[g] = rmb::g_err;
            mc.depart(rc != RMB200_OK);
        });
    }
    for (auto& w : workers) w.join();

    int rc = RMB200_OK;
    for (int g = 0; g < G && rc == RMB200_OK; g++)
        if (rcs[g] != RMB200_OK && rcs[g] != RMB200_ERR_INTERRUPTED) { rc = rcs[g]; rmb::g_err = errs[g]; }
    if (rc == RMB200_OK && g_interrupt.load()) {
        latch.restore();
        std::raise(SIGINT);
        set_err("interrupted", "procedure was interrupted");
        return RMB200_ERR_INTERRUPTED;
    }
    if (rc != RMB200_OK) return rc;

    metric_means.merge();
    beyond_means.merge();
    if (a0.expo) {          // the devices' counts added up (integers: exact), the statistics of the sum
        std::vector<int64_t> own;
        int64_t* sum = a0.expo->item_counts;
        if (!sum) { own.resize((size_t)a0.n); sum = own.data(); }
        int64_t users = 0;
        for (int j = 0; j < a0.n; j++) {
            int64_t c = 0;
            for (int g = 0; g < G; g++) c += item_counts[g][j];
            sum[j] = c;
        }
        for (int g = 0; g < G; g++) users += expos[g].users;
        a0.expo->users = users;
        TRY(exposure_stats(sum, a0.n, a0.expo));
    }
    if (ex->timing) {
        rmb200_timing_t t = tms[0];
        for (int g = 1; g < G; g++) {
            const rmb200_timing_t& o = tms[g];
            t.h2d_ms = std::max(t.h2d_ms, o.h2d_ms); t.prep_ms = std::max(t.prep_ms, o.prep_ms);
            t.score_select_ms = std::max(t.score_select_ms, o.score_select_ms); t.metrics_ms = std::max(t.metrics_ms, o.metrics_ms);
            t.d2h_ms = std::max(t.d2h_ms, o.d2h_ms); t.dominant_kernel_ms = std::max(t.dominant_kernel_ms, o.dominant_kernel_ms);
            t.kernel_launches += o.kernel_launches; t.h2d_bytes += o.h2d_bytes; t.d2h_bytes += o.d2h_bytes;
            t.filter_fallback_batches += o.filter_fallback_batches; t.filter_retry_rows += o.filter_retry_rows;
            t.filter_fallback_users += o.filter_fallback_users; t.noise_handback_users += o.noise_handback_users;
            t.filter_err_ratio_max = std::max(t.filter_err_ratio_max, o.filter_err_ratio_max);
        }
        t.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        t.devices_used = G;
        *ex->timing = t;
    }
    return RMB200_OK;
}

template <typename T>
int entry(const T* A, size_t lda, const T* B, size_t ldb, int32_t m, int32_t n, int32_t k,
          const int32_t* trp, const int32_t* tri, const int32_t* tep, const int32_t* tei, const T* tev,
          int32_t K, int cumulative, int noise,
          T* p, T* tp, T* r, T* ap, T* tap, T* ndcg, T* hit, T* rr, T* roc, T* pr,
          int ccs, int32_t mip, int32_t mpt, uint64_t seed, const T* bias, const rmb200_extra_t* ex, rmb200_exposure_t* expo = nullptr,
          rmb200_beyond_t* bey = nullptr)
{
    rmb::g_err.clear();
    if (expo && expo->struct_size != (int32_t)sizeof(rmb200_exposure_t)) { set_err("bad argument", "rmb200_exposure_t::struct_size mismatch"); return RMB200_ERR_BAD_ARG; }
    if (bey && bey->struct_size != (int32_t)sizeof(rmb200_beyond_t)) { set_err("bad argument", "rmb200_beyond_t::struct_size mismatch"); return RMB200_ERR_BAD_ARG; }
    CallArgs<T> a;
    a.A = A; a.lda = lda; a.B = B; a.ldb = ldb; a.m = m; a.n = n; a.k = k;
    a.trp = trp; a.tri = tri; a.tep = tep; a.tei = tei; a.tev = tev;
    a.K = K; a.cumulative = cumulative ? 1 : 0; a.noise = noise ? 1 : 0;
    T* outs[10] = {p, tp, r, ap, tap, ndcg, hit, rr, roc, pr};
    for (int q = 0; q < 10; q++) a.out[q] = outs[q];
    a.consider_cold_start = ccs ? 1 : 0; a.min_items_pool = mip; a.min_pos_test = mpt; a.seed = seed;
    a.bias = bias; a.ex = ex_or_default(ex); a.expo = expo; a.bey = bey;
    return rmb::guard([&] {
        std::vector<int> devs;
        TRY(resolve_devices(a.ex, devs));
        if (devs.size() > 1) return run_multi<T>(a, devs);
        if (devs.size() == 1) {                 // a list of one: that device
            rmb200_extra_t one = *a.ex;
            one.device = devs[0]; one.devices = nullptr; one.n_devices = 0;
            a.ex = &one;
            return run_call<T>(a);
        }
        return run_call<T>(a);
    });
}

// rmb200_item_popularity: the column count of CSR rows [rb, re) on the device, widened to int64 into `counts`
int item_popularity(const int32_t* indptr, const int32_t* indices, int rb, int re, int n, int device, bool on_dev, int64_t* counts)
{
    if (n <= 0 || !indptr || !counts || rb < 0 || re < rb) { set_err("bad argument", "item_popularity: n <= 0, a NULL array or a bad row range"); return RMB200_ERR_BAD_ARG; }
    int dev = 0;
    TRY(rmb::use_device(requested_device(device), &dev));
    std::lock_guard<std::mutex> lock(rmb::g_call_mutex);       // (the upload lanes belong to the holder)
    cudaStream_t st = nullptr;                             // legacy default stream, as the evaluation call
    int lo = 0, hi = 0;
    if (on_dev) {
        CK(cudaMemcpy(&lo, indptr + rb, sizeof(int), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(&hi, indptr + re, sizeof(int), cudaMemcpyDeviceToHost));
    } else { lo = indptr[rb]; hi = indptr[re]; }
    if (hi < lo) { set_err("bad argument", "CSR index pointers decrease"); return RMB200_ERR_BAD_ARG; }
    const long long nnz = (long long)hi - lo;
    if (nnz && !indices) { set_err("bad argument", "CSR indices missing"); return RMB200_ERR_BAD_ARG; }
    DevBuf d_idx, d_hist, d_counts;
    const int* idx_d = on_dev ? indices + lo : nullptr;
    if (!on_dev) {
        CK(d_idx.alloc((size_t)nnz * sizeof(int)));
        if (nnz) CK(upload_rows(d_idx.p, indices + lo, (size_t)nnz * sizeof(int), (size_t)nnz * sizeof(int), 1, st));
        idx_d = d_idx.as<int>();
    }
    CK(d_hist.alloc((size_t)n * sizeof(unsigned)));
    CK(cudaMemsetAsync(d_hist.p, 0, (size_t)n * sizeof(unsigned), st));
    int nsm = 148;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (nnz) {
        const long long want = (nnz + rmb::POPULARITY_THREADS - 1) / rmb::POPULARITY_THREADS;
        rmb::item_popularity_kernel<<<(int)(want < 8ll * nsm ? want : 8ll * nsm), rmb::POPULARITY_THREADS, 0, st>>>(idx_d, nnz, d_hist.as<unsigned>(), n);
        CK(cudaGetLastError());
    }
    long long* dst = on_dev ? reinterpret_cast<long long*>(counts) : nullptr;
    if (!dst) { CK(d_counts.alloc((size_t)n * sizeof(long long))); dst = d_counts.as<long long>(); }
    rmb::exposure_widen_kernel<<<(n + 255) / 256 < 4 * nsm ? (n + 255) / 256 : 4 * nsm, 256, 0, st>>>(d_hist.as<unsigned>(), n, dst);
    CK(cudaGetLastError());
    if (!on_dev) CK(cudaMemcpyAsync(counts, dst, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return RMB200_OK;
}

}  // namespace

extern "C" {

int rmb200_calc_metrics_f32(
    const float* A, size_t lda, const float* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const float* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float* p_at_k, float* tp_at_k, float* r_at_k, float* ap_at_k, float* tap_at_k,
    float* ndcg_at_k, float* hit_at_k, float* rr_at_k, float* roc_auc, float* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed)
{
    (void)nthreads;
    return entry<float>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                        k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                        ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                        min_pos_test, seed, nullptr, nullptr);
}

int rmb200_calc_metrics_f64(
    const double* A, size_t lda, const double* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const double* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double* p_at_k, double* tp_at_k, double* r_at_k, double* ap_at_k, double* tap_at_k,
    double* ndcg_at_k, double* hit_at_k, double* rr_at_k, double* roc_auc, double* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed)
{
    (void)nthreads;
    return entry<double>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                         k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                         ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                         min_pos_test, seed, nullptr, nullptr);
}

int rmb200_calc_metrics_ex_f32(
    const float* A, size_t lda, const float* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const float* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float* p_at_k, float* tp_at_k, float* r_at_k, float* ap_at_k, float* tap_at_k,
    float* ndcg_at_k, float* hit_at_k, float* rr_at_k, float* roc_auc, float* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed,
    const float* item_biases, const rmb200_extra_t* extra)
{
    (void)nthreads;
    return entry<float>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                        k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                        ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                        min_pos_test, seed, item_biases, extra);
}

int rmb200_calc_metrics_ex_f64(
    const double* A, size_t lda, const double* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const double* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double* p_at_k, double* tp_at_k, double* r_at_k, double* ap_at_k, double* tap_at_k,
    double* ndcg_at_k, double* hit_at_k, double* rr_at_k, double* roc_auc, double* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed,
    const double* item_biases, const rmb200_extra_t* extra)
{
    (void)nthreads;
    return entry<double>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                         k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                         ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                         min_pos_test, seed, item_biases, extra);
}

int rmb200_calc_metrics_exposure_f32(
    const float* A, size_t lda, const float* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const float* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float* p_at_k, float* tp_at_k, float* r_at_k, float* ap_at_k, float* tap_at_k,
    float* ndcg_at_k, float* hit_at_k, float* rr_at_k, float* roc_auc, float* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed,
    const float* item_biases, const rmb200_extra_t* extra, rmb200_exposure_t* exposure)
{
    (void)nthreads;
    return entry<float>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                        k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                        ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                        min_pos_test, seed, item_biases, extra, exposure);
}

int rmb200_calc_metrics_exposure_f64(
    const double* A, size_t lda, const double* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const double* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double* p_at_k, double* tp_at_k, double* r_at_k, double* ap_at_k, double* tap_at_k,
    double* ndcg_at_k, double* hit_at_k, double* rr_at_k, double* roc_auc, double* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed,
    const double* item_biases, const rmb200_extra_t* extra, rmb200_exposure_t* exposure)
{
    (void)nthreads;
    return entry<double>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                         k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                         ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                         min_pos_test, seed, item_biases, extra, exposure);
}

int rmb200_exposure_stats(const int64_t* counts, int32_t n, rmb200_exposure_t* out)
{
    rmb::g_err.clear();
    if (!out || out->struct_size != (int32_t)sizeof(rmb200_exposure_t)) { set_err("bad argument", "rmb200_exposure_t::struct_size mismatch"); return RMB200_ERR_BAD_ARG; }
    return exposure_stats(counts, n, out);
}

int rmb200_sizeof_exposure(void) { return (int)sizeof(rmb200_exposure_t); }

int rmb200_calc_metrics_beyond_f32(
    const float* A, size_t lda, const float* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const float* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    float* p_at_k, float* tp_at_k, float* r_at_k, float* ap_at_k, float* tap_at_k,
    float* ndcg_at_k, float* hit_at_k, float* rr_at_k, float* roc_auc, float* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed,
    const float* item_biases, const rmb200_extra_t* extra, rmb200_exposure_t* exposure, rmb200_beyond_t* beyond)
{
    (void)nthreads;
    return entry<float>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                        k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                        ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                        min_pos_test, seed, item_biases, extra, exposure, beyond);
}

int rmb200_calc_metrics_beyond_f64(
    const double* A, size_t lda, const double* B, size_t ldb, int32_t m, int32_t n, int32_t k,
    const int32_t* Xtrain_csr_p, const int32_t* Xtrain_csr_i,
    const int32_t* Xtest_csr_p, const int32_t* Xtest_csr_i, const double* Xtest_csr,
    int32_t k_metrics, int cumulative, int break_ties_with_noise,
    double* p_at_k, double* tp_at_k, double* r_at_k, double* ap_at_k, double* tap_at_k,
    double* ndcg_at_k, double* hit_at_k, double* rr_at_k, double* roc_auc, double* pr_auc,
    int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, int32_t nthreads, uint64_t seed,
    const double* item_biases, const rmb200_extra_t* extra, rmb200_exposure_t* exposure, rmb200_beyond_t* beyond)
{
    (void)nthreads;
    return entry<double>(A, lda, B, ldb, m, n, k, Xtrain_csr_p, Xtrain_csr_i, Xtest_csr_p, Xtest_csr_i, Xtest_csr,
                         k_metrics, cumulative, break_ties_with_noise, p_at_k, tp_at_k, r_at_k, ap_at_k, tap_at_k,
                         ndcg_at_k, hit_at_k, rr_at_k, roc_auc, pr_auc, consider_cold_start, min_items_pool,
                         min_pos_test, seed, item_biases, extra, exposure, beyond);
}

int rmb200_sizeof_beyond(void) { return (int)sizeof(rmb200_beyond_t); }

int rmb200_item_popularity(const int32_t* indptr, const int32_t* indices, int32_t row_begin, int32_t row_end, int32_t n,
                           int32_t device, int32_t inputs_on_device, int64_t* counts)
{
    rmb::g_err.clear();
    return rmb::guard([&] { return item_popularity(indptr, indices, row_begin, row_end, n, device, inputs_on_device != 0, counts); });
}

int rmb200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int rmb200_version(void) { return RMB200_VERSION; }

int rmb200_sizeof_extra(void) { return (int)sizeof(rmb200_extra_t); }

int rmb200_sizeof_timing(void) { return (int)sizeof(rmb200_timing_t); }

void rmb200_request_interrupt(void) { g_interrupt.store(1); }

double rmb200_measure_fma_peak(int device, int dtype_bytes, double* elapsed_ms)
{
    rmb::g_err.clear();
    if (rmb::use_device(device, &device) != RMB200_OK) return -1.0;
    int nsm = 148;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device);
    const int threads = 256, blocks = nsm * 8;
    const int iters = dtype_bytes == 4 ? 40000 : 20000;
    DevBuf out;
    if (out.alloc((size_t)blocks * threads * 8) != cudaSuccess) { set_err("alloc"); return -1.0; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 3; rep++) {
        cudaEventRecord(e0);
        if (dtype_bytes == 4) rmb::fma2_peak_kernel<<<blocks, threads>>>(out.as<float>(), iters, 1.0f);   // 4 x 16 FFMA2 = 8 x 16 FMA per iteration
        else rmb::fma_peak_kernel<double><<<blocks, threads>>>(out.as<double>(), iters, 1.0);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { set_err("fma peak kernel failed"); cudaGetLastError(); return -1.0; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (elapsed_ms) *elapsed_ms = best;
    const double flops = (double)blocks * threads * (double)iters * 8.0 * 16.0 * 2.0;
    return flops / (best * 1e-3) / 1e12;
}

}  // extern "C"
