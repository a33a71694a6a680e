// filter_select.cuh -- tensor-core (tcgen05) candidate filter + exact re-scoring: the top-K path
// when no rank counting (ROC/PR-AUC) is requested.
//
// Same job as score_select.cuh (reference: candidate list /root/reference/src/recometrics.hpp:491-497,
// dot1 scoring :84-112/:499-512, partial_sort :537-548) with the work split differently:
//
//   1. FILTER (filter_select_kernel) -- every (user, item) score is computed APPROXIMATELY on the
//      5th-generation tensor cores: fp16 copies of the factors, scaled by powers of two so that every element
//      is at most 1 (prep.cuh; item bias folded in as one more factor, as the reference's front-end does,
//      recometrics/__init__.py:548-551), fp32 accumulation in TMEM.
//      A CTA keeps a 128-user A tile resident in shared memory and streams 128-item B tiles through a
//      TMA ring; one elected lane issues tcgen05.mma (M=128, N=128, K=16 per instruction) into one of
//      four TMEM accumulator buffers; sixteen epilogue warps read them back with tcgen05.ld: the four
//      warps of a TMEM lane quarter (32 user rows; they also share a warp scheduler) each take one
//      32-column chunk of every tile.  Everything a warp needs per row is PRIVATE to it -- its own region
//      of the row's candidate buffer with the counter in a register, its own cursor into the row's train
//      items -- so the four warps never wait for each other inside a tile: while one of them appends
//      candidates, the others run ahead (up to the four accumulator buffers).  They meet at a named
//      barrier only every 1..64 tiles (the distance adapts to the append rate) to cut the row's four
//      regions back together and raise the row's shared threshold.
//
//      INTERVALS.  Every approximate score carries its own error bound
//          e_uj = c_rel ||a_u|| ||b_j|| + c_abs ||a_u|| + c_const        (scaled units, filter_err_coefs)
//      with ||b_j|| replaced by the largest item norm of j's 32-item chunk (prep.cuh row_norm_kernel), so
//      exact_uj lies in [lb, ub] = [approx - e, approx + e].  With tau' = the K-th best LOWER bound seen so far
//      the exact K-th best score is >= tau', and an item can only belong to the exact top K if its UPPER
//      bound reaches tau'.  The kernel keeps, per user, exactly the candidates with ub >= tau': one item with a
//      huge norm widens only its own interval, never the band of the whole row (a single global max_j ||b_j||
//      did).  Train items and padding columns are dropped when appended; >= 99.9 % of the catalogue is
//      rejected with one compare per 32 scores.
//   2. EXACT (exact_topk_kernel) -- one warp per user re-scores the few hundred survivors exactly
//      (sequential fma chain over the original fp32 / fp64 factors: the same chain, hence bit-identical
//      scores, as score_select_kernel / score_entries_kernel) and keeps the best K.  The final top-K,
//      their order and their scores are exactly those of the FP32 (FP64) FMA path; the tensor cores only
//      decide what is worth looking at.  A user whose kept band does not fit the buffer (near-constant scores),
//      or whose factors cannot be scaled into fp16 range, is flagged and the host re-runs THAT USER on the FMA
//      path (api.cu).  A user whose factors are all zero (every score equal: NaN row, hpp:541-548) is settled
//      without scoring.
//
// Shared-memory operand layout (no swizzle, K-major "interleaved"): [k/8][row][8 halves] -- a core matrix
// is 8 rows x 16 bytes contiguous; descriptor LBO = 128 rows * 16 B (next k chunk), SBO = 128 B (next 8
// rows).  The pack kernel writes tiles in exactly this image, so one bulk copy per tile lands it.
// Encodings pinned on hardware by tools/ubench/umma_probe.cu.
#pragma once
#include <cuda_fp16.h>
#include "prep.cuh"
#include "score_select.cuh"
#include "tie_noise.cuh"

namespace rmb {

constexpr int FN = 128;                  // items per MMA tile = TMEM columns per accumulator buffer
constexpr int F_EPI_WARPS = 16;          // warp w reads TMEM lanes (user rows) 32*(w%4)..+31, column chunk w/4 of every tile
constexpr int F_MMA_WARPS = 2;           // MMA-issuing warps, taking turns tile by tile: one warp's per-tile barrier waits and commits
                                         // (~300 cycles in which it issues nothing) overlap with the other warp's MMAs
constexpr int F_THREADS = (F_EPI_WARPS + 1 + F_MMA_WARPS) * 32;   // + TMA producer warp + MMA warps
constexpr int F_ACCBUFS = 4;             // TMEM accumulator buffers: slack between the MMA warp and the slowest epilogue warp
constexpr int F_ACCSHIFT = 2;            // log2(F_ACCBUFS): a buffer's phase parity flips every F_ACCBUFS iterations
constexpr int F_TMEM_COLS = F_ACCBUFS * FN;
constexpr int F_MAX_STAGES = 6;              // ring depth: as many B tiles as fit next to the A tile (5 at 128 factors)
constexpr int F_CHUNK = 32;              // TMEM columns per tcgen05.ld
constexpr int F_CUT_MARGIN = 48;         // a row's regions are cut back together once they hold this many more than the last cut kept
constexpr int F_MAIN_MARGIN = 250;       // ... in the pass that starts from the sampled guess: its thresholds are tight from the first tile on, a cut
                                         // (which stalls its warp and soon the CTA's pipeline) buys little there (A/B on B200: 52 -> 47.4 ms per batch)
constexpr int F_MAX_MEET = 64;           // most item tiles between two meetings of a quarter's warps
constexpr int F_CUT_BITS = 10;           // bisection steps of the cuts at the meetings (the cut at the end of a pass is exact: 32)

struct FilterParams {
    const __half* __restrict__ Ab;          // [user tiles][KB/8][128][8]  fp16 user factors (+1.0 bias column), each row scaled by pow2_scale_for(||a_u||)
    const __half* __restrict__ Bb;          // [item tiles][KB/8][128][8]  fp16 item factors (+bias column), all scaled by pow2_scale_for(max_j ||b_j||)
    int KB;                                 // fp16 factors per row, multiple of 16
    float c_rel, c_abs, c_const;            // error bound of an approximate score (host: filter_err_coefs)
    float noise_band;                       // break_ties_with_noise: how far the noise can move two scores apart (2e-12), else 0
    float score_max;                        // largest ||a|| * max ||b|| whose scores cannot overflow the input type (float:
                                            // FLT_MAX / 2; double: +inf, as both norms are below 6e29 here)
    int stages;                             // depth of the B ring
    int n, mb, user0;
    const float* __restrict__ anorm;        // [mb] ||a_u|| (with the 1.0 bias component), rounded up; 0 = all-zero row
    const unsigned* __restrict__ maxbn;     // float bits of max_j ||b_j|| (with the bias component)
    const float* __restrict__ chunk_norm;   // [ceil(n/128)*4] max ||b_j|| over the 32 items of a chunk (0 for padding chunks)
    const int* __restrict__ trp;
    const int* __restrict__ tri;
    const int* __restrict__ ustatus;
    uint2* cand;                            // [mb_pad][C] kept candidates: x = LOWER bound of the score (approximate score - error bound, float bits), y = item id
    int* cand_count;                        // [mb_pad] kept candidates; -1 = the user goes to the FMA path (band overflow / unscalable factors)
    int* overflow;                          // number of users flagged -1
    int* uflags;                            // [m] bit0: a candidate score was NaN
    int K;
    int sample_tiles, sample_stride, sample_rank;   // pass 0 (see filter_pass_tile); sample_tiles == 0: no sampling
    int* retries;                           // rows that needed the retry pass (statistics; may be nullptr)
};

struct FilterRowState {      // per user row of the CTA, shared by the four epilogue warps of its TMEM lane quarter
    float tau[BM];                   // K-th best lower bound so far (+inf: the row is closed, -inf: nothing known yet)
    float ca[BM], efl[BM];           // error bound of a score of this row: e = ca * chunk_norm + efl
    float guess[BM];
    int cnt[BM];                     // candidates left contiguous at the head of the row's buffer when a pass ends
    int cnt4[4][BM];                 // candidates in each warp's region of the buffer, published at the meeting points
    int trig[BM];                    // total above which the regions are cut back together
    int flags[BM];                   // 1 = NaN candidate score, 2 = buffer overflow (kept band / burst), 4 = guess failed (retry pass),
                                     // 8 = factors outside the range the fp16 image can be scaled into (FMA path)
    int nxt2_train[4][BM];           // per warp: the train item id after the cursor's next one (prefetched with cp.async)
    int tcur[4][BM];                 // per warp: position of the cursor in the train CSR (only touched in tiles holding train items)
    int tend[BM];                    // end of the row's train items in the CSR
    int tot_prev[4][BM];             // per warp: row total after the previous meeting (the same value in the quarter's four warps)
    int interval[F_EPI_WARPS];       // per warp: tiles between its last two meetings
    int retry;                       // some row of the CTA needs the retry pass
};


// Error bound of the filter's approximate scores, in the scaled units of the operand images (a' = a * 2^-ea with
// ||a'|| in [0.5, 1), b' = b * 2^-eb with max_j ||b'_j|| in [0.5, 1), every element at most 1 in magnitude):
//   fp16 rounding of an element x (|x| <= 1): x (1 + d) + h with |d| <= 2^-11 (normal range) and |h| <= 2^-25 (below 2^-14)
//       | sum_k a^_k b^_k - sum_k a'_k b'_k |  <=  (2^-10 + 2^-22) sum |a' b'|  +  2^-25 (1 + 2^-11) (sum |a'_k| + sum |b'_k|)  +  k 2^-50
//                                              <=  (2^-10 + 2^-22) ||a'|| ||b'_j||  +  2^-25 (1 + 2^-11) sqrt(k) (||a'|| + ||b'_j||)  +  k 2^-50
//   fp32 accumulation inside the tensor core plus the rounding of the exact fma chain it is compared with: k 2^-22 ||a'|| ||b'_j||
// With ||a'|| >= 0.5 the ||b'_j|| part of the second term is at most 2 x 2^-25 (1 + 2^-11) sqrt(k) ||a'|| ||b'_j||, so
//       e_uj = c_rel ||a'|| ||b'_j|| + c_abs ||a'|| + c_const        (and 1 % on top of every coefficient).
// The absolute terms matter for items whose norm is tiny next to the largest one: their fp16 image sits in the denormal
// range and its error no longer shrinks with ||b'_j||.
struct FilterErrCoef { float c_rel, c_abs, c_const; };
inline FilterErrCoef filter_err_coefs(int KB)
{
    const double c2 = std::ldexp(1.0, -25) * (1.0 + std::ldexp(1.0, -11)) * std::sqrt((double)KB);
    const double c1 = std::ldexp(1.0, -10) * (1.0 + std::ldexp(1.0, -10)) + KB * std::ldexp(1.0, -22);
    FilterErrCoef c;
    c.c_rel = (float)(1.01 * (c1 + 2.0 * c2));
    c.c_abs = (float)(1.01 * c2);
    c.c_const = (float)(1.01 * KB * std::ldexp(1.0, -50));
    return c;
}
// a norm the power-of-two scaling of prep.cuh can bring into [0.5, 1) (pow2_scale_for clamps its exponent at +-100)
__device__ __forceinline__ bool filter_scalable(const float nrm) { return nrm >= 1.6e-30f && nrm <= 6.0e29f; }

// dynamic shared memory: [row state, padded][barriers, 256 B][A tile][B ring]
constexpr size_t F_RS_BYTES = (sizeof(FilterRowState) + 1023) & ~size_t(1023);
inline size_t filter_smem_fixed_bytes() { return 256 + F_RS_BYTES; }
inline size_t filter_smem_bytes(int KB, int stages)
{
    return (size_t)(1 + stages) * KB * 128 * 2 + filter_smem_fixed_bytes();
}

// ------------------------------------------------------------------ tcgen05 wrappers
__device__ __forceinline__ uint64_t umma_desc(const unsigned saddr)
{
    // K-major, no swizzle: LBO = 128 rows * 16 B = 2048 (>>4 = 128), SBO = 128 B (>>4 = 8), version 1
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)128 << 16) | ((uint64_t)8 << 32) | (1ull << 46);
}
// the same descriptor `bytes` further into the tile: only the 14-bit address field (bytes >> 4) of the low word moves
// (shared-memory addresses stay below 2^18, so the field cannot carry into the LBO field)
__device__ __forceinline__ uint64_t umma_desc_advance(const uint64_t desc, const unsigned bytes) { return desc + (uint64_t)(bytes >> 4); }
__device__ __forceinline__ void umma_f16(const unsigned tmem_d, const uint64_t adesc, const uint64_t bdesc,
                                          const unsigned idesc, const unsigned accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(const unsigned bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// one lane of a converged warp (elect.sync): the compiler keeps what the elected lane computes in uniform registers
__device__ __forceinline__ bool elect_one()
{
    unsigned pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(const unsigned taddr, unsigned (&r)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// error bound of an approximate score of a row (ca, efl) against an item of a chunk with largest norm cn, rounded up
__device__ __forceinline__ float filter_err(const float ca, const float cn, const float efl) { return __fmaf_ru(ca, cn, efl); }

// One warp: cut a row's candidates back to those that can still belong to the exact top K.  Every candidate carries the
// LOWER bound lb = approx - e of its exact score (e from its item's chunk norm); its upper bound is lb + 2e.
// tau' = the K-th best lower bound; kept: ub >= tau' (whatever can still reach the exact top K).  The row's buffer is
// four regions of C/4 entries (one per epilogue warp of the quarter), region s holding cnt4[s] entries; all of them are
// read into registers first, so the survivors can be written back in place: CONTIG ? packed at the head of the buffer :
// dealt round-robin over the regions.
// tau' is found by bisection on the order-preserving keys: BITS halvings of [min key, max key], each one a count of the
// keys at or above the probe (compare + warp REDUX).  The interval's lower end always satisfies #(lb key >= lo) >= K,
// so it is a valid (slightly low: interval width = key range / 2^BITS) stand-in for tau'; BITS = 32 makes it exact.
// A cut stalls its warp -- and, once the four accumulator buffers have run full, the whole CTA -- for its duration:
// one load phase, no shared-memory traffic, no shuffles inside the search.  K <= total entries is required.
// Returns the number kept; *tau_out = (the stand-in for) tau'.
template <int C, int BITS, bool CONTIG>
__device__ __noinline__ int cut_regions(uint2* cd, const int c0, const int c1, const int c2, const int c3, const int K,
                                        const float ca, const float efl, const float* __restrict__ chunk_norm,
                                        const int lane, float* tau_out)
{
    constexpr int E = C / 32, RC = C / 4, EPR = E / 4;      // entries per lane, region capacity, per-lane entries per region
    const int ns = (max(max(c0, c1), max(c2, c3)) + 31) >> 5;      // occupied 32-entry slots per region (warp-uniform): the rest is skipped
    unsigned lbk[E];                                        // lower-bound key, 0 = empty slot (the key of -inf is 0x007fffff)
    int it[E];
    unsigned kmax = 0u, kmin = 0xffffffffu;
#pragma unroll
    for (int e = 0; e < E; e++) {
        lbk[e] = 0u; it[e] = 0;
        if ((e % EPR) < ns) {
            const int region = e / EPR, pos = (e % EPR) * 32 + lane;
            const int cr = region == 0 ? c0 : (region == 1 ? c1 : (region == 2 ? c2 : c3));
            if (pos < cr) {
                const uint2 c = cd[region * RC + pos];
                lbk[e] = NumTraits<float>::key(__uint_as_float(c.x));
                it[e] = (int)c.y;
                kmax = max(kmax, lbk[e]); kmin = min(kmin, lbk[e]);
            }
        }
    }
    kmax = __reduce_max_sync(FULL, kmax);
    kmin = __reduce_min_sync(FULL, kmin);
    unsigned lo = kmin, hi = kmax;              // #(key >= lo) >= K always; the K-th largest key lies in [lo, hi]
#pragma unroll 1
    for (int step = 0; step < BITS && lo < hi; step++) {
        const unsigned mid = lo + ((hi - lo + 1u) >> 1);
        int c = 0;
#pragma unroll
        for (int e = 0; e < E; e++)
            if ((e % EPR) < ns) c += (lbk[e] >= mid) ? 1 : 0;
        c = __reduce_add_sync(FULL, c);
        if (c >= K) lo = mid; else hi = mid - 1u;
    }
    const float tau = NumTraits<float>::from_orderable((u64)lo);
    *tau_out = tau;
    const unsigned cut = (tau == tau) ? lo : 1u;               // NaN bound (K NaN scores): keep everything
    // write-back: an entry whose lower bound reaches the cut stays; one below it stays iff its UPPER bound lb + 2e does
    // -- only those look their error bound up.
    int base = 0;
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; e++) {
        if ((e % EPR) < ns) {
            bool keep = lbk[e] != 0u && lbk[e] >= cut;
            if (!keep && lbk[e] != 0u) {
                const float er = filter_err(ca, chunk_norm[(unsigned)it[e] >> 5], efl);
                const float ub = __fadd_ru(NumTraits<float>::from_orderable((u64)lbk[e]), __fadd_ru(er, er));
                keep = NumTraits<float>::key(ub) >= cut;
            }
            const unsigned mask = __ballot_sync(FULL, keep);
            if (keep) {
                const int k = base + __popc(mask & ((1u << lane) - 1u));
                const int pos = CONTIG ? k : (k & 3) * RC + (k >> 2);
                cd[pos] = make_uint2(__float_as_uint(NumTraits<float>::from_orderable((u64)lbk[e])), (unsigned)it[e]);
            }
            base += __popc(mask);
        }
    }
    __syncwarp();
    return base;
}

// General slow path of the filter, out of line and in ONE copy: the 8 scores of a column group of which at least one is
// not below the threshold, in a tile where the row has train items, in the catalogue's last (partial) tile, or when the
// warp's region is nearly full.  Padding columns and train items are dropped (hpp:494-495; [t_lo, t_hi) = the part of
// the row's sorted train items that can intersect this tile: the few inside the tile are scanned linearly), the rest is
// appended to this warp's region of the row's candidate buffer (flag 2 when it is full).  NaN scores are appended like
// any other (a NaN is never below a threshold and sorts above everything at the cuts): the exact stage raises the
// user's NaN flag (hpp:195-197).  Returns the new fill of the region.
template <int RC>
__device__ __noinline__ int filter_append_group(const float s0, const float s1, const float s2, const float s3,
                                                const float s4, const float s5, const float s6, const float s7,
                                                const float thr, const float err, const int item0, const int n,
                                                const int* __restrict__ tri, const int t_lo, const int t_hi,
                                                uint2* cd, int mycnt, const int row)
{
    // which of the 8 pass (branch-free), then one trip per passing score (almost always a single one)
    unsigned m = (s0 < thr ? 0u : 1u) | (s1 < thr ? 0u : 2u) | (s2 < thr ? 0u : 4u) | (s3 < thr ? 0u : 8u) |
                 (s4 < thr ? 0u : 16u) | (s5 < thr ? 0u : 32u) | (s6 < thr ? 0u : 64u) | (s7 < thr ? 0u : 128u);
    while (m) {
        const int jj = __ffs(m) - 1;
        m &= m - 1;
        const float lo4 = (jj & 2) ? ((jj & 1) ? s3 : s2) : ((jj & 1) ? s1 : s0);
        const float hi4 = (jj & 2) ? ((jj & 1) ? s7 : s6) : ((jj & 1) ? s5 : s4);
        const float s = (jj & 4) ? hi4 : lo4;
        const int item = item0 + jj;
        if (item >= n) break;                                   // padding columns (and all after them)
        bool in_train = false;
        for (int lo = t_lo; lo < t_hi; lo++) {
            const int v = tri[lo];
            if (v >= item) { in_train = (v == item); break; }
        }
        if (in_train) continue;
        if (mycnt < RC) { cd[mycnt] = make_uint2(__float_as_uint(__fsub_rd(s, err)), (unsigned)item); mycnt++; }
        else atomicOr(&reinterpret_cast<FilterRowState*>(smem_raw)->flags[row], 2);
    }
    return mycnt;
}

// The item tiles a CTA walks, pass by pass (all roles -- TMA producer, MMA issuer, epilogue -- step through the same list):
//   pass 0  SAMPLE  every sample_stride-th tile (sample_tiles of them, ~1/16 of the catalogue; skipped when sample_tiles == 0).
//                   The rows run the same streaming selection with K = sample_rank on the LOWER bounds; the sample_rank-th best
//                   lower bound of the sample becomes the row's GUESS g: with sample_rank chosen by the host so that
//                   P(fewer than K of ALL items reach the sample's sample_rank-th best) <= 1e-6 per row.
//   pass 1  MAIN    every tile, tau' starts at g instead of -inf.  A streaming top-K appends K' (1 + ln(n / K'))
//                   candidates per row, more than half of them in the first percent of the catalogue while the threshold is
//                   still loose; starting from the guess leaves about (items whose upper bound reaches g) appends, 3x fewer at 1M items.
//                   The guess is VERIFIED: the pass is valid for a row iff at least K of its kept candidates have a lower
//                   bound >= g (then the final tau' >= g never fell below the threshold any item was tested against).
//   pass 2  RETRY   only if some row of the CTA failed the check (or had too few sample candidates): every tile again,
//                   failed rows from -inf, the others closed.  Costs the CTA a second walk; never changes a result.
__device__ __forceinline__ int filter_pass_tiles(const FilterParams& P, const int pass, const int NT) { return pass == 0 ? P.sample_tiles : NT; }
__device__ __forceinline__ int filter_pass_tile(const FilterParams& P, const int pass, const int j) { return pass == 0 ? j * P.sample_stride : j; }

template <int C>
__global__ void __launch_bounds__(F_THREADS, 1)
filter_select_kernel(const __grid_constant__ FilterParams P)
{
    const int KB = P.KB, S = P.stages;
    const unsigned tile_bytes = (unsigned)KB * 128u * 2u;          // one operand tile (A or B)
    FilterRowState* rs = reinterpret_cast<FilterRowState*>(smem_raw);
    u64* bars = reinterpret_cast<u64*>(smem_raw + F_RS_BYTES);
    unsigned char* a_tile = smem_raw + F_RS_BYTES + 256;
    unsigned char* b_ring = a_tile + tile_bytes;
    // barriers: full[F_MAX_STAGES], empty[F_MAX_STAGES], acc_full[4], acc_empty[4], a_full
    const unsigned bar_full = smem_u32(bars), bar_empty = bar_full + 8 * F_MAX_STAGES;
    const unsigned bar_accf = bar_empty + 8 * F_MAX_STAGES, bar_acce = bar_accf + 32, bar_a = bar_acce + 32;
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * F_MAX_STAGES + 9);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile_u0 = blockIdx.x * BM;
    const int NT = (P.n + FN - 1) / FN;

    if (tid == 0) {
        for (int s = 0; s < F_MAX_STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < F_ACCBUFS; b++) { mbar_init(bar_accf + 8 * b, 1); mbar_init(bar_acce + 8 * b, F_EPI_WARPS); }
        mbar_init(bar_a, 1);
        mbar_fence_init();
        rs->retry = 0;
    }
    if (warp == F_EPI_WARPS + 1) {      // the MMA warp owns the tensor-memory allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((unsigned)F_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = *tmem_slot;

    if (warp == F_EPI_WARPS && elect_one()) {
        mbar_arrive_expect_tx(bar_a, tile_bytes);
        tma_bulk_g2s(smem_u32(a_tile), P.Ab + (size_t)blockIdx.x * KB * 128, tile_bytes, bar_a);
    }

    int it0 = 0;                         // pipeline iterations before this pass (ring stage / accumulator buffer / parities follow it)
    for (int pass = P.sample_tiles > 0 ? 0 : 1; pass < 3; pass++) {
        const int ntiles = filter_pass_tiles(P, pass, NT);
        if (warp == F_EPI_WARPS) {
            // ===================== TMA producer (the warp stays converged, one elected lane issues) =====================
            int s = it0 % S, ph = (it0 / S) & 1;                             // ring stage and its phase parity
            for (int j = 0; j < ntiles; j++) {
                mbar_wait(bar_empty + 8 * s, ph ^ 1);                         // first round passes immediately
                if (elect_one()) {
                    mbar_arrive_expect_tx(bar_full + 8 * s, tile_bytes);
                    tma_bulk_g2s(smem_u32(b_ring) + (unsigned)s * tile_bytes, P.Bb + (size_t)filter_pass_tile(P, pass, j) * KB * 128,
                                 tile_bytes, bar_full + 8 * s);
                }
                __syncwarp();
                if (++s == S) { s = 0; ph ^= 1; }
            }
        } else if (warp > F_EPI_WARPS) {
            // ===================== MMA issuers (converged warps, one elected lane issues; warp w takes iterations it % F_MMA_WARPS == w) =====================
            // D fp32 (bit 4), A and B fp16 (format 0 at bits 7 and 10), both K-major, N=128 (>>3 at bit 17), M=128 (>>4 at bit 24)
            const unsigned idesc = (1u << 4) | ((unsigned)(FN >> 3) << 17) | ((128u >> 4) << 24);
            const uint64_t adesc0 = umma_desc(smem_u32(a_tile)), bdesc0 = umma_desc(smem_u32(b_ring));
            const int ksteps = KB / 16;                                       // K=16 per MMA = two 16-byte k chunks of 2048 B
            const int w = warp - (F_EPI_WARPS + 1);
            mbar_wait(bar_a, 0);
            int j = (w - it0 % F_MMA_WARPS + F_MMA_WARPS) % F_MMA_WARPS;      // first iteration of this pass that is this warp's
            int s = (it0 + j) % S, ph = ((it0 + j) / S) & 1;
            for (; j < ntiles; j += F_MMA_WARPS) {
                const int it = it0 + j, b = it & (F_ACCBUFS - 1);
                mbar_wait(bar_acce + 8 * b, ((it >> F_ACCSHIFT) & 1) ^ 1);     // accumulator buffer drained by the epilogue
                mbar_wait(bar_full + 8 * s, ph);                              // B tile landed
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t bdesc = umma_desc_advance(bdesc0, (unsigned)s * tile_bytes);
                    const unsigned d = tmem_base + (unsigned)(b * FN);
                    umma_f16(d, adesc0, bdesc, idesc, 0u);
#pragma unroll 7
                    for (int ks = 1; ks < ksteps; ks++)
                        umma_f16(d, umma_desc_advance(adesc0, ks * 4096), umma_desc_advance(bdesc, ks * 4096), idesc, 1u);
                    umma_commit(bar_empty + 8 * s);                       // stage reusable once these MMAs have read it
                    umma_commit(bar_accf + 8 * b);                        // accumulator complete
                }
                __syncwarp();
                s += F_MMA_WARPS;
                while (s >= S) { s -= S; ph ^= 1; }
            }
        } else {
            // ===================== epilogue warps =====================
            constexpr int RC = C / 4;                       // capacity of a warp's region of the row's candidate buffer
            const int q = warp & 3, slot = warp >> 2;       // TMEM lane quarter, 32-column chunk of the tile
            const int row = q * 32 + lane;                  // user row of this thread (shared with the 3 other slots)
            const int ul = tile_u0 + row;
            const unsigned qbar = 1 + q;                    // named barrier of the quarter's four warps
            const int Kp = pass == 0 ? P.sample_rank : P.K; // how many best candidates the pass keeps track of
            if (slot == 0) {
                bool ranked = (ul < P.mb) && (P.ustatus[P.user0 + ul] == 0);
                if (pass < 2 && (pass == 0 || P.sample_tiles == 0)) {            // first pass of the CTA: the row's error-bound terms
                    int fl = 0;
                    float ca = 0.f, efl = 0.f;
                    if (ranked) {
                        const float an = P.anorm[ul], bn = __uint_as_float(*P.maxbn);
                        if (an == 0.f) ranked = false;                           // all-zero user factors: every score equal, NaN row (hpp:541-548, :524-527)
                        else if (!(filter_scalable(an) && filter_scalable(bn))) { fl = 8; ranked = false; }
                        // |score| <= ||a|| ||b|| (the bias is one more factor of both norms): a user whose scores can
                        // overflow to +-inf goes back too, so that the path it lands on sees every infinite candidate
                        // (under the noise one anywhere makes the row NaN, hpp:524-527; the exact stage sees survivors only)
                        else if (!(an * bn <= P.score_max)) { fl = 8; ranked = false; }
                        else {
                            const float sa = pow2_scale_for(an), sb = pow2_scale_for(bn);
                            const float ap = an * sa;                                            // ||a'|| in [0.5, 1.002)
                            ca = __fmul_ru(__fmul_ru(P.c_rel, ap), sb);                          // x ||b_j|| (unscaled chunk norm)
                            efl = __fadd_ru(__fmaf_ru(P.c_abs, ap, P.c_const), 0.5f * P.noise_band * sa * sb);
                        }
                    }
                    rs->flags[row] = fl;
                    rs->guess[row] = -CUDART_INF_F;
                    rs->ca[row] = ca;
                    rs->efl[row] = efl;
                    rs->cnt[row] = 0;
                    rs->trig[row] = ranked ? 0 : -1;                             // (-1 marks rows that are never ranked, see below)
                }
                ranked = ranked && rs->trig[row] != -1 && !(rs->flags[row] & 8);
                float tau0 = CUDART_INF_F;                  // +inf: the row is closed
                if (pass == 0) { if (ranked) tau0 = -CUDART_INF_F; }
                else if (pass == 1) { if (ranked) { tau0 = rs->guess[row]; if (!(tau0 == tau0)) tau0 = -CUDART_INF_F; } }
                else if (ranked && (rs->flags[row] & 4)) tau0 = -CUDART_INF_F;
                rs->tau[row] = tau0;
                if (rs->trig[row] != -1) rs->trig[row] = Kp + (pass == 1 && P.sample_tiles > 0 ? F_MAIN_MARGIN : F_CUT_MARGIN);
                if (tau0 != CUDART_INF_F || pass < 2) rs->cnt[row] = 0;   // (a row closed in the retry pass keeps what pass 1 found)
            }
            asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
            // private per-thread row state: region fill, cursor into the row's sorted train items (hpp:494-495 takes those out
            // of the pool): t_nxt = the first train item id >= the current tile, the one after it prefetched in shared memory
            int mycnt = 0, t_nxt = INT_MAX;
            float tau = rs->tau[row];                       // the row's bound only moves at the meetings: kept in a register in between
            {
                int t_cur = 0, t_end = 0;
                if (tau != CUDART_INF_F) {
                    t_cur = P.trp[P.user0 + ul]; t_end = P.trp[P.user0 + ul + 1];
                    if (t_cur < t_end) t_nxt = P.tri[t_cur];
                    rs->nxt2_train[slot][row] = t_cur + 1 < t_end ? P.tri[t_cur + 1] : INT_MAX;
                }
                rs->tcur[slot][row] = t_cur;
                rs->tend[row] = t_end;                      // (the same value from the row's four warps)
                rs->tot_prev[slot][row] = 0;
                if (lane == 0) rs->interval[warp] = 1;
            }
            if (pass == 0) {
                // ===== SAMPLE pass: the guess is the sample_rank-th largest of the row's GROUP MAXIMA.  The sample tiles are cut into
                // up to F_GROUPS groups of consecutive tiles; a lane keeps the largest lower bound (chunk maximum - the chunk's error
                // bound) its warp's columns reach in the current group -- one FADD and one FMNMX per tile on top of the fast path, no
                // appends, no cuts, no meetings -- and stores it at the group's end.  The r largest group maxima are r different
                // items of the sample, so the r-th largest of them is <= the r-th best lower bound of the sample: a valid (slightly
                // lower) stand-in for it.  A chunk holding one of the row's train items is left out of the sample (hpp:494-495).
                constexpr int F_GROUPS = RC < 128 ? RC : 128;
                const int tpg = (ntiles + F_GROUPS - 1) / F_GROUPS;            // tiles per group
                const float ca_r = rs->ca[row], efl_r = rs->efl[row];
                uint2* const cdg = P.cand + ((size_t)ul * C + slot * RC);      // this warp's region holds its partial group maxima
                float gmax = -CUDART_INF_F;
                int tg = 0, g = 0;
                int buf = it0 & (F_ACCBUFS - 1);
                unsigned par = (unsigned)(it0 >> F_ACCSHIFT) & 1u;
                int item_base = slot * F_CHUNK;
                const int item_step = P.sample_stride * FN;
                const unsigned taddr0 = tmem_base + ((unsigned)(q * 32) << 16) + (unsigned)(slot * F_CHUNK);
#pragma unroll 1
                for (int left = ntiles; left > 0; left--, item_base += item_step) {
                    const int tile_end = item_base - slot * F_CHUNK + FN;
                    const float cn = __ldg(P.chunk_norm + (item_base >> 5));
                    mbar_wait(bar_accf + 8 * buf, par);
                    tc_fence_after();
                    unsigned v[32];
                    tmem_ld32(taddr0 + (unsigned)(buf * FN), v);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acce + 8 * buf);
                    if (++buf == F_ACCBUFS) { buf = 0; par ^= 1u; }
                    float m32 = __uint_as_float(v[0]);
#pragma unroll
                    for (int e = 1; e < 32; e++) m32 = max_nan(m32, __uint_as_float(v[e]));
                    bool skip = false;
                    if (t_nxt < tile_end) {
                        asm volatile("cp.async.wait_all;" ::: "memory");
                        skip = t_nxt >= item_base && t_nxt < item_base + F_CHUNK;
                        int nxt = rs->nxt2_train[slot][row];
                        int t_cur = rs->tcur[slot][row] + 1;
                        const int t_end = rs->tend[row];
                        while (nxt < tile_end) {
                            skip = skip || (nxt >= item_base && nxt < item_base + F_CHUNK);
                            t_cur++;
                            nxt = t_cur < t_end ? P.tri[t_cur] : INT_MAX;
                        }
                        t_nxt = nxt;
                        rs->tcur[slot][row] = t_cur;
                        if (t_cur + 1 < t_end)
                            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(&rs->nxt2_train[slot][row])), "l"(P.tri + t_cur + 1) : "memory");
                        else rs->nxt2_train[slot][row] = INT_MAX;
                    }
                    const float lbm = __fsub_rd(m32, filter_err(ca_r, cn, efl_r));
                    if (!skip) gmax = max_nan(gmax, lbm);
                    if (++tg == tpg || left == 1) {
                        cdg[g] = make_uint2(__float_as_uint(gmax), 0u);
                        g++; tg = 0; gmax = -CUDART_INF_F;
                    }
                }
                const int ngroups = (ntiles + tpg - 1) / tpg;
                asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");       // the quarter's four warps have stored their partial maxima
                for (int r = slot; r < 32; r += 4) {
                    const int rr = q * 32 + r;
                    const uint2* cr = P.cand + (size_t)(tile_u0 + rr) * C;
                    unsigned k[F_GROUPS / 32];
#pragma unroll
                    for (int j = 0; j < F_GROUPS / 32; j++) {
                        const int gg = j * 32 + lane;
                        k[j] = 0u;                                                 // (no group: below every score)
                        if (gg < ngroups) {
                            const float m01 = max_nan(__uint_as_float(cr[gg].x), __uint_as_float(cr[RC + gg].x));
                            const float m23 = max_nan(__uint_as_float(cr[2 * RC + gg].x), __uint_as_float(cr[3 * RC + gg].x));
                            k[j] = NumTraits<float>::key(max_nan(m01, m23));
                        }
                    }
                    unsigned lo = 0u, hi = 0xffffffffu;                           // the sample_rank-th largest key, by bisection (exact)
#pragma unroll 1
                    for (int step = 0; step < 32 && lo < hi; step++) {
                        const unsigned mid = lo + ((hi - lo) >> 1) + 1u;
                        int c = 0;
#pragma unroll
                        for (int j = 0; j < F_GROUPS / 32; j++) c += (k[j] >= mid) ? 1 : 0;
                        c = __reduce_add_sync(FULL, c);
                        if (c >= P.sample_rank) lo = mid; else hi = mid - 1u;
                    }
                    if (lane == 0) {
                        const float gs = NumTraits<float>::from_orderable((u64)lo);
                        rs->guess[rr] = (lo != 0u && gs == gs) ? gs : -CUDART_INF_F;   // too few groups / NaN scores: no guess
                    }
                }
                asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
            } else {
            // error bound in the tile loop: candidates pass on their upper bounds, approx + e >= tau'
            const float ca_l = rs->ca[row];
            float tau_m = __fsub_rd(tau, rs->efl[row]);     // tau' minus the row's constant error term
            int meet_in = 0;                                // tiles until the next meeting
            // loop-carried pipeline state, kept incrementally (no per-tile index arithmetic): accumulator buffer and its phase
            // parity, first item id of this warp's 32-column chunk
            int buf = it0 & (F_ACCBUFS - 1);
            unsigned par = (unsigned)(it0 >> F_ACCSHIFT) & 1u;
            int item_base = slot * F_CHUNK;
            const unsigned taddr0 = tmem_base + ((unsigned)(q * 32) << 16) + (unsigned)(slot * F_CHUNK);

#pragma unroll 1
            for (int left = ntiles; left > 0; left--, item_base += FN) {
                const int tile_end = item_base - slot * F_CHUNK + FN;
                const float cn = __ldg(P.chunk_norm + (item_base >> 5));       // largest item norm of this chunk (in flight while the warp waits)
                mbar_wait(bar_accf + 8 * buf, par);
                tc_fence_after();
                unsigned v[32];
                tmem_ld32(taddr0 + (unsigned)(buf * FN), v);
                tc_fence_before();                      // this warp's part of the accumulator is in registers
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_acce + 8 * buf);
                if (++buf == F_ACCBUFS) { buf = 0; par ^= 1u; }
                const bool has_train = t_nxt < tile_end;
                // NaN-propagating max of each group of 8 columns; one compare for the whole chunk, groups only when it passes
                float gm[4];
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const float m01 = max_nan(__uint_as_float(v[8 * g + 0]), __uint_as_float(v[8 * g + 1]));
                    const float m23 = max_nan(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3]));
                    const float m45 = max_nan(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5]));
                    const float m67 = max_nan(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7]));
                    gm[g] = max_nan(max_nan(m01, m23), max_nan(m45, m67));
                }
                const float thr = __fmaf_rd(-ca_l, cn, tau_m);                     // approx < thr: the upper bound stays below tau'
                if (!(max_nan(max_nan(gm[0], gm[1]), max_nan(gm[2], gm[3])) < thr)) {
                    uint2* cd = P.cand + ((size_t)ul * C + slot * RC);            // this warp's region of the row's buffer
                    asm volatile("" : "+l"(cd));                                  // (one pointer, indexed by the fill: keeps the address math to one IMAD.WIDE per store)
                    const float err = filter_err(rs->ca[row], cn, rs->efl[row]);  // candidates are stored with their lower bound
                    if (!has_train && tile_end <= P.n && mycnt <= RC - F_CHUNK) {
                        // common case (no train item of the row in this tile, no padding column, room for the whole chunk):
                        // predicated appends, no calls, no loops
#pragma unroll
                        for (int g = 0; g < 4; g++) {
                            if (!(gm[g] < thr)) {
#pragma unroll
                                for (int e8 = 0; e8 < 8; e8++) {
                                    if (!(__uint_as_float(v[8 * g + e8]) < thr)) {
                                        cd[mycnt] = make_uint2(__float_as_uint(__fsub_rd(__uint_as_float(v[8 * g + e8]), err)), (unsigned)(item_base + 8 * g + e8));
                                        mycnt++;
                                    }
                                }
                            }
                        }
                    } else {
#pragma unroll
                        for (int g = 0; g < 4; g++) {
                            if (!(gm[g] < thr)) {
                                const int t_cur = rs->tcur[slot][row];
                                mycnt = filter_append_group<RC>(__uint_as_float(v[8 * g + 0]), __uint_as_float(v[8 * g + 1]), __uint_as_float(v[8 * g + 2]),
                                                                __uint_as_float(v[8 * g + 3]), __uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5]),
                                                                __uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7]), thr, err, item_base + 8 * g, P.n,
                                                                P.tri, t_cur, has_train ? rs->tend[row] : t_cur, cd, mycnt, row);
                            }
                        }
                    }
                }
                // move the train cursor past this tile: the id after t_nxt was prefetched into shared memory when the cursor last moved
                if (has_train) {
                    asm volatile("cp.async.wait_all;" ::: "memory");
                    int nxt = rs->nxt2_train[slot][row];
                    int t_cur = rs->tcur[slot][row] + 1;
                    const int t_end = rs->tend[row];
                    while (nxt < tile_end) { t_cur++; nxt = t_cur < t_end ? P.tri[t_cur] : INT_MAX; }    // several train items in one tile
                    t_nxt = nxt;
                    rs->tcur[slot][row] = t_cur;
                    if (t_cur + 1 < t_end)
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(&rs->nxt2_train[slot][row])), "l"(P.tri + t_cur + 1) : "memory");
                    else rs->nxt2_train[slot][row] = INT_MAX;
                }
                if (--meet_in >= 0 && left > 1) continue;

                // ---- meeting point of the quarter's four warps: publish the region fills, cut rows that grew past their trigger
                rs->cnt4[slot][row] = mycnt;
                asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
                int c0 = rs->cnt4[0][row], c1 = rs->cnt4[1][row], c2 = rs->cnt4[2][row], c3 = rs->cnt4[3][row];
                int tot = c0 + c1 + c2 + c3;
                const int grown = tot - rs->tot_prev[slot][row];                   // appends to the row since the previous meeting
                unsigned need = __ballot_sync(FULL, tot > rs->trig[row] && rs->trig[row] >= 0 && !(rs->flags[row] & 2));
                if (left == 1) need = 0;                                       // the pass ends with the exact cut below
                if (need) {                                                    // (the same mask in all four warps)
                    while (need) {
                        const int r = __ffs(need) - 1;
                        need &= need - 1;
                        if ((r & 3) != slot) continue;                         // the quarter's warps share the work
                        const int rr = q * 32 + r;
                        float tau_r;
                        const int kept = cut_regions<C, F_CUT_BITS, false>(P.cand + (size_t)(tile_u0 + rr) * C, rs->cnt4[0][rr], rs->cnt4[1][rr],
                                                                              rs->cnt4[2][rr], rs->cnt4[3][rr], Kp, rs->ca[rr], rs->efl[rr], P.chunk_norm,
                                                                              lane, &tau_r);
                        if (lane == 0) {
                            float t_new = fmaxf(tau_r, rs->tau[rr]);            // an earlier (valid) bound may be the sharper one; a NaN bound is ignored
                            if (kept > 4 * (RC - 32)) { rs->flags[rr] |= 2; t_new = CUDART_INF_F; }     // the kept band does not fit
                            rs->tau[rr] = t_new;
                            rs->trig[rr] = kept + (pass == 1 && P.sample_tiles > 0 ? F_MAIN_MARGIN : F_CUT_MARGIN);
#pragma unroll
                            for (int sgm = 0; sgm < 4; sgm++) rs->cnt4[sgm][rr] = (kept + 3 - sgm) >> 2;
                        }
                    }
                    asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
                    c0 = rs->cnt4[0][row]; c1 = rs->cnt4[1][row]; c2 = rs->cnt4[2][row]; c3 = rs->cnt4[3][row];
                    tot = c0 + c1 + c2 + c3;
                    mycnt = slot == 0 ? c0 : (slot == 1 ? c1 : (slot == 2 ? c2 : c3));
                }
                tau = rs->tau[row];
                if (rs->flags[row] & 2) { mycnt = 0; tau = CUDART_INF_F; if (slot == 0) rs->tau[row] = CUDART_INF_F; }     // the row is closed: whatever it holds is void
                tau_m = __fsub_rd(tau, rs->efl[row]);
                const int interval = rs->interval[warp];
                // next meeting: far enough that barriers are rare, close enough that no region can fill up at twice the
                // append rate just seen (all of it into one region); a burst beyond that closes the row (flag 2)
                const int headroom = RC - max(max(c0, c1), max(c2, c3));
                int nxt_iv = grown > 0 ? (headroom * interval) / (2 * grown) : F_MAX_MEET;
                nxt_iv = __reduce_min_sync(FULL, nxt_iv);
                nxt_iv = nxt_iv < 1 ? 1 : (nxt_iv > F_MAX_MEET ? F_MAX_MEET : nxt_iv);
                meet_in = nxt_iv - 1;
                rs->tot_prev[slot][row] = tot;
                if (lane == 0) rs->interval[warp] = nxt_iv;
            }
            // end of the pass (all four warps are past the last meeting): the exact Kp-th best lower bound of what each
            // row kept, the survivors packed at the head of the row's buffer
            for (int r = slot; r < 32; r += 4) {
                const int rr = q * 32 + r;
                if (rs->tau[rr] == CUDART_INF_F && !(rs->flags[rr] & 2)) continue;    // closed row (not ranked / settled in pass 1)
                const int c0 = rs->cnt4[0][rr], c1 = rs->cnt4[1][rr], c2 = rs->cnt4[2][rr], c3 = rs->cnt4[3][rr];
                const int nv = c0 + c1 + c2 + c3;
                float tau_r = -CUDART_INF_F;
                const bool have_k = nv >= Kp && !(rs->flags[rr] & 2);
                if (nv > 0 && !(rs->flags[rr] & 2)) {
                    const int kept = cut_regions<C, 32, true>(P.cand + (size_t)(tile_u0 + rr) * C, c0, c1, c2, c3, have_k ? Kp : nv, rs->ca[rr], rs->efl[rr],
                                                             P.chunk_norm, lane, &tau_r);
                    if (lane == 0) rs->cnt[rr] = kept;                  // last cut: the exact stage gets only what can still be in the top K
                }
                if (lane == 0 && pass == 1 && !(rs->flags[rr] & 2)) {
                    const float g = rs->guess[rr];
                    const bool ok = (g == -CUDART_INF_F) || (have_k && !(tau_r < g));     // >= K kept lower bounds reach the guess (a NaN bound: everything was kept)
                    if (!ok) { rs->flags[rr] |= 4; rs->retry = 1; }
                }
            }
            asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
            }   // (passes 1 and 2)
        }
        it0 += ntiles;
        if (pass == 0) continue;         // the sample's result is consumed by the epilogue warps alone
        __syncthreads();
        const unsigned again = rs->retry != 0 ? 1u : 0u;
        if (pass == 2 || !__any_sync(FULL, again != 0u)) break;          // (a vote: the compiler keeps the pass loop warp-uniform)
    }

    if (warp < F_EPI_WARPS && (warp >> 2) == 0) {
        const int row = (warp & 3) * 32 + lane, ul = tile_u0 + row;
        if (ul < P.mb) {
            const int fl = rs->flags[row];
            const bool to_fma = (fl & (2 | 8)) != 0;
            P.cand_count[ul] = to_fma ? -1 : rs->cnt[row];
            if (to_fma) atomicAdd(P.overflow, 1);
            if ((fl & 4) && P.retries) atomicAdd(P.retries, 1);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == F_EPI_WARPS + 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((unsigned)F_TMEM_COLS));
}

// One warp per user: exact scores of the candidates the filter kept (sequential fma chain over the original
// factors, + bias: the chain of score_select_kernel / score_entries_kernel, so the values are bit-identical
// to the FMA path), NaN scores raise the user's NaN flag (hpp:195-197), best K (score descending, ties by
// ascending item id) left unordered at the head of cand_score / cand_item.
// MODE 1 / 2 (staged): the item-factor rows of 32 candidates at a time are fetched with cp.async into shared memory --
// all 32 rows in flight at once, no registers in between -- then every lane runs the chain of its own candidate from
// there.  MODE 2 moves 16 bytes per cp.async and reads the rows back with 16-byte loads (row stride p_pad + 16 bytes:
// conflict-free for 16-byte accesses); it needs factor rows that are 16-byte aligned and a multiple of 16 bytes long.
// MODE 1 moves single elements (row stride p_pad + 1).  MODE 0 reads the rows straight from global memory.
constexpr int EXACT_WARPS = 4;
__device__ __forceinline__ void cp_async_elem(float* dst, const float* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_elem(double* dst, const double* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* dst, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
// per warp: 32 rows of p_pad + 16 bytes (either staged mode fits) + the user's factors
inline size_t exact_topk_smem_bytes(int p_pad, size_t elem) { return (size_t)EXACT_WARPS * (32 * (size_t)(p_pad + 16 / elem) + p_pad) * elem; }

// Best K of the warp's scored candidates (key: order-preserving integer image of the score, 0 = empty slot; ties at the
// cut by ascending item id), written unordered to the head of the user's buffer.  Only the first EU of the E register
// slots per lane can be occupied.  Returns the number kept.
template <typename T, int E, int EU>
__device__ __forceinline__ int exact_select(const typename NumTraits<T>::key_t (&key)[E], const int (&it)[E], const int K, const int lane,
                                            T* cs, int* cio)
{
    typedef typename NumTraits<T>::key_t key_t;
    int nvalid = 0;
#pragma unroll
    for (int e = 0; e < EU; e++) nvalid += (key[e] != 0) ? 1 : 0;
    nvalid = __reduce_add_sync(FULL, nvalid);
    key_t t = 0;                  // keep key > t, and key == t with item id <= id_cut
    unsigned id_cut = 0x7fffffffu;
    if (nvalid > K) {
        for (int b = NumTraits<T>::KEYBITS - 1; b >= 0; b--) {
            const key_t cand = t | ((key_t)1 << b);
            int c = 0;
#pragma unroll
            for (int e = 0; e < EU; e++) c += (key[e] >= cand) ? 1 : 0;
            c = __reduce_add_sync(FULL, c);
            if (c >= K) t = cand;
        }
        int cgt = 0, cge = 0;
#pragma unroll
        for (int e = 0; e < EU; e++) { cgt += (key[e] > t) ? 1 : 0; cge += (key[e] >= t) ? 1 : 0; }
        cgt = __reduce_add_sync(FULL, cgt);
        cge = __reduce_add_sync(FULL, cge);
        if (cge > K) {
            const int need = K - cgt;
            unsigned x = 0;
            for (int b = 30; b >= 0; b--) {
                const unsigned cand = x | (1u << b);
                int c = 0;
#pragma unroll
                for (int e = 0; e < EU; e++) c += (key[e] == t && (unsigned)it[e] < cand) ? 1 : 0;
                c = __reduce_add_sync(FULL, c);
                if (c < need) x = cand;
            }
            id_cut = x;
        }
    }
    __syncwarp();
    int base = 0;
#pragma unroll
    for (int e = 0; e < EU; e++) {
        const bool keep = (key[e] != 0) && ((key[e] > t) || (key[e] == t && (unsigned)it[e] <= id_cut));
        const unsigned mask = __ballot_sync(FULL, keep);
        if (keep) {
            const int pos = base + __popc(mask & ((1u << lane) - 1u));
            cs[pos] = NumTraits<T>::from_orderable((u64)key[e]);
            cio[pos] = it[e];
        }
        base += __popc(mask);
    }
    return base;
}

// optional statistic (developer / tests): how close the observed error of the filter's approximate scores comes to its bound
struct FilterErrStat {
    const float* anorm;            // [mb]
    const unsigned* maxbn;
    const float* chunk_norm;
    float c_rel, c_abs, c_const;
    unsigned* max_ratio_bits;      // float bits of max over re-scored candidates of |approx - exact| / bound (nullptr: off)
};

template <typename T, int C, int MODE>
__global__ void __launch_bounds__(EXACT_WARPS * 32)
exact_topk_kernel(const uint2* __restrict__ cand, T* __restrict__ cand_score, int* __restrict__ cand_item,
                  int* __restrict__ cand_count, const int mb, const int user0,
                  const T* __restrict__ At, const int p_pad, const int p,
                  const T* __restrict__ Brow, const size_t ldb, const T* __restrict__ bias,
                  int* __restrict__ uflags, const int K,
                  const int noise, const unsigned long long seed_user0, const size_t mt_off,
                  const int* __restrict__ trp, const int* __restrict__ tri, const int n, const FilterErrStat es)
{
    typedef typename NumTraits<T>::key_t key_t;
    constexpr int E = C / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ul = blockIdx.x * EXACT_WARPS + warp;
    if (ul >= mb) return;
    const int nv = cand_count[ul];
    if (nv <= 0) return;
    const T* __restrict__ a = At + (size_t)(ul / BM) * p_pad * BM + (ul % BM);      // + k * BM
    const uint2* cd = cand + (size_t)ul * C;
    constexpr bool STAGED = MODE != 0;
    constexpr int V = 16 / (int)sizeof(T);                                                         // elements per 16 bytes
    const int RS = p_pad + (MODE == 2 ? V : 1);                                                    // row stride of the staged rows
    T* rows = reinterpret_cast<T*>(smem_raw) + (size_t)warp * (32 * (size_t)(p_pad + V) + p_pad);   // [32][RS]
    T* a_sm = rows + 32 * (size_t)(p_pad + V);                                                     // [p_pad]
    if (STAGED) {
        for (int k = lane; k < p; k += 32) a_sm[k] = a[(size_t)k * BM];
        __syncwarp();
    }
    key_t key[E];
    int it[E];
    int nanflag = 0;
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int idx = e * 32 + lane;
        key[e] = 0;
        it[e] = INT_MAX;
        if (e * 32 < nv) {                       // warp-uniform
            const bool valid = idx < nv;
            const uint2 cde = valid ? cd[idx] : make_uint2(0u, 0u);
            const int item = (int)cde.y;
            if (valid) it[e] = item;
            T acc = (T)0;
            if (STAGED) {
                // candidate j of this round: its factor row, 32 lanes wide, straight into shared memory (cp.async: all
                // 32 rows are in flight at once, no registers in between)
                for (int j = 0; j < 32; j++) {
                    const int item_j = __shfl_sync(FULL, item, j);
                    const T* __restrict__ b = Brow + (size_t)item_j * ldb;
                    T* dst = rows + (size_t)j * RS;
                    if (MODE == 2) { for (int k = lane * V; k < p; k += 32 * V) cp_async_16(dst + k, b + k); }
                    else { for (int k = lane; k < p; k += 32) cp_async_elem(dst + k, b + k); }
                }
                asm volatile("cp.async.wait_all;" ::: "memory");
                __syncwarp();
                const T* mine = rows + (size_t)lane * RS;
                if (MODE == 2) {
#pragma unroll 4
                    for (int k = 0; k < p; k += V) {
                        T av[V], bv[V];
                        lds_vec(a_sm + k, av);
                        lds_vec(mine + k, bv);
#pragma unroll
                        for (int x = 0; x < V; x++) acc = NumTraits<T>::fma(av[x], bv[x], acc);
                    }
                } else {
#pragma unroll 8
                    for (int k = 0; k < p; k++) acc = NumTraits<T>::fma(a_sm[k], mine[k], acc);
                }
                __syncwarp();
            } else if (valid) {
                const T* __restrict__ b = Brow + (size_t)item * ldb;
#pragma unroll 8
                for (int k = 0; k < p; k++) acc = NumTraits<T>::fma(a[(size_t)k * BM], b[k], acc);
            }
            if (valid) {
                if (bias != nullptr) acc += bias[item];
                if (acc != acc) nanflag = 1;
                else key[e] = NumTraits<T>::key(acc);
                if (es.max_ratio_bits != nullptr) {
                    // observed error of the approximate score against the bound the filter used for it (scaled units)
                    const float an = es.anorm[ul], bn = __uint_as_float(*es.maxbn);
                    const float sa = pow2_scale_for(an), sb = pow2_scale_for(bn), ap = an * sa;
                    const float bound = filter_err(__fmul_ru(__fmul_ru(es.c_rel, ap), sb), es.chunk_norm[item >> 5], __fmaf_ru(es.c_abs, ap, es.c_const));
                    // (the candidate carries its lower bound: approximate score = lower bound + bound, up to one rounding)
                    const double diff = fabs((double)__uint_as_float(cde.x) + (double)bound - (double)acc * (double)sa * (double)sb);
                    const float ratio = (float)(diff / (double)bound);
                    if (ratio == ratio && ratio < CUDART_INF_F) atomicMax(es.max_ratio_bits, __float_as_uint(ratio));
                }
            }
        }
    }
    if (__any_sync(FULL, nanflag)) { if (lane == 0) atomicOr(&uflags[user0 + ul], 1); }
    if (noise) {
        // break_ties_with_noise (hpp:531-534, tie_noise.cuh): candidate number ix of the user -- candidates in ascending item
        // order, i.e. item id minus the train items before it -- gets draw ix of mt19937(seed + user).  Only scores the
        // noise can change need their draw (every double score; float scores below 2^-14 in magnitude).
        bool want = false;
        int pos[E];
        const int t0 = trp[user0 + ul], t1 = trp[user0 + ul + 1];
        {
            // validity rule of the noise branch (hpp:524-527): all candidates equal => NaN row.  The filter keeps whatever can
            // reach the K-th best score: if it kept fewer than all candidates some score is lower than the rest; if it kept
            // them all, they are all here.
            key_t kmax = 0, kmin = ~(key_t)0;
            int cntv = 0;
#pragma unroll
            for (int e = 0; e < E; e++)
                if (key[e] != 0) { kmax = key[e] > kmax ? key[e] : kmax; kmin = key[e] < kmin ? key[e] : kmin; cntv++; }
            cntv = __reduce_add_sync(FULL, cntv);
            // warp-wide extremes (64-bit keys for double: reduce through shuffles)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const key_t omax = __shfl_xor_sync(FULL, kmax, o), omin = __shfl_xor_sync(FULL, kmin, o);
                kmax = omax > kmax ? omax : kmax;
                kmin = omin < kmin ? omin : kmin;
            }
            if (cntv == n - (t1 - t0) && cntv > 0 && kmax == kmin && lane == 0) atomicOr(&uflags[user0 + ul], 4);
        }
#pragma unroll
        for (int e = 0; e < E; e++) {
            pos[e] = -1;
            if (key[e] != 0 && TieNoise<T>::can_change(NumTraits<T>::from_orderable((u64)key[e]))) {
                int lo = t0, hi = t1;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (tri[mid] < it[e]) lo = mid + 1; else hi = mid; }
                pos[e] = it[e] - (lo - t0);
                want = true;
            }
        }
        if (__any_sync(FULL, want)) {
            int maxpos = -1;
#pragma unroll
            for (int e = 0; e < E; e++) maxpos = max(maxpos, pos[e]);
            maxpos = __reduce_max_sync(FULL, maxpos);
            unsigned* x = reinterpret_cast<unsigned*>(smem_raw + mt_off) + warp * MT_N;
            mt_seed_warp(x, seed_user0 + (unsigned long long)ul, lane);
            const int nblocks = (int)(((long long)(maxpos + 1) * TieNoise<T>::WORDS + MT_N - 1) / MT_N);
            for (int blk = 0; blk < nblocks; blk++) {
                mt_twist_warp(x, lane);
#pragma unroll
                for (int e = 0; e < E; e++) {
                    if (pos[e] < 0) continue;
                    const long long w = (long long)pos[e] * TieNoise<T>::WORDS - (long long)blk * MT_N;     // first word of the draw, inside this block?
                    if (w >= 0 && w < MT_N) {
                        const unsigned w0 = mt_temper(x[w]);
                        const unsigned w1 = TieNoise<T>::WORDS == 2 ? mt_temper(x[w + 1]) : 0u;
                        const T noisy = NumTraits<T>::from_orderable((u64)key[e]) + TieNoise<T>::draw(w0, w1);
                        key[e] = NumTraits<T>::key(noisy);
                    }
                }
                __syncwarp();
            }
        }
    }
    T* cs = cand_score + (size_t)ul * C;
    int* cio = cand_item + (size_t)ul * C;
    int base;
    if (E > 4 && nv <= 128) base = exact_select<T, E, (E < 4 ? E : 4)>(key, it, K, lane, cs, cio);      // (the filter rarely keeps more: K' ~ 1.2 K)
    else if (E > 8 && nv <= 256) base = exact_select<T, E, (E < 8 ? E : 8)>(key, it, K, lane, cs, cio);
    else base = exact_select<T, E, E>(key, it, K, lane, cs, cio);
    if (lane == 0) cand_count[ul] = base;
}

}  // namespace rmb
