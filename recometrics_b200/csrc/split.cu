// split.cu -- the train/test splitters behind rmb200_split_* (include/recometrics_b200.h).
//
// Stands where /root/reference/src/recometrics.hpp:1015-1505 stands: split_data_selected_users (every row of X split
// into a training and a held-out part), split_data_separate_users (a random sample of eligible users split that way, the
// other users returned untouched) and split_data_joined_users (the same with the other users appended below the training
// rows).
//
// What decides the result is ONE std::mt19937 stream consumed row after row by std::shuffle (hpp:1055-1060), plus one
// shuffle of the user ids (hpp:1223-1226): a row's draws start where the previous row's ended, and how many a row takes
// depends on the rejections of libstdc++'s bounded-integer method.  That replay is sequential by the definition of the
// output; Replay below does it on the host, on index arrays that never leave L1/L2, and emits ONE BYTE per entry
// ("held out" or not).  Everything else happens beside it, on a second host thread that drives the GPU: X goes up, the
// rows a split leaves alone are gathered and come back, and the split rows follow in CHUNKS of rows as the replay
// finishes them -- bytes up, scan, partition, results down -- so that when the replay ends only the last chunk is left.
// The result arrays are allocated and their pages touched (by a few more threads) before either starts.  On large inputs
// the replay itself runs on several threads without changing the stream: see struct Replay.
//
// All work on the matrix itself is on the GPU, phrased per ENTRY rather than per row so that a catalogue's power-law row
// lengths do not matter:
//   * the reference leaves each half of a split row ordered by item id (std::sort, hpp:1064-1066, :1075-1077).  With rows
//     that arrive sorted (what the reference's Python and R fronts guarantee) this is a STABLE PARTITION of the row; and
//     since the held-out entries of rows 0..r-1 fill exactly test_p[r] slots, the stable partition of all rows at once is
//     one global exclusive scan of the bytes: held-out entry j goes to slot scan[j] of the test arrays, any other entry to
//     slot j - scan[j] of the training arrays.  No per-row loop, no row lookup, coalesced reads.
//   * rows that arrive unsorted are first ordered by one segmented radix sort of (item id, position) pairs; rows that the
//     reference copies verbatim (nothing or everything held out, hpp:1043-1054) keep their input order.
//   * the rows of the users a split leaves alone (hpp:1303-1321) and the sub-matrix of the sampled users (hpp:1271-1284)
//     are gathers through a row list; the sub-matrix is never materialised -- the scatter reads X through the list.
#include "../../include/recometrics_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <deque>
#include <locale>
#include <memory>
#include <mutex>
#include <new>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <random>
#include <sstream>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "runtime.h"

namespace {

using clk = std::chrono::steady_clock;
double ms_since(clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); }

// ------------------------------------------------------------------------------------------------------------------
// Host: the replay of the reference's random stream
// ------------------------------------------------------------------------------------------------------------------
// zero-filled bytes that cost nothing until they are written (calloc hands out untouched pages; a std::vector would fault
// and fill all of them up front, on the call's critical path: 2-12 ms for 19 MB)
struct ZeroedBytes {
    uint8_t* p = nullptr;
    size_t n = 0;
    ZeroedBytes() = default;
    ZeroedBytes(const ZeroedBytes&) = delete;
    ZeroedBytes& operator=(const ZeroedBytes&) = delete;
    ~ZeroedBytes() { std::free(p); }
    void reset(size_t count)
    {
        std::free(p);
        n = count;
        p = (uint8_t*)std::calloc(count ? count : 1, 1);
        if (!p) throw std::bad_alloc();
    }
    uint8_t* data() const { return p; }
    size_t size() const { return n; }
};

struct SplitPlan {
    bool whole = true;                 // every row of X is split, in place (split_data_selected_users)
    std::vector<int32_t> sel_rows;     // rows of X that are split, ascending (empty when `whole`)
    std::vector<int32_t> rem_rows;     // the other rows, ascending
    std::vector<int32_t> sel_p;        // [ns+1] the split rows as a matrix of their own (when `whole`: X's own pointer)
    std::vector<int32_t> test_p;       // [ns+1]
    std::vector<int32_t> train_p;      // [ns+1]
    std::vector<int32_t> rem_p;        // [nr+1]
    ZeroedBytes held;                  // [nnz of the split rows] 1 = held out
    std::vector<int32_t> chunk_end;    // row after the last row of each chunk (ascending, last = ns)
    int32_t ns = 0, nr = 0, longest = 0;
};

// The threads of one call wait for each other here.  Blocking waits, not spinning: in a container with a CPU quota a handful of
// spinning threads burns the quota and the kernel then stalls ALL of the call's threads for the rest of the period.
struct Signal {
    std::mutex mu;
    std::condition_variable cv;
    template <class F> void update(F&& change) { { std::lock_guard<std::mutex> lk(mu); change(); } cv.notify_all(); }
    template <class Pred> void wait(Pred&& ready) { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, ready); }
};

// What the replay, the device thread and the page toucher of one call tell each other.
struct Progress {
    std::unique_ptr<std::atomic<int>[]> chunk_done;   // [chunks] set (release: the bytes are visible) when a chunk's bytes are final
    std::atomic<int> stop{0};                         // the device thread failed or the replay threw: the others need not go on
    std::atomic<int> touched{0};                      // the result arrays' pages have been touched: copies into them may start
    Signal sig;
    explicit Progress(size_t chunks) : chunk_done(new std::atomic<int>[chunks])
    {
        for (size_t c = 0; c < chunks; c++) chunk_done[c].store(0);
    }
};

// The replay's scout.  libstdc++'s std::shuffle consumes, for `cnt` elements, a number of raw mt19937 outputs that depends on the
// outputs themselves (the rejection loop of its bounded draw, bits/uniform_int_dist.h _S_nd; two positions per draw while
// cnt*cnt fits 32 bits, bits/stl_algo.h).  skip_row() consumes exactly those outputs WITHOUT shuffling anything: the raw
// outputs generated 624 at a time by the textbook in-place recurrence (the state array is laid out exactly like libstdc++'s, so
// a std::mt19937 can be made from it through the engine's own operator>>), and the draws of a whole row screened at once -- a
// bounded draw of range R can only be rejected when the low 32 bits of x * R fall below R (bits/uniform_int_dist.h), which for
// the ranges of a shuffle happens about once in 10^4 draws; only then are the row's draws walked one by one.  ~1.2 ns per draw
// against ~2.2 for std::mt19937 + the scalar rejection test.
// It is only ever used to run AHEAD of the real thing: usable() compares the generator and the state hand-over with
// std::mt19937 itself before the replay relies on them, and every state it predicts is checked against std::shuffle's own
// generator afterwards.
class RawScout {
    uint32_t x[624];
    uint32_t out[624];
    int p = 624;

    void refill()
    {
        const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, MAG = 0x9908b0dfu;
        for (int k = 0; k < 227; k++) {
            const uint32_t y = (x[k] & UP) | (x[k + 1] & LO);
            x[k] = x[k + 397] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
        }
        for (int k = 227; k < 623; k++) {
            const uint32_t y = (x[k] & UP) | (x[k + 1] & LO);
            x[k] = x[k - 227] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
        }
        const uint32_t y = (x[623] & UP) | (x[0] & LO);
        x[623] = x[396] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
        for (int k = 0; k < 624; k++) {
            uint32_t z = x[k];
            z ^= z >> 11;
            z ^= (z << 7) & 0x9d2c5680u;
            z ^= (z << 15) & 0xefc60000u;
            z ^= z >> 18;
            out[k] = z;
        }
        p = 0;
    }

    void bounded(uint32_t range)
    {
        uint32_t low = next() * range;
        if (low < range) {
            const uint32_t threshold = (uint32_t)(0u - range) % range;
            while (low < threshold) low = next() * range;
        }
    }

public:
    explicit RawScout(uint64_t seed)
    {
        x[0] = (uint32_t)seed;
        for (uint32_t i = 1; i < 624; i++) x[i] = 1812433253u * (x[i - 1] ^ (x[i - 1] >> 30)) + i;
    }

    uint32_t next()
    {
        if (p == 624) refill();
        return out[p++];
    }

    // the raw outputs one std::shuffle of `cnt` elements consumes
    void skip_row(uint32_t cnt)
    {
        if (cnt < 2) return;
        if (0xffffffffull / cnt < cnt) {                     // (rows of 65,536 entries and more: one position per draw)
            for (uint32_t i = 1; i < cnt; i++) bounded(i + 1);
            return;
        }
        uint32_t i = 1;
        if ((cnt & 1u) == 0) { bounded(2); i = 2; }
        uint32_t left = (cnt - i) / 2;                       // draws of two positions each, for elements i, i + 2, ...
        while (left) {
            if (p == 624) refill();
            const uint32_t take = std::min<uint32_t>(left, (uint32_t)(624 - p));
            const uint32_t* o = out + p;
            uint32_t suspect = 0;
            for (uint32_t j = 0; j < take; j++) {
                const uint32_t r = i + 1 + 2 * j, range = r * (r + 1);
                suspect |= (uint32_t)((o[j] * range) < range);
            }
            if (!suspect) p += (int)take;
            else for (uint32_t j = 0; j < take; j++) { const uint32_t r = i + 1 + 2 * j; bounded(r * (r + 1)); }
            i += 2 * take;
            left -= take;
        }
    }

    // a std::mt19937 in exactly this state, through the engine's own textual form (bits/random.tcc: the state words, then the position)
    std::mt19937 engine() const
    {
        std::string text;
        text.reserve(624 * 11 + 8);
        for (int k = 0; k < 624; k++) { text += std::to_string(x[k]); text += ' '; }
        text += std::to_string(p);
        std::istringstream is(text);
        is.imbue(std::locale::classic());     // (whatever the host application did to the global locale)
        std::mt19937 g;
        is >> g;
        return g;
    }

    // does this restatement walk in step with the std::mt19937 of the library the product is linked against?
    static bool usable(uint64_t seed)
    {
        RawScout s(seed);
        std::mt19937 ref(seed);
        if (!(s.engine() == ref)) return false;
        for (int k = 0; k < 1500; k++) if (s.next() != (uint32_t)ref()) return false;
        return s.engine() == ref;
    }
};

// /root/reference/src/recometrics.hpp:1041-1060 without the data movement: for rows with something on both sides, the
// positions std::shuffle puts first.  prog.chunk_done[c] is set when chunk c's bytes are final.
//
// sequential(): the reference's loop, one generator, row after row.
// parallel():   the same stream, several threads.  One thread (the scout) runs ahead with RawScout::skip_row() and leaves a
//               copy of the generator at every chunk boundary; the others pick chunks, start from the scout's copy, do the real
//               std::shuffle of every row -- and publish a chunk only if their generator ends in exactly the state the scout
//               left for the next chunk.  A mismatch (a libstdc++ whose shuffle draws differently) costs time, never the
//               result: the chunk that disagreed is kept (its start was verified, its end state is std::shuffle's own) and the
//               rest is redone sequentially from there.
struct Replay {
    SplitPlan& P;
    uint64_t seed;
    Progress& prog;
    int fault_chunk = -1;        // (tests) the scout miscounts in this chunk

    int32_t chunk_begin(size_t c) const { return c ? P.chunk_end[c - 1] : 0; }

    void rows(std::mt19937& rng, std::vector<int32_t>& order, int32_t r0, int32_t r1)
    {
        for (int32_t r = r0; r < r1; r++) {
            const int32_t cnt = P.sel_p[r + 1] - P.sel_p[r];
            const int32_t out = P.test_p[r + 1] - P.test_p[r];
            if (!cnt || !out) continue;
            uint8_t* mark = P.held.data() + P.sel_p[r];
            if (out == cnt) { std::memset(mark, 1, (size_t)cnt); continue; }
            std::iota(order.begin(), order.begin() + cnt, (int32_t)0);
            std::shuffle(order.begin(), order.begin() + cnt, rng);
            for (int32_t j = 0; j < out; j++) mark[order[j]] = 1;
        }
    }

    void sequential(size_t from_chunk, std::mt19937 rng)
    {
        std::vector<int32_t> order((size_t)P.longest);
        for (size_t c = from_chunk; c < P.chunk_end.size(); c++) {
            if (prog.stop.load(std::memory_order_relaxed)) return;
            rows(rng, order, chunk_begin(c), P.chunk_end[c]);
            prog.sig.update([&]() { prog.chunk_done[c].store(1, std::memory_order_release); });
        }
    }

    void parallel(int workers)
    {
        const size_t nc = P.chunk_end.size();
        std::vector<std::mt19937> start(nc + 1);
        std::atomic<size_t> scouted{0};            // start[0 .. scouted) are known
        std::atomic<size_t> next{0};
        std::atomic<size_t> first_bad{nc};         // lowest chunk whose end state disagreed with the scout
        const std::atomic<int>& stop = prog.stop;
        Signal& sig = prog.sig;
        auto give_up = [&]() { return stop.load(std::memory_order_relaxed) || first_bad.load(std::memory_order_relaxed) < nc; };
        // a chunk ABOVE one that disagreed started from a state nobody vouches for; the chunks below it still have to be finished
        auto doomed = [&](size_t c) { return stop.load(std::memory_order_relaxed) || first_bad.load(std::memory_order_relaxed) < c; };
        auto work = [&]() {
            std::vector<int32_t> order((size_t)P.longest);
            for (size_t c = next.fetch_add(1); c < nc; c = next.fetch_add(1)) {
                sig.wait([&]() { return scouted.load(std::memory_order_acquire) > c || doomed(c); });
                if (doomed(c)) return;
                std::mt19937 rng = start[c];
                rows(rng, order, chunk_begin(c), P.chunk_end[c]);
                // (the scout stops after a disagreement at chunk b, but it had passed b + 1 by then: no chunk below b waits in vain)
                sig.wait([&]() { return scouted.load(std::memory_order_acquire) > c + 1 || doomed(c); });
                if (doomed(c)) return;
                if (rng == start[c + 1]) { sig.update([&]() { prog.chunk_done[c].store(1, std::memory_order_release); }); continue; }
                sig.update([&]() {
                    if (c < first_bad.load()) { first_bad.store(c); start[c + 1] = rng; }   // (only the lowest disagreeing chunk's state is used below)
                });
                return;
            }
        };
        std::vector<std::thread> pool;
        struct JoinAll { std::vector<std::thread>& v; ~JoinAll() { for (auto& t : v) if (t.joinable()) t.join(); } } join_all{pool};
        for (int w = 0; w < workers; w++) pool.emplace_back(work);
        {   // the scout
            RawScout raw(seed);
            start[0] = std::mt19937(seed);
            sig.update([&]() { scouted.store(1, std::memory_order_release); });
            for (size_t c = 0; c < nc && !give_up(); c++) {
                for (int32_t r = chunk_begin(c); r < P.chunk_end[c]; r++) {
                    const int32_t cnt = P.sel_p[r + 1] - P.sel_p[r];
                    const int32_t out = P.test_p[r + 1] - P.test_p[r];
                    if (out <= 0 || out >= cnt) continue;
                    raw.skip_row((uint32_t)cnt);
                }
                if ((int)c == fault_chunk) raw.next();
                const std::mt19937 g = raw.engine();
                // (a worker that disagreed with this scout may already have put std::shuffle's own state into start[c + 1]: the
                //  scout stops at the next give_up(); what it writes after a disagreement is never used)
                sig.update([&]() { if (first_bad.load() >= nc) { start[c + 1] = g; } scouted.store(c + 2, std::memory_order_release); });
            }
        }
        work();                                    // the scout's thread joins the others
        for (auto& t : pool) t.join();
        const size_t bad = first_bad.load();
        if (bad >= nc || stop.load()) return;
        // chunks 0 .. bad-1 were verified and published; chunk `bad` started from a verified state and start[bad + 1] is where
        // std::shuffle itself left the generator.  Anything written further on started from the scout's wrong guess.
        for (size_t c = bad + 1; c < nc; c++) prog.chunk_done[c].store(0, std::memory_order_relaxed);
        if (bad + 1 < nc) std::memset(P.held.data() + P.sel_p[P.chunk_end[bad]], 0, (size_t)(P.sel_p[P.ns] - P.sel_p[P.chunk_end[bad]]));
        sig.update([&]() { prog.chunk_done[bad].store(1, std::memory_order_release); });
        sequential(bad + 1, start[bad + 1]);
    }

    // in parallel only where the scout is known to walk in step with this library's std::mt19937 (RawScout::usable)
    void run()
    {
        int workers = (int)std::min(4u, std::max(1u, std::thread::hardware_concurrency() / 4));
        if (const char* env = std::getenv("RMB200_SPLIT_THREADS")) workers = std::max(0, std::atoi(env));
        if (const char* env = std::getenv("RMB200_SPLIT_SCOUT_FAULT")) fault_chunk = std::atoi(env);
        if (workers >= 1 && P.chunk_end.size() >= 4 && RawScout::usable(seed)) parallel(workers);
        else sequential(0, std::mt19937(seed));
    }
};

// /root/reference/src/recometrics.hpp:1223-1269: which users are split.  Returns the reference's error text or nullptr.
const char* pick_users(const int32_t* Xp, int32_t m, int32_t n, int32_t n_users_test, double test_fraction,
                       bool consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, uint64_t seed, SplitPlan& P)
{
    if (n_users_test > m) return "Target number of test users is larger than available users.\n";
    if (min_items_pool >= n) return "Selected minimum number of items is larger than total number of items.\n";
    std::vector<int32_t> ids((size_t)m);
    std::iota(ids.begin(), ids.end(), (int32_t)0);
    std::mt19937 rng(seed);
    std::shuffle(ids.begin(), ids.end(), rng);

    auto eligible = [&](int32_t u) {
        const int32_t cnt = Xp[u + 1] - Xp[u];
        if (!cnt) return false;
        const int32_t out = (int32_t)std::round(cnt * test_fraction);
        if (out < min_pos_test) return false;
        if (n - (cnt - out) < min_items_pool) return false;
        if (!consider_cold_start && out == cnt) return false;
        return cnt + 1 < n;
    };
    int32_t taken = 0, end = m;
    do {   // (a do-while in the reference as well: the first candidate is looked at even for n_users_test = 0)
        if (eligible(ids[taken])) taken++;
        else std::swap(ids[taken], ids[--end]);
    } while (taken < n_users_test && taken < end);
    if (!taken) return "No users satisfy criteria for test inclusion.\n";

    std::sort(ids.begin(), ids.begin() + taken);
    std::sort(ids.begin() + taken, ids.end());
    P.whole = false;
    P.sel_rows.assign(ids.begin(), ids.begin() + taken);
    P.rem_rows.assign(ids.begin() + taken, ids.end());
    P.nr = m - taken;
    P.rem_p.resize((size_t)P.nr + 1);
    P.rem_p[0] = 0;
    for (int32_t r = 0; r < P.nr; r++) P.rem_p[r + 1] = P.rem_p[r] + (Xp[P.rem_rows[r] + 1] - Xp[P.rem_rows[r]]);
    return nullptr;
}

// Everything the result's shape depends on: which rows are split (a sample of the users when `sample_users`, else every row of
// X), how many entries of each are held out (/root/reference/src/recometrics.hpp:1037-1040), the chunks the device thread works
// on, and the held-out bytes, all 0.  Returns the reference's error text or nullptr.
const char* plan_split(const int32_t* Xp, int32_t m, int32_t n, bool sample_users, int32_t n_users_test, double test_fraction,
                       bool consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, uint64_t seed, SplitPlan& P)
{
    if (sample_users)
        if (const char* refusal = pick_users(Xp, m, n, n_users_test, test_fraction, consider_cold_start, min_items_pool,
                                             min_pos_test, seed, P))
            return refusal;
    const int32_t ns = P.whole ? m : (int32_t)P.sel_rows.size();
    P.ns = ns;
    P.sel_p.resize((size_t)ns + 1);
    P.test_p.resize((size_t)ns + 1);
    P.train_p.resize((size_t)ns + 1);
    P.sel_p[0] = P.test_p[0] = P.train_p[0] = 0;
    P.longest = 0;
    for (int32_t r = 0; r < ns; r++) {
        const int32_t u = P.whole ? r : P.sel_rows[r];
        const int32_t cnt = Xp[u + 1] - Xp[u];
        P.sel_p[r + 1] = P.sel_p[r] + cnt;
        P.test_p[r + 1] = P.test_p[r] + (int32_t)std::round(cnt * test_fraction);
        P.train_p[r + 1] = P.sel_p[r + 1] - P.test_p[r + 1];
        P.longest = std::max(P.longest, cnt);
    }
    // chunks of whole rows, about a sixteenth of the entries each but not below a million: what the device thread works on
    const int64_t total = P.sel_p[ns];
    int64_t floor_entries = 1 << 20;
    if (const char* env = std::getenv("RMB200_SPLIT_CHUNK")) { const long long v = std::atoll(env); if (v >= 1) floor_entries = v; }   // (tests)
    const int64_t per_chunk = std::max<int64_t>(floor_entries, (total + 15) / 16);
    P.chunk_end.clear();
    int64_t next = per_chunk;
    for (int32_t r = 0; r < ns; r++)
        if (P.sel_p[r + 1] >= next && r + 1 < ns) { P.chunk_end.push_back(r + 1); next = P.sel_p[r + 1] + per_chunk; }
    P.chunk_end.push_back(ns);
    P.held.reset((size_t)total);
    return nullptr;
}

// ------------------------------------------------------------------------------------------------------------------
// Device
// ------------------------------------------------------------------------------------------------------------------
constexpr int TPB = 256;

// last row r with ptr[r] <= j (rows may be empty)
__device__ __forceinline__ int row_of(const int* __restrict__ ptr, int rows, int j)
{
    int lo = 0, hi = rows;          // invariant: ptr[lo] <= j < ptr[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(ptr + mid) <= j) lo = mid; else hi = mid;
    }
    return lo;
}

struct SplitView {
    const int* Xp; const int* Xi;
    const int* sel_rows;            // nullptr: the split rows are X's rows
    const int* sel_p; const int* test_p;
    int ns;
    int j0, j1;                     // the entries (of the split rows' own matrix) this launch works on
};

// entry of X behind position j of the split rows' own matrix
__device__ __forceinline__ int source_entry(const SplitView& V, int r, int j)
{
    return V.sel_rows ? __ldg(V.Xp + __ldg(V.sel_rows + r)) + (j - __ldg(V.sel_p + r)) : j;
}

// rows the reference reorders: something held out AND something kept (hpp:1043-1054 copies the others verbatim)
__device__ __forceinline__ bool row_is_split(const SplitView& V, int r)
{
    const int cnt = __ldg(V.sel_p + r + 1) - __ldg(V.sel_p + r);
    const int out = __ldg(V.test_p + r + 1) - __ldg(V.test_p + r);
    return out > 0 && out < cnt;
}

#define FOR_EACH_ENTRY(jj, first, last)                                                                                        \
    for (long long jj = (long long)(first) + (long long)blockIdx.x * TPB + threadIdx.x; jj < (long long)(last);                \
         jj += (long long)gridDim.x * TPB)

// 1 into *unsorted when a split row has a descending pair of item ids
__global__ void __launch_bounds__(TPB) check_sorted_kernel(SplitView V, int* __restrict__ unsorted)
{
    FOR_EACH_ENTRY(jj, V.j0, V.j1) {
        const int j = (int)jj;
        const int r = row_of(V.sel_p, V.ns, j);
        if (j == __ldg(V.sel_p + r) || !row_is_split(V, r)) continue;
        const int e = source_entry(V, r, j);
        if (__ldg(V.Xi + e) < __ldg(V.Xi + e - 1)) *unsorted = 1;
    }
}

// sort input of the unsorted case: key = item id, value = position in the split rows' matrix
__global__ void __launch_bounds__(TPB) sort_input_kernel(SplitView V, int* __restrict__ keys, int* __restrict__ vals)
{
    FOR_EACH_ENTRY(jj, V.j0, V.j1) {
        const int j = (int)jj;
        const int r = row_of(V.sel_p, V.ns, j);
        keys[j] = __ldg(V.Xi + source_entry(V, r, j));
        vals[j] = j;
    }
}

// position j of the ORDERED split rows -> its position before ordering
__device__ __forceinline__ int unordered_pos(const SplitView& V, const int* __restrict__ perm, int j, int* row)
{
    if (!perm && !V.sel_rows) { *row = -1; return j; }
    const int r = row_of(V.sel_p, V.ns, j);
    *row = r;
    return (perm && row_is_split(V, r)) ? __ldg(perm + j) : j;
}

// the held-out bytes in the order the entries will be written (only needed when rows were reordered)
__global__ void __launch_bounds__(TPB) ordered_flags_kernel(SplitView V, const int* __restrict__ perm,
                                                            const uint8_t* __restrict__ held, uint8_t* __restrict__ flags)
{
    FOR_EACH_ENTRY(jj, V.j0, V.j1) {
        const int j = (int)jj;
        int r;
        flags[j] = held[unordered_pos(V, perm, j, &r)];
    }
}

// the stable partition of every row at once: base + scan[j] = held-out entries before j (scan restarts at V.j0, where
// `base` = test_p[first row of the chunk] of them came before)
template <typename T>
__global__ void __launch_bounds__(TPB) partition_kernel(SplitView V, const T* __restrict__ Xv, const int* __restrict__ perm,
                                                        const uint8_t* __restrict__ flags, const int* __restrict__ scan, int base,
                                                        int* __restrict__ train_i, T* __restrict__ train_v,
                                                        int* __restrict__ test_i, T* __restrict__ test_v)
{
    FOR_EACH_ENTRY(jj, V.j0, V.j1) {
        const int j = (int)jj;
        int r;
        const int s = unordered_pos(V, perm, j, &r);
        const int e = (r >= 0) ? source_entry(V, r, s) : s;
        const int item = __ldg(V.Xi + e);
        const T val = __ldg(Xv + e);
        const int before = base + scan[j];
        if (flags[j]) { test_i[before] = item; test_v[before] = val; }
        else { train_i[j - before] = item; train_v[j - before] = val; }
    }
}

// rows of X listed in `rows`, copied one below the other (hpp:1303-1321)
template <typename T>
__global__ void __launch_bounds__(TPB) gather_rows_kernel(const int* __restrict__ Xp, const int* __restrict__ Xi,
                                                          const T* __restrict__ Xv, const int* __restrict__ rows,
                                                          const int* __restrict__ out_p, int n_rows, int total,
                                                          int* __restrict__ out_i, T* __restrict__ out_v)
{
    FOR_EACH_ENTRY(jj, 0, total) {
        const int j = (int)jj;
        const int r = row_of(out_p, n_rows, j);
        const int e = __ldg(Xp + __ldg(rows + r)) + (j - __ldg(out_p + r));
        out_i[j] = __ldg(Xi + e);
        out_v[j] = __ldg(Xv + e);
    }
}

struct ByteToInt {
    __host__ __device__ __forceinline__ int operator()(const uint8_t& b) const { return (int)b; }
};

// one block per call, carved into the call's arrays (256-byte aligned)
struct Slot { void* p = nullptr; template <typename U> U* as() const { return (U*)p; } };
struct Carver {
    size_t total = 0;
    char* base = nullptr;
    size_t reserve(size_t bytes) { const size_t at = total; total += (bytes + 255) & ~(size_t)255; return at; }
    template <typename U> U* at(size_t offset) const { return (U*)(base + offset); }
};

// what rmb200_split_t::owner points to
struct SplitOwner { std::vector<void*> blocks; std::vector<size_t> sizes; std::vector<char> device_filled; };

// device_filled: the block's content comes from the GPU (indices, values) -- the host writes nothing into it itself
void* host_block(SplitOwner* own, size_t bytes, bool device_filled = false)
{
    void* p = std::malloc(bytes ? bytes : 1);
    if (p) { own->blocks.push_back(p); own->sizes.push_back(bytes); own->device_filled.push_back(device_filled ? 1 : 0); }
    return p;
}

// first touch of the result's index / value arrays (the ones the GPU fills), spread over a few threads (a fresh 150 MB block costs tens of milliseconds of page
// faults when the device-to-host copy has to take them one by one)
void touch_pages(const SplitOwner* own)
{
    const size_t page = 4096, slice = (size_t)8 << 20;
    std::vector<std::pair<char*, size_t>> work;
    for (size_t b = 0; b < own->blocks.size(); b++)
        for (size_t off = 0; own->device_filled[b] && off < own->sizes[b]; off += slice)
            work.emplace_back((char*)own->blocks[b] + off, std::min(slice, own->sizes[b] - off));
    std::atomic<size_t> next{0};
    auto run = [&]() {
        for (size_t w = next.fetch_add(1); w < work.size(); w = next.fetch_add(1))
            for (size_t off = 0; off < work[w].second; off += page) work[w].first[off] = 0;
    };
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const int nt = (int)std::min<size_t>(std::min<unsigned>(4, hw), work.size());
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; t++) pool.emplace_back(run);
    run();
    for (auto& t : pool) t.join();
}

int fail(int code, const char* what, const char* detail = nullptr)
{
    rmb::set_err(what, detail);
    return code;
}

enum SplitKind { SPLIT_WHOLE = 0, SPLIT_SEPARATE = 1, SPLIT_JOINED = 2 };

// Result pieces on their way back to the host: a few threads, each with a stream of its own, copy finished pieces into the
// (pageable, already touched) result arrays while the device thread goes on with the next chunk.  Two copies in flight also
// means two host threads doing the driver's staging memcpy: ~2x the 12 GB/s of one blocking copy after the other.
struct Downloads {
    struct Piece { void* dst; const void* src; size_t bytes; };
    std::mutex mu;
    std::condition_variable cv;
    std::deque<Piece> queue;
    bool closing = false;
    cudaError_t err = cudaSuccess;
    double copy_ms = 0.0;              // summed over the threads
    std::vector<std::thread> threads;

    void start(int device, int n, Progress& prog)
    {
        for (int t = 0; t < n; t++)
            threads.emplace_back([this, device, &prog]() {
                cudaStream_t st = nullptr;
                cudaError_t e = cudaSetDevice(device);
                if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
                prog.sig.wait([&]() { return prog.touched.load(std::memory_order_acquire) != 0; });
                double ms = 0.0;
                for (;;) {
                    Piece p;
                    {
                        std::unique_lock<std::mutex> lk(mu);
                        cv.wait(lk, [&]() { return closing || !queue.empty(); });
                        if (queue.empty()) break;
                        p = queue.front();
                        queue.pop_front();
                    }
                    if (e != cudaSuccess) continue;            // (drain the queue; the error is reported at finish())
                    const auto t0 = clk::now();
                    e = cudaMemcpyAsync(p.dst, p.src, p.bytes, cudaMemcpyDeviceToHost, st);
                    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
                    ms += ms_since(t0);
                }
                if (st) cudaStreamDestroy(st);
                std::lock_guard<std::mutex> lk(mu);
                copy_ms += ms;
                if (e != cudaSuccess && err == cudaSuccess) err = e;
            });
    }
    void push(void* dst, const void* src, size_t bytes)
    {
        if (!bytes) return;
        { std::lock_guard<std::mutex> lk(mu); queue.push_back(Piece{dst, src, bytes}); }
        cv.notify_one();
    }
    cudaError_t finish()
    {
        { std::lock_guard<std::mutex> lk(mu); closing = true; }
        cv.notify_all();
        for (auto& t : threads) if (t.joinable()) t.join();
        threads.clear();
        return err;
    }
    ~Downloads() { finish(); }
};

struct Stream { cudaStream_t s = nullptr; ~Stream() { if (s) cudaStreamDestroy(s); } };
struct Event { cudaEvent_t e = nullptr; ~Event() { if (e) cudaEventDestroy(e); } };

// The device side of one call, run on its own host thread: upload(), order_unsorted_rows(), gather_untouched_rows() and
// partition_chunks(), in that order, sharing what they set up through the members below.  A step that fails records the
// error, sets prog.stop and returns false.
#define JOB_CUDA(call) do { if (bad((call), #call)) return false; } while (0)
template <typename T>
struct DeviceJob {
    SplitKind kind;
    int device;
    const int32_t *Xp, *Xi; const T* Xv;
    int32_t m; int64_t nnz;
    const SplitPlan& Q;
    rmb200_split_t* out;
    Progress& prog;
    // results
    int status = RMB200_OK;
    std::string what, detail;
    double h2d_ms = 0, d2h_ms = 0, kernel_ms = 0;
    int64_t launches = 0, h2d_bytes = 0, d2h_bytes = 0;
    int sorted_on_device = 0;
    // shared by the steps
    int32_t ns = 0, nr = 0;
    int64_t sel_nnz = 0, test_nnz = 0, rem_nnz = 0, kept_nnz = 0;
    Stream stream;
    Event ev0, ev1;
    cudaStream_t st = nullptr;
    int nsm = 148;
    size_t scan_bytes = 0;
    rmb::DevBuf block;
    Slot dXp, dXi, dXv, d_selrows, d_selp, d_testp, d_remrows, d_remp, d_held, d_scan, d_tri, d_trv, d_tei, d_tev, d_unsorted,
         d_scan_temp, d_rei, d_rev;
    rmb::DevBuf d_keys0, d_keys1, d_vals0, d_perm, d_sort_temp, d_flags;     // (the rare unsorted input: blocks of their own)
    const int* perm = nullptr;
    SplitView V;
    Downloads downloads;

    bool bad(cudaError_t e, const char* where)
    {
        if (e == cudaSuccess) return false;
        cudaGetLastError();
        status = (e == cudaErrorMemoryAllocation) ? RMB200_ERR_OOM : RMB200_ERR_CUDA;
        what = where;
        detail = cudaGetErrorString(e);
        prog.sig.update([&]() { prog.stop.store(1); });
        return true;
    }

    cudaError_t up(void* dst, const void* src, size_t bytes)
    {
        h2d_bytes += (int64_t)bytes;
        if (!bytes) return cudaSuccess;
        return rmb::upload_bytes_pageable(dst, src, bytes, st, 2);
    }

    cudaError_t down(void* dst, const void* src, size_t bytes)      // (pageable destination: returns when the bytes are there)
    {
        if (!bytes) return cudaSuccess;
        prog.sig.wait([&]() { return prog.touched.load(std::memory_order_acquire) != 0; });
        const auto t0 = clk::now();
        const cudaError_t e = rmb::download_bytes_pageable(dst, src, bytes, st, 2);
        d2h_ms += ms_since(t0);
        d2h_bytes += (int64_t)bytes;
        return e;
    }

    cudaError_t down_later(void* dst, const void* src, size_t bytes)      // (on the copy threads, while this thread goes on)
    {
        d2h_bytes += (int64_t)bytes;
        downloads.push(dst, src, bytes);
        return cudaSuccess;
    }

    cudaError_t kernels_begin() { return cudaEventRecord(ev0.e, st); }

    cudaError_t kernels_end()
    {
        float span = 0.f;
        cudaError_t e = cudaEventRecord(ev1.e, st);
        if (e == cudaSuccess) e = cudaEventSynchronize(ev1.e);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&span, ev0.e, ev1.e);
        if (e == cudaSuccess) kernel_ms += span;
        return e;
    }

    int grid_for(int64_t work) const { return (int)std::max<int64_t>(1, std::min<int64_t>((work + TPB - 1) / TPB, (int64_t)nsm * 16)); }

    // The stream, one device block for the call, X and the plan's index arrays up.  The block comes from the library's workspace
    // cache: cudaMalloc / cudaFree of a call's ~600 MB cost 10-200 ms on a busy box, more than the rest of the call.
    bool upload()
    {
        ns = Q.ns; nr = Q.nr;
        sel_nnz = Q.sel_p[ns]; test_nnz = Q.test_p[ns]; rem_nnz = nr ? Q.rem_p[nr] : 0;
        kept_nnz = sel_nnz - test_nnz;
        const int64_t train_nnz = kept_nnz + (kind == SPLIT_JOINED ? rem_nnz : 0);
        JOB_CUDA(cudaSetDevice(device));
        JOB_CUDA(cudaStreamCreateWithFlags(&stream.s, cudaStreamNonBlocking));
        JOB_CUDA(cudaEventCreate(&ev0.e));
        JOB_CUDA(cudaEventCreate(&ev1.e));
        st = stream.s;

        const auto t_up = clk::now();
        int64_t longest_chunk = 0;
        for (size_t c = 0, rb = 0; c < Q.chunk_end.size(); rb = (size_t)Q.chunk_end[c++])
            longest_chunk = std::max<int64_t>(longest_chunk, Q.sel_p[Q.chunk_end[c]] - Q.sel_p[rb]);
        if (longest_chunk) {
            auto probe = thrust::make_transform_iterator((const uint8_t*)nullptr, ByteToInt());
            JOB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, probe, (int*)nullptr, (int)longest_chunk, st));
        }
        const bool own_rem = (kind == SPLIT_SEPARATE) && rem_nnz;
        const std::pair<Slot*, size_t> layout[] = {
            {&dXp, sizeof(int32_t) * ((size_t)m + 1)}, {&dXi, sizeof(int32_t) * (size_t)nnz}, {&dXv, sizeof(T) * (size_t)nnz},
            {&d_selrows, Q.whole ? 0 : sizeof(int32_t) * (size_t)ns}, {&d_selp, Q.whole ? 0 : sizeof(int32_t) * ((size_t)ns + 1)},
            {&d_testp, sizeof(int32_t) * ((size_t)ns + 1)}, {&d_remrows, sizeof(int32_t) * (size_t)nr},
            {&d_remp, nr ? sizeof(int32_t) * ((size_t)nr + 1) : 0}, {&d_held, (size_t)sel_nnz}, {&d_scan, sizeof(int32_t) * (size_t)sel_nnz},
            {&d_tri, sizeof(int32_t) * (size_t)train_nnz}, {&d_trv, sizeof(T) * (size_t)train_nnz},
            {&d_tei, sizeof(int32_t) * (size_t)test_nnz}, {&d_tev, sizeof(T) * (size_t)test_nnz}, {&d_unsorted, sizeof(int)},
            {&d_scan_temp, scan_bytes}, {&d_rei, own_rem ? sizeof(int32_t) * (size_t)rem_nnz : 0}, {&d_rev, own_rem ? sizeof(T) * (size_t)rem_nnz : 0}};
        Carver carve;
        size_t offsets[sizeof(layout) / sizeof(layout[0])];
        for (size_t k = 0; k < sizeof(layout) / sizeof(layout[0]); k++) offsets[k] = carve.reserve(layout[k].second);
        JOB_CUDA(block.alloc(carve.total));
        carve.base = block.as<char>();
        for (size_t k = 0; k < sizeof(layout) / sizeof(layout[0]); k++) layout[k].first->p = carve.at<char>(offsets[k]);
        JOB_CUDA(up(dXp.p, Xp, sizeof(int32_t) * ((size_t)m + 1)));
        JOB_CUDA(up(dXi.p, Xi, sizeof(int32_t) * (size_t)nnz));
        JOB_CUDA(up(dXv.p, Xv, sizeof(T) * (size_t)nnz));
        if (!Q.whole) {
            JOB_CUDA(up(d_selrows.p, Q.sel_rows.data(), sizeof(int32_t) * (size_t)ns));
            JOB_CUDA(up(d_selp.p, Q.sel_p.data(), sizeof(int32_t) * ((size_t)ns + 1)));
            if (nr) {
                JOB_CUDA(up(d_remrows.p, Q.rem_rows.data(), sizeof(int32_t) * (size_t)nr));
                JOB_CUDA(up(d_remp.p, Q.rem_p.data(), sizeof(int32_t) * ((size_t)nr + 1)));
            }
        }
        JOB_CUDA(up(d_testp.p, Q.test_p.data(), sizeof(int32_t) * ((size_t)ns + 1)));
        JOB_CUDA(cudaMemsetAsync(d_unsorted.p, 0, sizeof(int), st));
        JOB_CUDA(cudaStreamSynchronize(st));
        h2d_ms = ms_since(t_up);

        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device);
        V.Xp = dXp.as<int>(); V.Xi = dXi.as<int>();
        V.sel_rows = Q.whole ? nullptr : d_selrows.as<int>();
        V.sel_p = Q.whole ? dXp.as<int>() : d_selp.as<int>();
        V.test_p = d_testp.as<int>();
        V.ns = ns; V.j0 = 0; V.j1 = (int)sel_nnz;
        return true;
    }

    // Does not wait for the replay: check_sorted_kernel, and when a split row is out of order, the segmented sort of every split
    // row's (item id, position) pairs into `perm`.
    bool order_unsorted_rows()
    {
        if (!sel_nnz) return true;
        JOB_CUDA(kernels_begin());
        check_sorted_kernel<<<grid_for(sel_nnz), TPB, 0, st>>>(V, d_unsorted.as<int>());
        launches++;
        JOB_CUDA(kernels_end());
        int unsorted = 0;
        JOB_CUDA(cudaMemcpyAsync(&unsorted, d_unsorted.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        JOB_CUDA(cudaStreamSynchronize(st));
        if (!unsorted) return true;
        sorted_on_device = 1;
        JOB_CUDA(d_keys0.alloc(sizeof(int) * (size_t)sel_nnz));
        JOB_CUDA(d_keys1.alloc(sizeof(int) * (size_t)sel_nnz));
        JOB_CUDA(d_vals0.alloc(sizeof(int) * (size_t)sel_nnz));
        JOB_CUDA(d_perm.alloc(sizeof(int) * (size_t)sel_nnz));
        JOB_CUDA(d_flags.alloc((size_t)sel_nnz));
        size_t temp_bytes = 0;
        JOB_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(nullptr, temp_bytes, (const int*)d_keys0.as<int>(), d_keys1.as<int>(),
                                                          (const int*)d_vals0.as<int>(), d_perm.as<int>(), (int)sel_nnz, ns,
                                                          V.sel_p, V.sel_p + 1, 0, 32, st));
        JOB_CUDA(d_sort_temp.alloc(temp_bytes));
        JOB_CUDA(kernels_begin());
        sort_input_kernel<<<grid_for(sel_nnz), TPB, 0, st>>>(V, d_keys0.as<int>(), d_vals0.as<int>());
        JOB_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(d_sort_temp.p, temp_bytes, (const int*)d_keys0.as<int>(), d_keys1.as<int>(),
                                                          (const int*)d_vals0.as<int>(), d_perm.as<int>(), (int)sel_nnz, ns,
                                                          V.sel_p, V.sel_p + 1, 0, 32, st));
        launches += 3;     // (cub's segmented sort: at least its partition + sort kernels)
        JOB_CUDA(kernels_end());
        perm = d_perm.as<int>();
        return true;
    }

    // Does not wait for the replay either: the rows the split leaves alone, gathered below the training rows (joined) or into
    // a matrix of their own (separated), and brought down.
    bool gather_untouched_rows()
    {
        if (!rem_nnz) return true;
        int* dst_i; T* dst_v;
        if (kind == SPLIT_JOINED) { dst_i = d_tri.as<int>() + kept_nnz; dst_v = d_trv.as<T>() + kept_nnz; }
        else { dst_i = d_rei.as<int>(); dst_v = d_rev.as<T>(); }
        JOB_CUDA(kernels_begin());
        gather_rows_kernel<T><<<grid_for(rem_nnz), TPB, 0, st>>>(dXp.as<int>(), dXi.as<int>(), dXv.as<T>(), d_remrows.as<int>(),
                                                                  d_remp.as<int>(), nr, (int)rem_nnz, dst_i, dst_v);
        launches++;
        JOB_CUDA(kernels_end());
        rmb200_csr_t& M = (kind == SPLIT_JOINED) ? out->train : out->rem;
        const int64_t at = (kind == SPLIT_JOINED) ? kept_nnz : 0;
        JOB_CUDA(down(M.indices + at, dst_i, sizeof(int32_t) * (size_t)rem_nnz));
        JOB_CUDA(down((T*)M.values + at, dst_v, sizeof(T) * (size_t)rem_nnz));
        return true;
    }

    // The split rows, chunk by chunk behind the replay: the chunk's bytes up, scan, partition, and its pieces to the copy threads.
    bool partition_chunks()
    {
        downloads.start(device, 2, prog);
        int32_t r0 = 0;
        for (size_t c = 0; c < Q.chunk_end.size(); c++) {
            const int32_t r1 = Q.chunk_end[c];
            prog.sig.wait([&]() { return prog.chunk_done[c].load(std::memory_order_acquire) != 0 || prog.stop.load() != 0; });
            if (prog.stop.load()) return false;
            const int j0 = Q.sel_p[r0], j1 = Q.sel_p[r1];
            const int t0 = Q.test_p[r0], t1 = Q.test_p[r1];
            if (j1 > j0) {
                JOB_CUDA(up(d_held.as<uint8_t>() + j0, Q.held.data() + j0, (size_t)(j1 - j0)));
                V.j0 = j0; V.j1 = j1;
                JOB_CUDA(kernels_begin());
                const uint8_t* flags = d_held.as<uint8_t>();
                if (perm) {
                    ordered_flags_kernel<<<grid_for(j1 - j0), TPB, 0, st>>>(V, perm, d_held.as<uint8_t>(), d_flags.as<uint8_t>());
                    launches++;
                    flags = d_flags.as<uint8_t>();
                }
                auto as_int = thrust::make_transform_iterator(flags + j0, ByteToInt());
                JOB_CUDA(cub::DeviceScan::ExclusiveSum(d_scan_temp.p, scan_bytes, as_int, d_scan.as<int>() + j0, j1 - j0, st));
                partition_kernel<T><<<grid_for(j1 - j0), TPB, 0, st>>>(V, dXv.as<T>(), perm, flags, d_scan.as<int>(), t0,
                                                                        d_tri.as<int>(), d_trv.as<T>(), d_tei.as<int>(), d_tev.as<T>());
                launches += 3;     // (cub's scan: two kernels)
                JOB_CUDA(cudaGetLastError());
                JOB_CUDA(kernels_end());
                const int k0 = j0 - t0, k1 = j1 - t1;      // the chunk's training entries
                // (kernels_end() has waited for the chunk's kernels: its pieces may leave on the copy threads' own streams)
                JOB_CUDA(down_later(out->train.indices + k0, d_tri.as<int>() + k0, sizeof(int32_t) * (size_t)(k1 - k0)));
                JOB_CUDA(down_later((T*)out->train.values + k0, d_trv.as<T>() + k0, sizeof(T) * (size_t)(k1 - k0)));
                JOB_CUDA(down_later(out->test.indices + t0, d_tei.as<int>() + t0, sizeof(int32_t) * (size_t)(t1 - t0)));
                JOB_CUDA(down_later((T*)out->test.values + t0, d_tev.as<T>() + t0, sizeof(T) * (size_t)(t1 - t0)));
            }
            r0 = r1;
        }
        JOB_CUDA(downloads.finish());
        d2h_ms += downloads.copy_ms;          // (thread time: two copies run side by side)
        return true;
    }
};
#undef JOB_CUDA

template <typename T>
int run_split_impl(SplitKind kind, const int32_t* Xp, const int32_t* Xi, const T* Xv, int32_t m, int32_t n,
                   int32_t n_users_test, double test_fraction, bool consider_cold_start, int32_t min_items_pool,
                   int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    rmb::g_err.clear();
    if (!out) return fail(RMB200_ERR_BAD_ARG, "rmb200_split: out is NULL");
    std::memset(out, 0, sizeof(*out));
    out->value_bytes = (int32_t)sizeof(T);
    const auto t_call = clk::now();

    // the reference's own argument checks come first, in its order (hpp:1033-1036, :1225-1228)
    if (kind == SPLIT_WHOLE) {
        if (!m) return RMB200_OK;          // hpp:1033: nothing is written, every output stays empty
        if (m < 0 || n < 0) return fail(RMB200_ERR_RUNTIME, "Passed negative dimensions.\n");
    } else {
        if (n_users_test > m) return fail(RMB200_ERR_RUNTIME, "Target number of test users is larger than available users.\n");
        if (min_items_pool >= n) return fail(RMB200_ERR_RUNTIME, "Selected minimum number of items is larger than total number of items.\n");
        if (m <= 0) return fail(RMB200_ERR_BAD_ARG, "rmb200_split: X has no rows");
    }
    if (!Xp) return fail(RMB200_ERR_BAD_ARG, "rmb200_split: X_csr_p is NULL");
    const int64_t nnz = Xp[m];
    if (Xp[0] != 0) return fail(RMB200_ERR_BAD_ARG, "rmb200_split: X_csr_p[0] must be 0");
    if (nnz < 0 || (nnz > 0 && (!Xi || !Xv))) return fail(RMB200_ERR_BAD_ARG, "rmb200_split: X_csr_i / X_csr missing");

    TRY(rmb::use_device(device, &device));
    out->device = device;

    // ---- which rows, and how many entries of each are held out: everything the result's shape depends on ----
    SplitPlan P;
    if (const char* refusal = plan_split(Xp, m, n, kind != SPLIT_WHOLE, n_users_test, test_fraction, consider_cold_start,
                                         min_items_pool, min_pos_test, seed, P))
        return fail(RMB200_ERR_RUNTIME, refusal);
    const int32_t ns = P.ns, nr = P.nr;
    const int64_t sel_nnz = P.sel_p[ns], test_nnz = P.test_p[ns], rem_nnz = nr ? P.rem_p[nr] : 0;
    const int64_t train_nnz = sel_nnz - test_nnz + (kind == SPLIT_JOINED ? rem_nnz : 0);

    // ---- the result (host side): pointer arrays come straight from the plan ----
    SplitOwner* own = new (std::nothrow) SplitOwner();
    if (!own) return fail(RMB200_ERR_OOM, "host allocation");
    out->owner = own;
    auto csr_alloc = [&](rmb200_csr_t& M, int32_t rows, int64_t count) {
        M.rows = rows; M.cols = n; M.nnz = count;
        M.indptr = (int32_t*)host_block(own, sizeof(int32_t) * ((size_t)rows + 1));
        M.indices = (int32_t*)host_block(own, sizeof(int32_t) * (size_t)count, true);
        M.values = host_block(own, sizeof(T) * (size_t)count, true);
        return M.indptr && M.indices && M.values;
    };
    bool ok = csr_alloc(out->test, ns, test_nnz) && csr_alloc(out->train, ns + (kind == SPLIT_JOINED ? nr : 0), train_nnz);
    if (ok && kind == SPLIT_SEPARATE) ok = csr_alloc(out->rem, nr, rem_nnz);
    if (ok && kind != SPLIT_WHOLE) {
        out->users_test = (int32_t*)host_block(own, sizeof(int32_t) * (size_t)ns);
        ok = out->users_test != nullptr;
    }
    if (!ok) { rmb200_split_free(out); return fail(RMB200_ERR_OOM, "host allocation of the split"); }
    std::memcpy(out->test.indptr, P.test_p.data(), sizeof(int32_t) * ((size_t)ns + 1));
    std::memcpy(out->train.indptr, P.train_p.data(), sizeof(int32_t) * ((size_t)ns + 1));
    if (kind == SPLIT_JOINED)       // concat_csr_matrices, hpp:1324-1359: the remainder's pointer shifted by the training entries above it
        for (int32_t r = 1; r <= nr; r++) out->train.indptr[ns + r] = P.train_p[ns] + P.rem_p[r];
    if (kind == SPLIT_SEPARATE) std::memcpy(out->rem.indptr, P.rem_p.data(), sizeof(int32_t) * ((size_t)nr + 1));
    if (kind != SPLIT_WHOLE) {
        std::memcpy(out->users_test, P.sel_rows.data(), sizeof(int32_t) * (size_t)ns);
        out->n_users_test = ns;
    }

    // ---- three things at once: pages of the result touched, the GPU driven, the random stream replayed (this thread) ----
    Progress prog(P.chunk_end.size());
    DeviceJob<T> job{kind, device, Xp, Xi, Xv, m, nnz, P, out, prog};
    struct Joiner { std::thread t; ~Joiner() { if (t.joinable()) t.join(); } };
    double replay_ms = 0.0;
    {
        Joiner toucher{std::thread([&]() { try { touch_pages(own); } catch (...) {} prog.sig.update([&]() { prog.touched.store(1, std::memory_order_release); }); })};
        Joiner driver{std::thread([&]() {
            try {
                if (job.upload() && job.order_unsorted_rows() && job.gather_untouched_rows()) job.partition_chunks();
            } catch (...) { job.status = RMB200_ERR_OOM; job.what = "device thread"; prog.sig.update([&]() { prog.stop.store(1); }); }
            job.downloads.finish();      // (after a failure too: the copy threads write into the result, which is freed below)
        })};
        const auto t_replay = clk::now();
        try {
            Replay replay{P, seed, prog};
            replay.run();
        } catch (...) {
            prog.sig.update([&]() { prog.stop.store(1); });
            throw;                   // (Joiner joins the device thread first)
        }
        replay_ms = ms_since(t_replay);
    }
    out->plan_ms = replay_ms;
    out->h2d_ms = job.h2d_ms; out->d2h_ms = job.d2h_ms; out->kernel_ms = job.kernel_ms;
    out->kernel_launches = job.launches; out->h2d_bytes = job.h2d_bytes; out->d2h_bytes = job.d2h_bytes;
    out->rows_sorted_on_device = job.sorted_on_device;
    if (job.status != RMB200_OK) {
        rmb200_split_free(out);
        return fail(job.status, job.what.c_str(), job.detail.c_str());
    }
    out->total_ms = ms_since(t_call);
    return RMB200_OK;
}

// a failed split hands back no matrices
template <typename T, typename... Args>
int run_split(rmb200_split_t* out, Args... args)
{
    const int rc = rmb::guard([&] { return run_split_impl<T>(args..., out); });
    if (rc != RMB200_OK && out) rmb200_split_free(out);
    return rc;
}

}  // namespace

extern "C" {

int rmb200_split_selected_users_f32(const int32_t* Xp, const int32_t* Xi, const float* Xv, int32_t m, int32_t n,
                                    double test_fraction, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    return run_split<float>(out, SPLIT_WHOLE, Xp, Xi, Xv, m, n, 0, test_fraction, false, 0, 0, seed, device);
}

int rmb200_split_selected_users_f64(const int32_t* Xp, const int32_t* Xi, const double* Xv, int32_t m, int32_t n,
                                    double test_fraction, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    return run_split<double>(out, SPLIT_WHOLE, Xp, Xi, Xv, m, n, 0, test_fraction, false, 0, 0, seed, device);
}

int rmb200_split_separate_users_f32(const int32_t* Xp, const int32_t* Xi, const float* Xv, int32_t m, int32_t n,
                                    int32_t n_users_test, double test_fraction, int consider_cold_start, int32_t min_items_pool,
                                    int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    return run_split<float>(out, SPLIT_SEPARATE, Xp, Xi, Xv, m, n, n_users_test, test_fraction, consider_cold_start != 0,
                            min_items_pool, min_pos_test, seed, device);
}

int rmb200_split_separate_users_f64(const int32_t* Xp, const int32_t* Xi, const double* Xv, int32_t m, int32_t n,
                                    int32_t n_users_test, double test_fraction, int consider_cold_start, int32_t min_items_pool,
                                    int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    return run_split<double>(out, SPLIT_SEPARATE, Xp, Xi, Xv, m, n, n_users_test, test_fraction, consider_cold_start != 0,
                             min_items_pool, min_pos_test, seed, device);
}

int rmb200_split_joined_users_f32(const int32_t* Xp, const int32_t* Xi, const float* Xv, int32_t m, int32_t n,
                                  int32_t n_users_test, double test_fraction, int consider_cold_start, int32_t min_items_pool,
                                  int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    return run_split<float>(out, SPLIT_JOINED, Xp, Xi, Xv, m, n, n_users_test, test_fraction, consider_cold_start != 0,
                            min_items_pool, min_pos_test, seed, device);
}

int rmb200_split_joined_users_f64(const int32_t* Xp, const int32_t* Xi, const double* Xv, int32_t m, int32_t n,
                                  int32_t n_users_test, double test_fraction, int consider_cold_start, int32_t min_items_pool,
                                  int32_t min_pos_test, uint64_t seed, int32_t device, rmb200_split_t* out)
{
    return run_split<double>(out, SPLIT_JOINED, Xp, Xi, Xv, m, n, n_users_test, test_fraction, consider_cold_start != 0,
                             min_items_pool, min_pos_test, seed, device);
}

int rmb200_split_plan(const int32_t* Xp, int32_t m, int32_t n, int32_t sample_users, int32_t n_users_test, double test_fraction,
                      int consider_cold_start, int32_t min_items_pool, int32_t min_pos_test, uint64_t seed,
                      int32_t* users_test, int32_t* n_users_out, uint8_t* held, int64_t* n_entries_out)
{
    rmb::g_err.clear();
    if (!Xp || m <= 0 || !held || !n_entries_out) return fail(RMB200_ERR_BAD_ARG, "rmb200_split_plan: bad arguments");
    return rmb::guard([&] {
        if (sample_users && (!users_test || !n_users_out)) return fail(RMB200_ERR_BAD_ARG, "rmb200_split_plan: users_test missing");
        SplitPlan P;
        if (const char* refusal = plan_split(Xp, m, n, sample_users != 0, n_users_test, test_fraction, consider_cold_start != 0,
                                             min_items_pool, min_pos_test, seed, P))
            return fail(RMB200_ERR_RUNTIME, refusal);
        Progress prog(P.chunk_end.size());
        Replay replay{P, seed, prog};
        replay.run();
        for (size_t c = 0; c < P.chunk_end.size(); c++)
            if (!prog.chunk_done[c].load()) return fail(RMB200_ERR_CUDA, "rmb200_split_plan: a chunk was never published");
        if (sample_users) {
            std::memcpy(users_test, P.sel_rows.data(), sizeof(int32_t) * P.sel_rows.size());
            *n_users_out = (int32_t)P.sel_rows.size();
        } else if (n_users_out) *n_users_out = m;
        std::memcpy(held, P.held.data(), P.held.size());
        *n_entries_out = (int64_t)P.held.size();
        return (int)RMB200_OK;
    });
}

void rmb200_split_free(rmb200_split_t* split)
{
    if (!split) return;
    if (SplitOwner* own = (SplitOwner*)split->owner) {
        for (void* p : own->blocks) std::free(p);
        delete own;
    }
    const int32_t vb = split->value_bytes;
    std::memset(split, 0, sizeof(*split));
    split->value_bytes = vb;
}

int rmb200_sizeof_split(void) { return (int)sizeof(rmb200_split_t); }

}  // extern "C"
