// C ABI of the batched ICP library (include/icpb.h).  Plain CUDA runtime: no torch types, no
// C++ exceptions across the boundary.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include <new>
#include <vector>
#include <algorithm>
#include <atomic>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <sched.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "icpb.h"
#include "icpb_kernels.cuh"
#include "icpb_candidates.cuh"
#include "icpb_sgd.cuh"
#include "icpb_grid.cuh"
#include "icpb_compose.cuh"
#include "icpb_multistart.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, const char *detail = "")
{
    snprintf(g_err, sizeof g_err, fmt, detail);
    return code;
}

#define CU(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            snprintf(g_err, sizeof g_err, "%s failed: %s", #call, cudaGetErrorString(e_)); \
            return (int)e_;                                                               \
        }                                                                                 \
    } while (0)

// Every entry point runs on the handle's device and puts the caller's current device back on the
// way out (a torch process with several devices must not find its current device changed).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) {
            const cudaError_t e = cudaSetDevice(device);
            if (e != cudaSuccess) {
                snprintf(g_err, sizeof g_err, "cudaSetDevice(%d) failed: %s", device, cudaGetErrorString(e));
                ok = false;
            }
        } else {
            prev = -1;                                        // nothing to restore
        }
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ON_DEVICE(h)                                      \
    DeviceGuard guard_((h)->device);                      \
    if (!guard_.ok) return (int)cudaErrorInvalidDevice

#ifndef ICPB_R
#define ICPB_R 2
#endif
constexpr int kPointsPerThread = ICPB_R;
constexpr int kQueueRing = 64;
constexpr int kQueueWords = kQueueRing + 3;       // the ring, the work counter, the two acceptance counters


struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return (int)e; }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinnedBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e)); return (int)e; }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// The layout of one synchronous call's arrays in the handle's scratch arena (icpb_ctx::arena): every
// carve() names one array and returns its 256-byte-aligned offset; `used`, the total, is reserved once at
// the top of the call, and at() turns an offset into the array.  Nothing carved outlives its call.
struct Carve {
    size_t used = 0;
    size_t operator()(size_t bytes) { const size_t o = used; used += (bytes + 255) & ~size_t(255); return o; }
};
template <class T> T *at(const DevBuf &b, size_t o) { return (T *)((unsigned char *)b.p + o); }

constexpr int kMaxSegments = 64;        // pieces of the streaming scan-table upload (icpb_align_host)

struct LaunchCfg {
    int threads, smem, ctas_per_sm;
    icpb::SmemLayout L;
    int cluster;   // CTAs per problem (1 = ordinary launch)
    bool big;      // large-scan variant: the arrays before L.o_tw live in per-CTA device scratch
    int64_t big_stride;   // bytes of one CTA's scratch region
};

typedef void (*kernel_fn)(const icpb::KernelArgs);
// The exhaustive variant (every source point sweeps every target) keeps 4 points per thread in
// 256-thread CTAs: with no pruning there is nothing to balance, and the wider register tile
// amortises the shared-memory loads and the per-chunk bookkeeping over twice the distances.
constexpr int kPointsExhaustive = 4;
bool is_exhaustive(const icpb_params *p) { return p && (p->flags & ICPB_FLAG_EXHAUSTIVE); }
int points_per_thread(const icpb_params *p) { return is_exhaustive(p) ? kPointsExhaustive : kPointsPerThread; }
// The six instances of the alignment kernel: exhaustive, pruned, pruned in a cluster; the first three keep
// their arrays in shared memory, the last three are the large-scan variants (KernelArgs::big_scratch: same
// code, arrays in device scratch).
const kernel_fn kAlignKernels[6] = {
    icpb::icp_align_kernel<kPointsExhaustive, false, false>, icpb::icp_align_kernel<kPointsPerThread, true, false>,
    icpb::icp_align_kernel<kPointsPerThread, true, true>,
    icpb::icp_align_kernel<kPointsExhaustive, false, false, true>,
    icpb::icp_align_kernel<kPointsPerThread, true, false, true>,
    icpb::icp_align_kernel<kPointsPerThread, true, true, true>};
// (make_cfg never gives an exhaustive run a cluster: the cluster instance is a pruned one)
kernel_fn align_kernel(bool big, bool exhaustive, bool cluster)
{
    return kAlignKernels[(big ? 3 : 0) + (cluster ? 2 : exhaustive ? 0 : 1)];
}
// Scratch of the large-scan variant: one region per resident CTA, the grid capped so that all regions
// together stay within this budget (a 100,000-point scan needs ~1.7 MB per CTA: ~600 CTAs).
constexpr int64_t kBigScratchBudget = int64_t(1) << 30;

}  // namespace

namespace {

// A few host threads that copy scans from the caller's (pageable, scattered) arrays into the pinned
// staging table, one job = a run of consecutive scans.  Jobs are handed out in table order, so the
// first upload piece is complete first; `done[k]` counts the finished jobs of piece k and the
// dispatching thread enqueues the piece's copy as soon as it is full.
struct PackJob {
    const double *const *scan_xy;       // n_scans pointers to (m_i, 2) float64 rows
    const int64_t *offsets;             // CSR offsets of the packed table
    double *dst;                        // pinned staging
    const int64_t *job_first, *job_last;  // scans [first, last) of job j
    const int32_t *job_piece;           // upload piece of job j
    int64_t n_jobs = 0;
    std::atomic<int64_t> next{0};
    std::atomic<int32_t> *done;         // per piece
    std::atomic<uint64_t> bad{0};       // a coordinate beyond ICPB_MAX_COORD (or NaN) seen
};

// One scan into the pinned staging table with NON-TEMPORAL stores, checking on the way that every
// coordinate is within ICPB_MAX_COORD (!(|v| <= bound): NaN fails too).
// Ordinary stores leave the freshly written lines dirty in the writing core's private cache; the
// copy engine's reads then have to snoop them out of cores that have already gone idle, and the
// last pieces of the table -- the ones still cache resident when the packing ends -- crawl at
// ~8 GB/s instead of 55 (measured: the last two 5 MB pieces took 0.43 and 0.85 ms against 0.10 ms
// for the others).  Streaming stores go to memory through the write-combining buffers and skip
// the read-for-ownership as well.
static inline uint64_t copy_scan(double *dst, const double *src, int64_t n_doubles)
{
    uint64_t bad = 0;
#if defined(__x86_64__)
    const __m128d sign = _mm_set1_pd(-0.0), lim = _mm_set1_pd(ICPB_MAX_COORD);
    // not (|v| <= lim): the unordered compare is true for NaN
    auto out = [&](__m128d v) { return _mm_cmpnle_pd(_mm_andnot_pd(sign, v), lim); };
    __m128d acc = _mm_setzero_pd();
    int64_t k = 0;
    for (; k + 8 <= n_doubles; k += 8) {                                    // one 64-byte line per trip
        const __m128d a = _mm_loadu_pd(src + k), b = _mm_loadu_pd(src + k + 2);
        const __m128d c = _mm_loadu_pd(src + k + 4), d = _mm_loadu_pd(src + k + 6);
        _mm_stream_pd(dst + k, a); _mm_stream_pd(dst + k + 2, b);
        _mm_stream_pd(dst + k + 4, c); _mm_stream_pd(dst + k + 6, d);
        acc = _mm_or_pd(acc, _mm_or_pd(_mm_or_pd(out(a), out(b)), _mm_or_pd(out(c), out(d))));
    }
    for (; k + 2 <= n_doubles; k += 2) {
        const __m128d a = _mm_loadu_pd(src + k);
        _mm_stream_pd(dst + k, a);
        acc = _mm_or_pd(acc, out(a));
    }
    bad = (uint64_t)(_mm_movemask_pd(acc) != 0);
#else
    memcpy(dst, src, sizeof(double) * (size_t)n_doubles);
    for (int64_t k = 0; k < n_doubles; ++k)
        bad |= (uint64_t)!(fabs(dst[k]) <= ICPB_MAX_COORD);
#endif
    return bad;
}

static void pack_one(PackJob *job, int64_t j)
{
    uint64_t bad = 0;
    for (int64_t s = job->job_first[j]; s < job->job_last[j]; ++s) {
        const int64_t o = job->offsets[s], m = job->offsets[s + 1] - o;
        bad |= copy_scan(job->dst + 2 * o, job->scan_xy[s], 2 * m);
    }
#if defined(__x86_64__)
    _mm_sfence();                                       // the streamed lines are in memory before the piece is announced
#endif
    if (bad) job->bad.fetch_or(1, std::memory_order_relaxed);
    job->done[job->job_piece[j]].fetch_add(1, std::memory_order_release);
}

struct PackPool {
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv;
    PackJob *job = nullptr;
    uint64_t generation = 0;
    int running = 0;
    bool stop = false;

    explicit PackPool(int n)
    {
        for (int t = 0; t < n; ++t)
            workers.emplace_back([this] {
                uint64_t seen = 0;
                for (;;) {
                    PackJob *j;
                    {
                        std::unique_lock<std::mutex> lk(mu);
                        cv.wait(lk, [&] { return stop || generation != seen; });
                        if (stop) return;
                        seen = generation;
                        j = job;
                    }
                    for (int64_t i; (i = j->next.fetch_add(1, std::memory_order_relaxed)) < j->n_jobs;) pack_one(j, i);
                    {
                        std::lock_guard<std::mutex> lk(mu);
                        --running;
                    }
                    cv.notify_all();
                }
            });
    }
    void start(PackJob *j)
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            job = j; ++generation; running = (int)workers.size();
        }
        cv.notify_all();
    }
    void finish()                                       // the caller packs too, then waits for the workers
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return running == 0; });
        job = nullptr;
    }
    ~PackPool()
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv.notify_all();
        for (auto &w : workers) w.join();
    }
};

}  // namespace

struct icpb_ctx {
    int device = 0;
    int sm_count = 0;
    int smem_limit = 0;                             // dynamic shared memory an alignment launch may ask for
    // scan table
    const double *xy = nullptr;
    const int64_t *offsets = nullptr;
    int64_t n_scans = 0, longest = 0;
    std::vector<int64_t> host_off;                  // the table's offsets on the host (table_host_offsets)
    // queue counters
    unsigned long long *queue = nullptr;      // kQueueWords: kQueueRing counters, the work counter, then the
                                              // acceptance epilogue's [appended, CTAs left] counters
    unsigned long long *executed = nullptr;   // non-null while work counting is enabled
    int64_t launches = 0;
    // The scratch arrays of every entry point that synchronises before it returns, carved per call (Carve).
    // Memory that outlives a call stays out of it:
    //   own_xy, own_off  the resident table;
    //   prep             the table's staging images, kept until the table changes;
    //   s_big            launch()'s per-CTA scratch of the large-scan variant, also used by the asynchronous
    //                    icpb_run_device*, whose kernels may still run when the next call starts (launches
    //                    on different streams share it, as they share the acceptance counters);
    //   stage, stage_xy  pinned: reallocating pinned memory is slow, and their sizes vary independently
    //                    (the batch size and the table size).
    DevBuf arena;
    DevBuf own_xy, own_off;
    cudaStream_t stream = nullptr;
    cudaStream_t cstream[2] = {nullptr, nullptr};   // compute streams of the pipelined host entry point
    // align_impl: the arrival counter is zero / the pairs block is up / the kernel is done
    cudaEvent_t counter_zeroed = nullptr, inputs_up = nullptr, kernel_done = nullptr;
    int32_t *arrived_dev = nullptr;                 // streaming upload: segments delivered so far
    // cuStreamWriteValue32 (driver API, looked up at run time): a stream-ordered 4-byte store, cheaper
    // than a 4-byte DMA for the "segment k has arrived" counter; nullptr -> the counter is copied
    int (*write32)(cudaStream_t, unsigned long long, unsigned int, unsigned int) = nullptr;
    int32_t *seg_vals_pinned = nullptr;             // 0..kMaxSegments in pinned host memory (sources of the flag copies)
    PinnedBuf stage;                                // pinned staging of align_impl's per-pair blocks
    DevBuf s_big;                                   // large-scan variant: one scratch region per CTA
    // per-scan staging images of the resident table (KernelArgs::prep_in), built on first use
    DevBuf prep;
    const double *prep_for = nullptr;               // the table (h->xy) the images were built from
    int64_t prep_stride = 0, prep_scans = 0, prep_longest = 0;
    PinnedBuf stage_xy;                             // pinned copy of a scan table packed from a list of arrays
    PackPool *pool = nullptr;                       // host threads that pack scans into stage_xy
    // tuning / test hooks (icpb_set_tuning); 0 or -1 = the library's own choice
    int tune_threads = 0, tune_cluster = -1, tune_segments = 0, tune_pack_threads = 0, tune_large = -1;
    bool tune_drop_counter = false;
};

namespace {

// A pair fits the shared-memory kernel when the layout of its longer scan fits at the widest CTA a
// launch may pick (8 warps), so that it fits whatever width the launch settles on.
bool fits_smem(const icpb_ctx *h, int64_t n)
{
    const icpb::SmemLayout L = icpb::smem_layout(n, 8);
    return L.bytes != 0x7fffffff && L.bytes <= h->smem_limit;
}

// The handle's scan table; a new table has no staging images yet (ensure_prep).  off_host: the offsets
// on the host, kept when a batch on the table may be split by scan length (null for a borrowed table).
void set_table(icpb_ctx *h, const double *xy, const int64_t *off, int64_t n_scans, int64_t longest,
               const int64_t *off_host)
{
    h->prep_for = nullptr; h->xy = xy; h->offsets = off; h->n_scans = n_scans; h->longest = longest;
    h->host_off.clear();
    if (off_host && !fits_smem(h, longest)) h->host_off.assign(off_host, off_host + n_scans + 1);
}

void drop_table(icpb_ctx *h) { set_table(h, nullptr, nullptr, 0, 0, nullptr); }

// The table's offsets on the host, for split_queue: kept by set_table for a table from host memory,
// fetched on first need for a borrowed one and kept until the next set_table.
int table_host_offsets(icpb_ctx *h, const int64_t **out)
{
    if (h->host_off.empty()) {
        std::vector<int64_t> off((size_t)h->n_scans + 1);
        CU(cudaMemcpyAsync(off.data(), h->offsets, sizeof(int64_t) * off.size(), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        h->host_off.swap(off);
    }
    *out = h->host_off.data();
    return 0;
}

// A whole table from host memory into the handle's own buffers (reserved by the caller), which then hold
// the handle's table.
int upload_table(icpb_ctx *h, const double *xy, const int64_t *off, int64_t n_scans, int64_t longest)
{
    CU(cudaMemcpyAsync(h->own_xy.p, xy, sizeof(double) * 2 * (size_t)off[n_scans], cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->own_off.p, off, sizeof(int64_t) * (size_t)(n_scans + 1), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    set_table(h, (const double *)h->own_xy.p, (const int64_t *)h->own_off.p, n_scans, longest, off);
    return 0;
}

// Launch geometry for a batch whose longest scan has `longest` points.  When the layout does not fit
// one CTA's shared memory (or `big` asks for it) the launch uses the large-scan variant.
int make_cfg(icpb_ctx *h, int64_t longest, int64_t B, LaunchCfg *c, const icpb_params *p, bool big = false)
{
    if (longest <= 0) return fail(ICPB_EINVAL, "empty scan table%s");
    const int R = points_per_thread(p);
    const int64_t ntile = (longest + 63) / 64;              // 64-point reduction tiles (independent of R)
    const int64_t nwork = (ntile + R / 2 - 1) / (R / 2);    // warp work items of 32*R points
    // Warps per CTA.  Small CTAs keep more independent problems in flight per SM (less idling at the
    // per-pass barrier); large CTAs finish a problem sooner, which matters when the batch is only a few
    // problems per resident CTA (tail) or a single pair (latency).  Within the cap, the count that leaves
    // the fewest warps idle in the last round of a pass wins (360-beam scans have 6 tiles: 3 warps take
    // two each, 12.2 M pairs/s, where 4 warps left two idle every second round, 11.5 M), larger on ties.
    int max_warps = (B >= 2048 && R < 4) ? 4 : 8;
    if (h->tune_threads >= 32 && h->tune_threads <= 256 && h->tune_threads % 32 == 0)
        max_warps = h->tune_threads / 32;                 // icpb_set_tuning("threads")
    int warps = 1;
    {
        int64_t best_waste = -1;
        for (int w = max_warps < nwork ? max_warps : (int)nwork; w >= (max_warps >= 2 && nwork >= 2 ? 2 : 1); --w) {
            const int64_t waste = (nwork + w - 1) / w * w - nwork;
            if (best_waste < 0 || waste < best_waste) { best_waste = waste; warps = w; }
        }
        if (h->tune_threads > 0) warps = max_warps < nwork ? max_warps : (int)nwork;   // forced: no search
    }
    int threads = warps * 32;
    const icpb::SmemLayout L = icpb::smem_layout(longest, threads / 32);
    if (L.bytes == 0x7fffffff) {
        snprintf(g_err, sizeof g_err, "scan of %lld points is beyond the kernel's 32-bit layout offsets",
                 (long long)longest);
        return ICPB_ETOOLONG;
    }
    if (L.bytes > h->smem_limit) big = true;
    const kernel_fn fn = align_kernel(big, is_exhaustive(p), false);
    // large-scan variant: Tw, S0 and the transpose scratch stay in shared memory, at offsets from 0
    const int64_t smem = big ? L.bytes - L.o_tw : L.bytes;
    c->threads = threads; c->smem = (int)smem; c->L = L; c->big = big;
    c->big_stride = big ? ((int64_t)L.o_tw + 255) & ~int64_t(255) : 0;
    // Latency mode: when every CTA of every cluster can have an SM of its own and a CTA's eight warps
    // would each get more than one tile per pass, spread each problem over a thread-block cluster (a
    // power of two, at most 8 CTAs) so that every tile has a warp.  Measured with one cluster per
    // problem resident (tools/latency.py, tools/midsize_probe.py, round 2): one 1,024-point pair 0.165 ms
    // in a CTA, 0.153 in a cluster of two, 0.141 in eight; 40 such pairs 0.37 -> 0.31 ms with clusters of
    // two, 80 pairs 0.41 -> 0.38; from 120 pairs on (more CTAs than SMs) single CTAs win; one 4,096-point
    // pair 0.78 -> 0.41 ms in a cluster of eight.
    c->cluster = 1;
    if (!is_exhaustive(p) && nwork > 8) {
        int cl = 2;
        while (cl < 8 && (int64_t)cl * 8 < nwork) cl *= 2;
        while (cl > 1 && B * cl > h->sm_count) cl /= 2;
        c->cluster = cl;
    }
    if (h->tune_cluster >= 0) {                           // icpb_set_tuning("cluster"): force a size (0 = never)
        const int v = h->tune_cluster;
        if (v == 0 || v == 1) c->cluster = 1;
        else if ((v == 2 || v == 4 || v == 8) && !is_exhaustive(p)) c->cluster = v;
    }
    // (the kernels' dynamic shared-memory limit is raised to the device maximum once, in icpb_create: the
    // attribute belongs to the function, not to a handle, so it must not follow one handle's history)
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
    if (per_sm < 1) return fail(ICPB_EINVAL, "kernel does not fit on an SM%s");
    c->ctas_per_sm = per_sm;
    return 0;
}

int check_params(const icpb_params *p, int64_t B)
{
    if (!p) return fail(ICPB_EINVAL, "params is null%s");
    if (B < 0) return fail(ICPB_EINVAL, "negative batch size%s");
    if (p->hist_cap < 0 || p->corr_stride < 0) return fail(ICPB_EINVAL, "negative hist_cap/corr_stride%s");
    if (p->pair_mode != 0 && p->pair_mode != 1) return fail(ICPB_EINVAL, "pair_mode must be 0 or 1%s");
    if (p->pair_mode == 1 && p->k_block < 1) return fail(ICPB_EINVAL, "pair_mode 1 needs k_block >= 1%s");
    if (isnan(p->epsilon) || isnan(p->stopping_thresh)) return fail(ICPB_EINVAL, "NaN epsilon/stopping_thresh%s");
    return 0;
}

int check_epilogue(const icpb_epilogue *ep)
{
    if (!ep) return 0;
    const bool gather = ep->d_peer_ptrs != nullptr;
    const bool accept = ep->d_accept_rec != nullptr || ep->d_accept_peer_ptrs != nullptr;
    if ((gather || ep->d_accept_peer_ptrs) && (ep->n_peers < 1 || ep->n_peers > 64))
        return fail(ICPB_EINVAL, "epilogue: 1..64 peer buffers expected%s");
    if (ep->row0 < 0 || ep->row_stride < 0) return fail(ICPB_EINVAL, "epilogue: negative row0 / row_stride%s");
    if (accept) {
        if (ep->accept_cap < 1) return fail(ICPB_EINVAL, "epilogue: accept_cap must be >= 1%s");
        if (isnan(ep->accept_thresh)) return fail(ICPB_EINVAL, "epilogue: NaN accept_thresh%s");
        if (ep->d_accept_peer_ptrs && (!ep->d_accept_count_peer_ptrs || ep->rank < 0 || ep->rank >= ep->n_peers))
            return fail(ICPB_EINVAL, "epilogue: peer acceptance needs the peers' count arrays and a rank in range%s");
        if (!ep->d_accept_peer_ptrs && !ep->d_accept_count) return fail(ICPB_EINVAL, "epilogue: d_accept_count is null%s");
    }
    return 0;
}

// The checks of icpb_run_device, icpb_run_device_ex and icpb_run_host, in this order: handle, parameters,
// table, then the (host or device) buffers.  empty_ok: a batch of no pairs needs no buffers.
int run_check(const icpb_ctx *h, const icpb_params *p, int64_t B, bool empty_ok, const void *pairs,
              const void *T, const void *err, const void *passes, const void *hist, const void *corr)
{
    if (!h) return fail(ICPB_EINVAL, "handle is null%s");
    int rc = check_params(p, B);
    if (rc) return rc;
    if (!h->xy) return fail(ICPB_ENOSCANS, "no scan table set%s");
    if (B == 0 && empty_ok) return 0;
    if (B > 0 && (!T || !err || !passes)) return fail(ICPB_EINVAL, "output pointer is null%s");
    if (B > 0 && p->pair_mode == 0 && !pairs) return fail(ICPB_EINVAL, "pairs is null with pair_mode 0%s");
    if (p->hist_cap > 0 && !hist) return fail(ICPB_EINVAL, "hist_cap > 0 without a history buffer%s");
    if (p->corr_stride > 0 && !corr) return fail(ICPB_EINVAL, "corr_stride > 0 without a correspondence buffer%s");
    if (p->corr_stride > 0 && p->corr_stride < h->longest)
        return fail(ICPB_EINVAL, "corr_stride is smaller than the longest scan%s");
    return 0;
}

// Every scan id of B explicit pairs names a scan of the table.
int check_pairs(const int32_t *pairs, int64_t B, int64_t n_scans)
{
    int32_t lo = 0, hi = 0;                                   // branch-free range check
    for (int64_t b = 0; b < 2 * B; ++b) { lo = pairs[b] < lo ? pairs[b] : lo; hi = pairs[b] > hi ? pairs[b] : hi; }
    if (lo < 0 || hi >= n_scans) return fail(ICPB_EINVAL, "pair index out of range%s");
    return 0;
}

int ensure_prep(icpb_ctx *h, cudaStream_t stream);

// A batch whose longest scan does not fit shared memory, on an entry point that sees the pairs, runs as
// two launches: the pairs that fit (fits_smem of the longer scan) on the shared-memory kernel at the
// layout of the longest scan among them, then the others on the large-scan variant.  Both write the
// outputs by pair id; the queue holds the first part's pairs, then the second's, each in its original
// order.  The two variants give the same bits, so the split decides speed only.
struct Split {
    int64_t ns = 0;            // pairs in the first part
    int64_t Ls = 0, Ll = 0;    // longest scan of each part
};

// One batch of alignment problems as launch() enqueues it.  Fields a caller does not set stay null / 0.
struct Batch {
    const double *xy = nullptr;                     // the scan table
    const int64_t *offsets = nullptr;
    int64_t n_scans = 0, longest = 0;
    const int32_t *pairs = nullptr;                 // the problems
    const double *init = nullptr;
    int64_t B = 0;
    const icpb_params *p = nullptr;
    double *T = nullptr, *err = nullptr, *hist = nullptr;   // the outputs, by pair id
    int32_t *passes = nullptr, *corr = nullptr;
    cudaStream_t stream = nullptr;
    const icpb_epilogue *ep = nullptr;
    const int32_t *order = nullptr;                 // queue position -> pair id (nullptr: identity)
    // streaming upload: a pair waits until *arrived > seg_of_pair[its queue position]
    const int32_t *seg_of_pair = nullptr, *arrived = nullptr;
    int32_t *upload_timeout = nullptr;
    unsigned char *prep_out = nullptr;              // prep mode: build the table's staging images (ensure_prep)
    int64_t prep_stride = 0;
    const Split *split = nullptr;                   // split by scan length; `order` holds the split queue
};

// Enqueues a batch: one kernel launch, or two for a split batch (queue positions [0, ns) on the
// shared-memory kernel at the layout of Ls, the others on the large-scan variant at Ll).  A batch
// without a split is one whose first part holds every pair.
int launch(icpb_ctx *h, const Batch &b)
{
    const icpb_params *p = b.p;
    const bool prep_building = b.prep_out != nullptr;
    const Split whole = {b.B, b.longest, 0};
    const Split &sp = b.split ? *b.split : whole;
    for (int part = 0; part < 2; ++part) {
        const int64_t q0 = part ? sp.ns : 0;                  // queue position of the part's first pair
        const int64_t B = part ? b.B - sp.ns : sp.ns, longest = part ? sp.Ll : sp.Ls;
        if (B == 0) continue;
        LaunchCfg cfg;
        int rc = make_cfg(h, longest, B, &cfg, p, part == 1 || (h->tune_large == 1 && !prep_building));
        if (rc) return rc;
        const kernel_fn fn = align_kernel(cfg.big, is_exhaustive(p), cfg.cluster > 1);
        icpb::KernelArgs a;
        a.xy = b.xy; a.offsets = b.offsets; a.pairs = b.pairs; a.init = b.init; a.B = B; a.n_scans = b.n_scans;
        a.p = *p;
        a.T_out = b.T; a.err_out = b.err; a.passes_out = b.passes;
        a.hist = p->hist_cap > 0 ? b.hist : nullptr;
        a.corr = p->corr_stride > 0 ? b.corr : nullptr;
        a.queue = h->queue + (h->launches % kQueueRing);
        a.n2pad_cap = cfg.L.n2pad; a.n1_cap = cfg.L.n1c; a.nchunk_cap = cfg.L.nchunk; a.ntile_cap = cfg.L.ntile;
        a.o_tqy = cfg.L.o_tqy; a.o_cb = cfg.L.o_cb; a.o_tc = cfg.L.o_tc; a.o_mm = cfg.L.o_mm; a.o_corr = cfg.L.o_corr;
        a.o_red = cfg.L.o_red; a.o_tw = cfg.L.o_tw; a.o_s0 = cfg.L.o_s0; a.o_scr = cfg.L.o_scr;
        a.big_scratch = nullptr; a.big_stride = 0;
        if (cfg.big) { a.o_tw = 0; a.o_s0 = cfg.L.o_s0 - cfg.L.o_tw; a.o_scr = cfg.L.o_scr - cfg.L.o_tw; }
        a.executed = h->executed;
        a.seg_of_pair = b.seg_of_pair ? b.seg_of_pair + q0 : nullptr; a.arrived = b.arrived;
        a.order = b.order ? b.order + q0 : nullptr; a.upload_timeout = b.upload_timeout;
        a.prep_out = b.prep_out; a.prep_in = nullptr; a.prep_stride = b.prep_stride;
        if (b.arrived == nullptr && b.xy == h->xy && h->xy != nullptr && !prep_building && longest == h->longest) {
            // a resident table: stage every pair by copy from the per-scan images (built once per table)
            int rc2 = ensure_prep(h, b.stream);
            if (rc2) return rc2;
            if (h->prep_for == h->xy) { a.prep_in = (const unsigned char *)h->prep.p; a.prep_stride = h->prep_stride; }
        }
        // epilogue rows are pair ids of the whole batch
        a.peers = nullptr; a.n_peers = 0; a.rec_row0 = 0; a.rec_block = b.B; a.rec_stride = 0;
        a.accept_thresh = 0.0; a.accept_rec = nullptr; a.accept_peers = nullptr; a.accept_ctr = nullptr;
        a.accept_count_out = nullptr; a.accept_count_peers = nullptr; a.accept_cap = 0; a.accept_rank = 0;
        if (const icpb_epilogue *ep = b.ep) {
            a.peers = (double *const *)ep->d_peer_ptrs; a.n_peers = ep->n_peers;
            a.rec_row0 = ep->row0; a.rec_stride = ep->row_stride;
            if (ep->row_block > 0) a.rec_block = ep->row_block;
            if (ep->d_accept_rec || ep->d_accept_peer_ptrs) {
                a.accept_thresh = ep->accept_thresh; a.accept_cap = ep->accept_cap; a.accept_rank = ep->rank;
                a.accept_rec = ep->d_accept_peer_ptrs ? nullptr : ep->d_accept_rec;
                a.accept_peers = (double *const *)ep->d_accept_peer_ptrs;
                a.accept_count_peers = (long long *const *)ep->d_accept_count_peer_ptrs;
                a.accept_count_out = (long long *)ep->d_accept_count;
                a.accept_ctr = h->queue + kQueueRing + 1;
                // [0] rows appended: zeroed by the first launch of a batch only; [1] CTAs that have left: per launch
                const bool cont = q0 > 0;
                CU(cudaMemsetAsync(a.accept_ctr + (cont ? 1 : 0), 0, (cont ? 1 : 2) * sizeof(unsigned long long), b.stream));
            }
        }
        CU(cudaMemsetAsync(a.queue, 0, sizeof(unsigned long long), b.stream));
        int64_t grid = (int64_t)cfg.ctas_per_sm * h->sm_count;
        if (grid > B) grid = B;
        int64_t max_ctas = grid * cfg.cluster;                    // CTAs the launch may have
        if (cfg.big) {
            // one scratch region per CTA, within kBigScratchBudget; with less device memory free, fewer
            // CTAs, down to one cluster (or CTA) -- only if that cannot be had does the call fail
            int64_t cap = kBigScratchBudget / cfg.big_stride / cfg.cluster * cfg.cluster;
            if (cap < cfg.cluster) cap = cfg.cluster;
            if (max_ctas > cap) max_ctas = cap;
            for (;;) {
                const int rc2 = h->s_big.reserve((size_t)(max_ctas * cfg.big_stride));
                if (rc2 == 0) break;
                cudaGetLastError();
                if (max_ctas <= cfg.cluster) return rc2;          // g_err names the allocation that failed
                max_ctas = (max_ctas / 2 + cfg.cluster - 1) / cfg.cluster * cfg.cluster;
            }
            a.big_scratch = (unsigned char *)h->s_big.p; a.big_stride = cfg.big_stride;
            if (grid > max_ctas) grid = max_ctas;
        }
        if (cfg.cluster > 1) {
            cudaLaunchConfig_t lc = {};
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = (unsigned)cfg.cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
            lc.blockDim = dim3((unsigned)cfg.threads);
            lc.dynamicSmemBytes = (size_t)cfg.smem; lc.stream = b.stream; lc.attrs = attr; lc.numAttrs = 1;
            // one cluster per problem, as many as the device can co-schedule (the occupancy query needs a
            // grid that is a multiple of the cluster size; it answers in clusters)
            lc.gridDim = dim3((unsigned)cfg.cluster);
            int max_clusters = 0;
            CU(cudaOccupancyMaxActiveClusters(&max_clusters, fn, &lc));
            int64_t clusters = max_clusters > 0 ? max_clusters : 1;
            if (clusters > B) clusters = B;
            if (clusters > max_ctas / cfg.cluster) clusters = max_ctas / cfg.cluster;
            lc.gridDim = dim3((unsigned)(clusters * cfg.cluster));
            CU(cudaLaunchKernelEx(&lc, fn, a));
        } else {
            fn<<<(unsigned)grid, cfg.threads, cfg.smem, b.stream>>>(a);
        }
        CU(cudaGetLastError());
        h->launches++;
    }
    return 0;
}

// The device form of a resident scan table: besides the fp64 points, one staging image per scan (fp32
// target arrays, chunk circles, group circles, S0, largest coordinate), built by one launch of the
// alignment kernel in prep mode the first time the table is used.  A pair's staging is then a 10 KB copy
// instead of ~11,000 warp instructions; scans that take part in many pairs (loop-closure candidates, all
// pairs) are prepared once instead of once per pair.  Tables whose images would exceed 8 GB are staged
// per pair as before.  So are tables whose longest scan does not fit shared memory (the images are laid
// out for the table's longest scan, and a launch reads them at its own layout's offsets: the short pairs
// of such a table run at a smaller layout, its long pairs stage into scratch per pair).
int ensure_prep(icpb_ctx *h, cudaStream_t stream)
{
    if (h->prep_for == h->xy && h->prep_scans == h->n_scans && h->prep_longest == h->longest) return 0;
    h->prep_for = nullptr;
    const icpb::SmemLayout L = icpb::smem_layout(h->longest, 4);
    const int64_t stride = ((int64_t)L.o_mm + 32 + 15) & ~int64_t(15);
    if (stride * h->n_scans > (int64_t(8) << 30)) return 0;
    int rc;
    icpb_params p;
    icpb_default_params(&p);
    p.k_block = h->n_scans;
    LaunchCfg cfg;
    if ((rc = make_cfg(h, h->longest, h->n_scans, &cfg, &p))) return rc;
    if (cfg.big) return 0;
    if ((rc = h->prep.reserve((size_t)(stride * h->n_scans)))) return rc;
    Batch b;
    b.xy = h->xy; b.offsets = h->offsets; b.n_scans = h->n_scans; b.longest = h->longest;
    b.B = h->n_scans; b.p = &p; b.stream = stream;
    b.prep_out = (unsigned char *)h->prep.p; b.prep_stride = stride;
    if ((rc = launch(h, b))) return rc;
    h->prep_for = h->xy; h->prep_stride = stride; h->prep_scans = h->n_scans; h->prep_longest = h->longest;
    return 0;
}

// Whether a batch has to be split: its longest scan does not fit and "large" does not force the variant.
bool needs_split(icpb_ctx *h, int64_t longest, int64_t B, const icpb_params *p)
{
    if (h->tune_large == 1 || B < 1 || p->pair_mode != 0) return false;
    LaunchCfg cfg;
    return make_cfg(h, longest, B, &cfg, p) == 0 && cfg.big;
}

// order[q] (queue position q -> pair id) for the split; queue: the queue before it (nullptr: identity).
// seg (by queue position, optional) is permuted along.
Split split_queue(const icpb_ctx *h, const int64_t *off, const int32_t *pairs, int64_t B, const int32_t *queue,
                  int32_t *order, int32_t *seg)
{
    Split sp;
    std::vector<int32_t> lo, hi, slo, shi;
    for (int64_t q = 0; q < B; ++q) {
        const int32_t b = queue ? queue[q] : (int32_t)q;
        const int64_t n1 = off[pairs[2 * b] + 1] - off[pairs[2 * b]], n2 = off[pairs[2 * b + 1] + 1] - off[pairs[2 * b + 1]];
        const int64_t n = n1 > n2 ? n1 : n2;
        const bool fit = fits_smem(h, n);
        (fit ? lo : hi).push_back(b);
        if (seg) (fit ? slo : shi).push_back(seg[q]);
        int64_t &L = fit ? sp.Ls : sp.Ll;
        if (n > L) L = n;
    }
    sp.ns = (int64_t)lo.size();
    std::copy(lo.begin(), lo.end(), order);
    std::copy(hi.begin(), hi.end(), order + sp.ns);
    if (seg) { std::copy(slo.begin(), slo.end(), seg); std::copy(shi.begin(), shi.end(), seg + sp.ns); }
    return sp;
}

}  // namespace

extern "C" {

void icpb_default_params(icpb_params *p)
{
    memset(p, 0, sizeof *p);
    p->epsilon = 0.01;
    p->stopping_thresh = 0.0001;
    p->max_iters = 100;
    p->k_block = 1;
}

int icpb_abi_version(void) { return ICPB_ABI_VERSION; }

const char *icpb_last_error(void) { return g_err; }

int icpb_create(int device, icpb_handle *out)
{
    if (!out) return fail(ICPB_EINVAL, "out is null%s");
    *out = nullptr;
    int count = 0;
    CU(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return fail(ICPB_EINVAL, "no such CUDA device%s");
    DeviceGuard guard_(device);
    if (!guard_.ok) return (int)cudaErrorInvalidDevice;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        snprintf(g_err, sizeof g_err, "device %d is sm_%d%d; this library is built for sm_100a only",
                 device, prop.major, prop.minor);
        return ICPB_EINVAL;
    }
    icpb_ctx *h = new (std::nothrow) icpb_ctx();
    if (!h) return fail(ICPB_EINVAL, "out of host memory%s");
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    cudaError_t e = cudaMalloc(&h->queue, sizeof(unsigned long long) * kQueueWords);
    if (e == cudaSuccess) e = cudaMemset(h->queue, 0, sizeof(unsigned long long) * kQueueWords);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaStreamCreateWithFlags(&h->cstream[k], cudaStreamNonBlocking);
    for (cudaEvent_t *ev : {&h->counter_zeroed, &h->inputs_up, &h->kernel_done})
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
    // dynamic shared memory up to the device's opt-in maximum minus each kernel's static part, set
    // once: the attribute belongs to the function, not to a handle.  The large-scan variants keep only
    // a few KB in shared memory but ask for the same maximum; the limit a layout must fit comes from
    // the three shared-memory instances.
    h->smem_limit = (int)prop.sharedMemPerBlockOptin;
    for (int k = 0; k < 6 && e == cudaSuccess; ++k) {
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, kAlignKernels[k]);
        if (e != cudaSuccess) break;
        const int lim = (int)prop.sharedMemPerBlockOptin - (int)fa.sharedSizeBytes;
        e = cudaFuncSetAttribute(kAlignKernels[k], cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
        if (k < 3 && lim < h->smem_limit) h->smem_limit = lim;
    }
    if (e == cudaSuccess) e = cudaMalloc(&h->arrived_dev, sizeof(int32_t));
    if (e == cudaSuccess) e = cudaHostAlloc(&h->seg_vals_pinned, sizeof(int32_t) * (kMaxSegments + 1), cudaHostAllocDefault);
    if (e == cudaSuccess) for (int k = 0; k <= kMaxSegments; ++k) h->seg_vals_pinned[k] = k;
    if (e == cudaSuccess) {
        void *fp = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &fp, cudaEnableDefault, &qr) == cudaSuccess &&
            qr == cudaDriverEntryPointSuccess)
            h->write32 = (int (*)(cudaStream_t, unsigned long long, unsigned int, unsigned int))fp;
        else
            cudaGetLastError();
    }
    if (e != cudaSuccess) {
        icpb_destroy(h);                                      // frees whatever was created so far
        snprintf(g_err, sizeof g_err, "icpb_create: %s", cudaGetErrorString(e));
        return (int)e;
    }
    *out = h;
    return 0;
}

int icpb_set_tuning(icpb_handle h, const char *key, int64_t value)
{
    if (!h || !key) return fail(ICPB_EINVAL, "icpb_set_tuning: bad argument%s");
    const int v = (int)value;
    if (!strcmp(key, "threads")) h->tune_threads = v;
    else if (!strcmp(key, "cluster")) h->tune_cluster = v;
    else if (!strcmp(key, "large")) h->tune_large = v;
    else if (!strcmp(key, "segments")) h->tune_segments = v;
    else if (!strcmp(key, "pack_threads")) {
        if (h->pool && (int)h->pool->workers.size() != v - 1) { delete h->pool; h->pool = nullptr; }
        h->tune_pack_threads = v;
    }
    else if (!strcmp(key, "drop_counter")) h->tune_drop_counter = v != 0;
    else return fail(ICPB_EINVAL, "icpb_set_tuning: unknown key %s", key);
    return 0;
}

int icpb_destroy(icpb_handle h)
{
    if (!h) return 0;
    DeviceGuard guard_(h->device);
    delete h->pool;
    h->pool = nullptr;
    if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
    for (int k = 0; k < 2; ++k) if (h->cstream[k]) { cudaStreamSynchronize(h->cstream[k]); cudaStreamDestroy(h->cstream[k]); }
    for (cudaEvent_t ev : {h->counter_zeroed, h->inputs_up, h->kernel_done}) if (ev) cudaEventDestroy(ev);
    if (h->arrived_dev) cudaFree(h->arrived_dev);
    if (h->seg_vals_pinned) cudaFreeHost(h->seg_vals_pinned);
    h->arena.release(); h->own_xy.release(); h->own_off.release(); h->prep.release(); h->s_big.release();
    h->stage.release(); h->stage_xy.release();
    if (h->queue) cudaFree(h->queue);
    delete h;
    return 0;
}

static int validate_offsets(const int64_t *off, int64_t n_scans, int64_t *longest)
{
    if (off[0] != 0) return fail(ICPB_EINVAL, "offsets[0] must be 0%s");
    int64_t L = 0;
    for (int64_t s = 0; s < n_scans; ++s) {
        const int64_t m = off[s + 1] - off[s];
        if (m <= 0) return fail(ICPB_EINVAL, "empty scan in the table (the reference's argmin raises on it)%s");
        if (m > L) L = m;
    }
    *longest = L;
    return 0;
}

int icpb_upload_scans(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans)
{
    if (!h || !h_xy || !h_offsets || n_scans <= 0) return fail(ICPB_EINVAL, "icpb_upload_scans: bad argument%s");
    int64_t longest = 0;
    int rc = validate_offsets(h_offsets, n_scans, &longest);
    if (rc) return rc;
    ON_DEVICE(h);
    drop_table(h);                                  // reserving may free the old table's memory
    if ((rc = h->own_xy.reserve(sizeof(double) * 2 * (size_t)h_offsets[n_scans]))) return rc;
    if ((rc = h->own_off.reserve(sizeof(int64_t) * (size_t)(n_scans + 1)))) return rc;
    return upload_table(h, h_xy, h_offsets, n_scans, longest);
}

int icpb_set_scans_device(icpb_handle h, const double *d_xy, const int64_t *d_offsets,
                          int64_t n_scans, int64_t longest_scan)
{
    if (!h || !d_xy || !d_offsets || n_scans <= 0 || longest_scan <= 0)
        return fail(ICPB_EINVAL, "icpb_set_scans_device: bad argument%s");
    set_table(h, d_xy, d_offsets, n_scans, longest_scan, nullptr);
    return 0;
}

int icpb_run_device(icpb_handle h, const int32_t *d_pairs, const double *d_init, int64_t B,
                    const icpb_params *p, double *d_T, double *d_err, int32_t *d_passes,
                    double *d_hist, int32_t *d_corr, void *stream)
{
    int rc = run_check(h, p, B, false, d_pairs, d_T, d_err, d_passes, d_hist, d_corr);
    if (rc) return rc;
    ON_DEVICE(h);
    Batch b;
    b.xy = h->xy; b.offsets = h->offsets; b.n_scans = h->n_scans; b.longest = h->longest;
    b.pairs = d_pairs; b.init = d_init; b.B = B; b.p = p;
    b.T = d_T; b.err = d_err; b.passes = d_passes; b.hist = d_hist; b.corr = d_corr;
    b.stream = (cudaStream_t)stream;
    return launch(h, b);
}

int icpb_run_device_ex(icpb_handle h, const int32_t *d_pairs, const double *d_init, int64_t B,
                       const icpb_params *p, double *d_T, double *d_err, int32_t *d_passes,
                       const icpb_epilogue *ep, void *stream)
{
    int rc = check_epilogue(ep);
    // no history or correspondence buffers here: the shared check rejects hist_cap or corr_stride > 0
    if (rc == 0) rc = run_check(h, p, B, false, d_pairs, d_T, d_err, d_passes, nullptr, nullptr);
    if (rc) return rc;
    ON_DEVICE(h);
    Batch b;
    b.xy = h->xy; b.offsets = h->offsets; b.n_scans = h->n_scans; b.longest = h->longest;
    b.pairs = d_pairs; b.init = d_init; b.B = B; b.p = p;
    b.T = d_T; b.err = d_err; b.passes = d_passes;
    b.stream = (cudaStream_t)stream; b.ep = ep;
    return launch(h, b);
}

int icpb_run_device_gather(icpb_handle h, const int32_t *d_pairs, const double *d_init, int64_t B,
                           const icpb_params *p, double *d_T, double *d_err, int32_t *d_passes,
                           const uint64_t *d_peer_ptrs, int32_t n_peers, int64_t row0, void *stream)
{
    if (!d_peer_ptrs) return fail(ICPB_EINVAL, "icpb_run_device_gather: peer buffers expected%s");
    icpb_epilogue ep;
    memset(&ep, 0, sizeof ep);
    ep.d_peer_ptrs = d_peer_ptrs; ep.n_peers = n_peers; ep.row0 = row0;
    return icpb_run_device_ex(h, d_pairs, d_init, B, p, d_T, d_err, d_passes, &ep, stream);
}

// A batch from host buffers on the handle's table (cloud null; host offsets from table_host_offsets if the
// batch is split), or on a table of two clouds that go up with the call (icpb_icp_pair_host: cloud[0],
// cloud[1] at the host offsets off).
static int run_host_common(icpb_handle h, const double *const *cloud, const int64_t *off, int64_t n_scans,
                           int64_t longest, const int32_t *h_pairs, const double *h_init, int64_t B,
                           const icpb_params *p, double *h_T, double *h_err, int32_t *h_passes,
                           double *h_hist, int32_t *h_corr)
{
    int rc;
    cudaStream_t st = h->stream;
    const size_t nbP = sizeof(int32_t) * 2 * (size_t)B, nbI = sizeof(double) * 6 * (size_t)B;
    const size_t nbH = sizeof(double) * 6 * (size_t)B * (size_t)p->hist_cap;
    const size_t nbC = sizeof(int32_t) * (size_t)B * (size_t)p->corr_stride;
    const bool split = needs_split(h, longest, B, p);
    Carve c;
    const size_t o_xy = c(cloud ? sizeof(double) * 2 * (size_t)off[n_scans] : 0);
    const size_t o_off = c(cloud ? sizeof(int64_t) * (size_t)(n_scans + 1) : 0);
    const size_t o_pairs = c(p->pair_mode == 0 ? nbP : 0), o_init = c(h_init ? nbI : 0);
    const size_t o_T = c(nbI), o_err = c(sizeof(double) * (size_t)B), o_passes = c(sizeof(int32_t) * (size_t)B);
    const size_t o_hist = c(nbH), o_corr = c(nbC), o_order = c(split ? sizeof(int32_t) * (size_t)B : 0);
    if ((rc = h->arena.reserve(c.used))) return rc;
    Batch b;
    b.xy = h->xy; b.offsets = h->offsets; b.n_scans = n_scans; b.longest = longest;
    if (cloud) {
        double *xy = at<double>(h->arena, o_xy);
        int64_t *d_off = at<int64_t>(h->arena, o_off);
        CU(cudaMemcpyAsync(xy, cloud[0], sizeof(double) * 2 * (size_t)off[1], cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(xy + 2 * off[1], cloud[1], sizeof(double) * 2 * (size_t)(off[2] - off[1]),
                           cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_off, off, sizeof(int64_t) * (size_t)(n_scans + 1), cudaMemcpyHostToDevice, st));
        b.xy = xy; b.offsets = d_off;
    }
    int32_t *d_pairs = at<int32_t>(h->arena, o_pairs);
    double *d_init = at<double>(h->arena, o_init);
    b.pairs = p->pair_mode == 0 ? d_pairs : nullptr; b.init = h_init ? d_init : nullptr; b.B = B; b.p = p;
    b.T = at<double>(h->arena, o_T); b.err = at<double>(h->arena, o_err); b.passes = at<int32_t>(h->arena, o_passes);
    b.hist = at<double>(h->arena, o_hist); b.corr = at<int32_t>(h->arena, o_corr); b.stream = st;
    if (p->pair_mode == 0) CU(cudaMemcpyAsync(d_pairs, h_pairs, nbP, cudaMemcpyHostToDevice, st));
    if (h_init) CU(cudaMemcpyAsync(d_init, h_init, nbI, cudaMemcpyHostToDevice, st));
    if (nbH) CU(cudaMemsetAsync(b.hist, 0, nbH, st));
    if (nbC) CU(cudaMemsetAsync(b.corr, 0xff, nbC, st));
    Split sp;
    if (split) {
        if (!cloud && (rc = table_host_offsets(h, &off))) return rc;
        std::vector<int32_t> order((size_t)B);
        sp = split_queue(h, off, h_pairs, B, nullptr, order.data(), nullptr);
        int32_t *d_order = at<int32_t>(h->arena, o_order);
        CU(cudaMemcpyAsync(d_order, order.data(), sizeof(int32_t) * (size_t)B, cudaMemcpyHostToDevice, st));
        b.order = d_order; b.split = &sp;
    }
    if ((rc = launch(h, b))) return rc;
    CU(cudaMemcpyAsync(h_T, b.T, nbI, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_err, b.err, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_passes, b.passes, sizeof(int32_t) * (size_t)B, cudaMemcpyDeviceToHost, st));
    if (nbH) CU(cudaMemcpyAsync(h_hist, b.hist, nbH, cudaMemcpyDeviceToHost, st));
    if (nbC) CU(cudaMemcpyAsync(h_corr, b.corr, nbC, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

int icpb_run_host(icpb_handle h, const int32_t *h_pairs, const double *h_init, int64_t B,
                  const icpb_params *p, double *h_T, double *h_err, int32_t *h_passes,
                  double *h_hist, int32_t *h_corr)
{
    int rc = run_check(h, p, B, true, h_pairs, h_T, h_err, h_passes, h_hist, h_corr);
    if (rc || B == 0) return rc;
    if (p->pair_mode == 0 && (rc = check_pairs(h_pairs, B, h->n_scans))) return rc;
    ON_DEVICE(h);
    return run_host_common(h, nullptr, nullptr, h->n_scans, h->longest, h_pairs, h_init, B, p,
                           h_T, h_err, h_passes, h_hist, h_corr);
}

}  // extern "C"

namespace {

// Problems of one multi-start launch: a slice holds floor(kMaxMultistart / K) pairs with all K of their
// starts, so the int32 queue order of a split slice stays in range and its scratch (116 bytes per
// problem: pair, guess, transform, error, passes) within ~490 MB.
constexpr int64_t kMaxMultistart = int64_t(1) << 22;

// Every composed guess G = init[b] . S[k] (the formula of icpb.h, identity for a null init) is within the
// guess bounds, tested as !(|v| <= bound) like check_align_inputs; evaluated in one pass, not stored.
// Contraction is off so that a product is never fused into the sum that follows it.
#if defined(__GNUC__) && !defined(__clang__)
__attribute__((optimize("fp-contract=off")))
#endif
int check_composed(const double *init, int64_t B, const double *S, int32_t K)
{
    static const double kI[6] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0};
    bool bad = false;
    for (int64_t b = 0; b < B; ++b) {
        const double *I = init ? init + 6 * b : kI;
        for (int32_t k = 0; k < K; ++k) {
            const double *s = S + 6 * (int64_t)k;
            for (int r = 0; r < 2; ++r) {
                const double a = I[3 * r], c = I[3 * r + 1], t = I[3 * r + 2];
                const double p0 = a * s[0], q0 = c * s[3], p1 = a * s[1], q1 = c * s[4];
                const double p2 = a * s[2], q2 = c * s[5];
                const double g0 = p0 + q0, g1 = p1 + q1, g2 = (p2 + q2) + t;
                bad |= !(fabs(g0) <= ICPB_MAX_GUESS_LINEAR) | !(fabs(g1) <= ICPB_MAX_GUESS_LINEAR) |
                       !(fabs(g2) <= ICPB_MAX_GUESS_SHIFT);
            }
        }
    }
    if (bad) return fail(ICPB_EINVAL, "a composed guess init . start holds non-finite values or values beyond the bounds of icpb.h%s");
    return 0;
}

int run_multistart(icpb_ctx *h, const int32_t *h_pairs, const double *h_init, int64_t B, const double *h_starts,
                   int32_t K, const icpb_params *p_in, double *h_T, double *h_err, int32_t *h_passes, int32_t *h_start,
                   double *h_err_all, int32_t *h_passes_all)
{
    int rc;
    cudaStream_t st = h->stream;
    const int64_t per = kMaxMultistart / K;                           // pairs per slice
    const int64_t n_max = B < per ? B : per, q_max = n_max * K;
    // a slice's pairs, guesses, queue order and results, the K starts, then the slice's expanded problems
    // (a queue order only on a table that may be split: split_queue)
    Carve c;
    const size_t o_pairs = c(8 * (size_t)n_max), o_init = c(h_init ? 48 * (size_t)n_max : 0);
    const size_t o_order = c(4 * (size_t)n_max), o_starts = c(48 * (size_t)K);
    const size_t o_T = c(48 * (size_t)n_max), o_err = c(8 * (size_t)n_max);
    const size_t o_passes = c(4 * (size_t)n_max), o_start = c(4 * (size_t)n_max);
    const size_t o_epairs = c(8 * (size_t)q_max), o_eG = c(48 * (size_t)q_max), o_eT = c(48 * (size_t)q_max);
    const size_t o_eerr = c(8 * (size_t)q_max), o_epasses = c(4 * (size_t)q_max);
    const size_t o_eorder = c(fits_smem(h, h->longest) ? 0 : 4 * (size_t)q_max);
    if ((rc = h->arena.reserve(c.used))) return rc;
    int32_t *d_pairs = at<int32_t>(h->arena, o_pairs), *d_order = at<int32_t>(h->arena, o_order);
    double *d_init = h_init ? at<double>(h->arena, o_init) : nullptr, *d_starts = at<double>(h->arena, o_starts);
    double *d_T = at<double>(h->arena, o_T), *d_err = at<double>(h->arena, o_err);
    int32_t *d_passes = at<int32_t>(h->arena, o_passes), *d_start = at<int32_t>(h->arena, o_start);
    int32_t *epairs = at<int32_t>(h->arena, o_epairs), *epasses = at<int32_t>(h->arena, o_epasses);
    double *eG = at<double>(h->arena, o_eG), *eT = at<double>(h->arena, o_eT), *eerr = at<double>(h->arena, o_eerr);
    int32_t *eorder = at<int32_t>(h->arena, o_eorder);
    CU(cudaMemcpyAsync(d_starts, h_starts, 48 * (size_t)K, cudaMemcpyHostToDevice, st));
    icpb_params p = *p_in;
    p.k_first = 0; p.k_stride = 0;
    std::vector<int32_t> pair_order;
    for (int64_t p0 = 0; p0 < B; p0 += per) {
        const int64_t n = B - p0 < per ? B - p0 : per, nq = n * K;
        p.k_block = nq;
        CU(cudaMemcpyAsync(d_pairs, h_pairs + 2 * p0, 8 * (size_t)n, cudaMemcpyHostToDevice, st));
        if (h_init) CU(cudaMemcpyAsync(d_init, h_init + 6 * p0, 48 * (size_t)n, cudaMemcpyHostToDevice, st));
        Split sp;
        const bool split = needs_split(h, h->longest, nq, &p);
        if (split) {
            const int64_t *off;
            if ((rc = table_host_offsets(h, &off))) return rc;
            // the slice's pairs in queue order; the expansion turns every pair into its K problems
            pair_order.resize((size_t)n);
            const Split ps = split_queue(h, off, h_pairs + 2 * p0, n, nullptr, pair_order.data(), nullptr);
            sp.ns = ps.ns * K; sp.Ls = ps.Ls; sp.Ll = ps.Ll;
            CU(cudaMemcpyAsync(d_order, pair_order.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, st));
        }
        int64_t blocks = (nq + icpb::kMultistartThreads - 1) / icpb::kMultistartThreads;
        if (blocks > 16 * (int64_t)h->sm_count) blocks = 16 * (int64_t)h->sm_count;
        icpb::multistart_expand_kernel<<<(unsigned)blocks, icpb::kMultistartThreads, 0, st>>>(
            d_pairs, d_init, d_starts, K, n, split ? d_order : nullptr, epairs, eG, split ? eorder : nullptr);
        CU(cudaGetLastError());
        Batch b;
        b.xy = h->xy; b.offsets = h->offsets; b.n_scans = h->n_scans; b.longest = h->longest;
        b.pairs = epairs; b.init = eG; b.B = nq; b.p = &p;
        b.T = eT; b.err = eerr; b.passes = epasses; b.stream = st;
        if (split) { b.order = eorder; b.split = &sp; }
        if ((rc = launch(h, b))) return rc;
        blocks = (n + icpb::kMultistartThreads - 1) / icpb::kMultistartThreads;
        if (blocks > 16 * (int64_t)h->sm_count) blocks = 16 * (int64_t)h->sm_count;
        icpb::multistart_select_kernel<<<(unsigned)blocks, icpb::kMultistartThreads, 0, st>>>(
            eT, eerr, epasses, K, n, d_T, d_err, d_passes, d_start);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(h_T + 6 * p0, d_T, 48 * (size_t)n, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_err + p0, d_err, 8 * (size_t)n, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_passes + p0, d_passes, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_start + p0, d_start, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
        // problem p_local * K + k is row p, column k of the (B, K) arrays
        if (h_err_all) CU(cudaMemcpyAsync(h_err_all + p0 * K, eerr, 8 * (size_t)nq, cudaMemcpyDeviceToHost, st));
        if (h_passes_all) CU(cudaMemcpyAsync(h_passes_all + p0 * K, epasses, 4 * (size_t)nq, cudaMemcpyDeviceToHost, st));
        // the next slice overwrites the scratch: its copies are enqueued behind these on the same stream
    }
    CU(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace

extern "C" {

int icpb_run_multistart_host(icpb_handle h, const int32_t *h_pairs, const double *h_init, int64_t B,
                             const double *h_starts, int32_t K, const icpb_params *p,
                             double *h_T, double *h_err, int32_t *h_passes, int32_t *h_start,
                             double *h_err_all, int32_t *h_passes_all)
{
    if (!h) return fail(ICPB_EINVAL, "handle is null%s");
    if (!p) return fail(ICPB_EINVAL, "params is null%s");
    if (p->hist_cap > 0 || p->corr_stride > 0)
        return fail(ICPB_EINVAL, "multi-start runs record no history or correspondences: rerun icpb_run_host on "
                                 "the winning guesses for them%s");
    if (p->pair_mode != 0) return fail(ICPB_EINVAL, "multi-start runs take explicit pairs (pair_mode 0)%s");
    if (K < 1 || K > kMaxMultistart) return fail(ICPB_EINVAL, "the number of starts must be in 1 .. 2^22%s");
    if (!h_starts) return fail(ICPB_EINVAL, "starts is null%s");
    int rc = run_check(h, p, B, true, h_pairs, h_T, h_err, h_passes, nullptr, nullptr);
    if (rc || B == 0) return rc;
    if (!h_start) return fail(ICPB_EINVAL, "output pointer is null%s");
    if ((rc = check_pairs(h_pairs, B, h->n_scans))) return rc;
    if ((rc = check_composed(h_init, B, h_starts, K))) return rc;
    ON_DEVICE(h);
    return run_multistart(h, h_pairs, h_init, B, h_starts, K, p, h_T, h_err, h_passes, h_start,
                          h_err_all, h_passes_all);
}

/* Upload + align with the upload hidden behind the kernels: the scan table goes up in segments on
 * the copy stream; pairs are grouped by the segment that completes them (the larger of their two
 * scan ids) and every group is launched as soon as its segment has arrived. */
/* Pieces of the streaming scan-table upload (pure host logic, no CUDA call).
 * Equal pieces of about 4 MB, at most 16 by default (the first pairs start ~0.1 ms into the upload;
 * the kernel is launched before any piece has arrived and its CTAs wait on the counter).  Measured on
 * the 81 MB chain table with counter copies: 4 pieces 2.49 ms, 16 2.35 ms, 32 2.55 ms, 64 2.86 ms per
 * call; with cuStreamWriteValue32 16 and 32 pieces cost the same.
 * A piece must end on a 32-byte sector boundary (an even point offset): the kernel reads scans
 * through L1, and a sector that straddled two pieces could be cached while its second half had not
 * arrived yet.  Boundaries on a 128-byte line (offset % 8 == 0) are preferred when one is near; a
 * wanted boundary with no even offset within 64 scans is dropped (its piece merges with the next). */
int icpb_plan_upload(const int64_t *h_offsets, int64_t n_scans, int32_t pieces_wanted,
                     int64_t *piece_end, int32_t *n_pieces)
{
    if (!h_offsets || n_scans <= 0 || !piece_end || !n_pieces)
        return fail(ICPB_EINVAL, "icpb_plan_upload: bad argument%s");
    const int64_t total = h_offsets[n_scans];
    const size_t nb_xy = sizeof(double) * 2 * (size_t)total;
    int nseg = (int)(nb_xy / (4u << 20)) + 1;
    if (nseg > 16) nseg = 16;
    // Default plan: the first two and the last two pieces are a quarter and a half of a standard
    // piece, so the first bytes are on the wire (and the first pairs running) sooner and fewer pairs
    // are left waiting for the last piece.  An explicit piece count gives equal pieces.
    const bool graded = !(pieces_wanted >= 1 && pieces_wanted <= kMaxSegments) && nseg >= 8;
    if (graded) nseg += 2;
    if (pieces_wanted >= 1 && pieces_wanted <= kMaxSegments) nseg = pieces_wanted;
    if (nseg > n_scans) nseg = (int)n_scans;
    double cum[kMaxSegments + 1];
    cum[0] = 0.0;
    for (int k = 0; k < nseg; ++k) {
        double w = 1.0;
        if (graded && (k == 0 || k == nseg - 1)) w = 0.25;
        if (graded && (k == 1 || k == nseg - 2)) w = 0.5;
        cum[k + 1] = cum[k] + w;
    }
    int64_t s = 0;
    int made = 0;
    for (int k = 0; k < nseg - 1; ++k) {
        const int64_t want = (int64_t)((double)total * (cum[k + 1] / cum[nseg]));
        while (s < n_scans && h_offsets[s] < want) ++s;
        int64_t pick = -1;
        for (int64_t c = s; c < n_scans && c < s + 64; ++c) {
            if (h_offsets[c] % 8 == 0) { pick = c; break; }
            if (pick < 0 && h_offsets[c] % 2 == 0) pick = c;
        }
        if (pick <= 0 || pick >= n_scans || (made > 0 && pick <= piece_end[made - 1])) continue;   // merge with the next piece
        piece_end[made++] = pick;
        s = pick;
    }
    piece_end[made++] = n_scans;
    *n_pieces = made;
    return 0;
}

namespace {

// Where icpb_align_host*'s scan table comes from: one packed (sum m_i, 2) array with its offsets, or the
// reference's own `lidar_points` form -- a list of separate (m_i, 2) arrays in pageable memory.
struct TableSrc {
    const double *xy = nullptr;                 // packed form
    const int64_t *offsets = nullptr;           // n_scans + 1 (computed from the lengths for the list form)
    const double *const *scan_xy = nullptr;     // list form
};

// Everything that was enqueued is drained before an error is reported, and the handle is left without
// a table: its buffer may hold a mixture of the old and the new scans.
int align_abort(icpb_ctx *h, int rc)
{
    char keep[sizeof g_err];
    memcpy(keep, g_err, sizeof keep);
    cudaStreamSynchronize(h->stream); cudaStreamSynchronize(h->cstream[0]); cudaStreamSynchronize(h->cstream[1]);
    cudaGetLastError();
    memcpy(g_err, keep, sizeof keep);
    drop_table(h);
    return rc;
}
#define CUA(call)                                                                         \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            snprintf(g_err, sizeof g_err, "%s failed: %s", #call, cudaGetErrorString(e_)); \
            return align_abort(h, (int)e_);                                               \
        }                                                                                 \
    } while (0)

int host_threads_available()
{
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof set, &set) == 0) {
        const int n = CPU_COUNT(&set);
        if (n > 0) return n;
    }
    const unsigned n = std::thread::hardware_concurrency();
    return n > 0 ? (int)n : 1;
}

// icpb_align_host_accept: only the pairs that pass the acceptance test come back to the host
struct AcceptHost {
    double thresh;
    int64_t cap;
    int64_t *n_out, *rows;
    double *T;
    int32_t T_ld;
    double *err;
    int32_t *passes;
};

// The caller's pairs and initial guesses (init_ld 6: 2x3 rows, 9: 3x3 matrices).  icpb_align_host* checks
// them before any state of the handle changes: a rejected call leaves the old table usable.
int check_align_inputs(const int32_t *pairs, const double *init, int32_t init_ld, int64_t B, int64_t n_scans)
{
    int rc = check_pairs(pairs, B, n_scans);
    if (rc || !init || B == 0) return rc;
    for (int64_t b = 0; b < B && init_ld == 9; ++b) {
        const double *m = init + 9 * b;
        if (!(m[6] == 0.0 && m[7] == 0.0 && m[8] == 1.0))
            return fail(ICPB_EINVAL, "transform bottom row must be [0, 0, 1] (an SE(2) matrix)%s");
    }
    bool bad = false;                                         // !(|v| <= bound): NaN fails too
    for (int64_t b = 0; b < B; ++b) {
        const double *m = init + (int64_t)init_ld * b;
        bad |= !(fabs(m[0]) <= ICPB_MAX_GUESS_LINEAR) | !(fabs(m[1]) <= ICPB_MAX_GUESS_LINEAR) |
               !(fabs(m[3]) <= ICPB_MAX_GUESS_LINEAR) | !(fabs(m[4]) <= ICPB_MAX_GUESS_LINEAR) |
               !(fabs(m[2]) <= ICPB_MAX_GUESS_SHIFT) | !(fabs(m[5]) <= ICPB_MAX_GUESS_SHIFT);
    }
    if (bad) return fail(ICPB_EINVAL, "transform holds non-finite values or values beyond the bounds of icpb.h%s");
    return 0;
}

// The list form of the scan table: host threads (the handle's PackPool and the calling thread) pack the
// caller's arrays into the pinned staging table, every upload piece split into one run of scans per thread.
// The workers write through this object, which lives on the calling frame: the destructor stops them on
// every way out of the call.
struct ListPacker {
    PackJob job;
    std::vector<int64_t> job_first, job_last;
    std::vector<int32_t> job_piece;
    int32_t jobs_of_piece[kMaxSegments];
    std::atomic<int32_t> piece_done[kMaxSegments];
    PackPool *pool = nullptr;                           // set while its workers may be running `job`

    void start(icpb_ctx *h, const double *const *scan_xy, const int64_t *offsets, double *dst,
               const int64_t *seg_end, int nseg)
    {
        const int nthr = h->tune_pack_threads > 0 ? std::min(h->tune_pack_threads, 32)
                                                  : std::min(host_threads_available(), 8);   // default: at most 8
        if (!h->pool && nthr > 1) h->pool = new (std::nothrow) PackPool(nthr - 1);
        int64_t s0 = 0;
        for (int k = 0; k < nseg; ++k) {
            const int64_t s1 = seg_end[k], n = s1 - s0;
            const int parts = (int)(n < nthr ? n : nthr);
            for (int q = 0; q < parts; ++q) {
                job_first.push_back(s0 + n * q / parts); job_last.push_back(s0 + n * (q + 1) / parts);
                job_piece.push_back(k);
            }
            jobs_of_piece[k] = parts;
            piece_done[k].store(0, std::memory_order_relaxed);
            s0 = s1;
        }
        job.scan_xy = scan_xy; job.offsets = offsets; job.dst = dst;
        job.job_first = job_first.data(); job.job_last = job_last.data(); job.job_piece = job_piece.data();
        job.n_jobs = (int64_t)job_first.size(); job.done = piece_done;
        pool = h->pool;
        if (pool) pool->start(&job);
    }
    // Returns once piece k is packed; this thread packs too while it waits.  true: a bad coordinate was seen.
    bool wait_piece(int k)
    {
        while (piece_done[k].load(std::memory_order_acquire) < jobs_of_piece[k]) {
            const int64_t j = job.next.fetch_add(1, std::memory_order_relaxed);
            if (j < job.n_jobs) pack_one(&job, j);
        }
        return job.bad.load(std::memory_order_relaxed) != 0;
    }
    // Hands out no more jobs and waits for the workers.  true: a bad coordinate was seen.
    bool finish()
    {
        job.next.store(job.n_jobs, std::memory_order_relaxed);
        if (pool) pool->finish();
        pool = nullptr;
        return job.bad.load() != 0;
    }
    ~ListPacker() { finish(); }
};

// Piece k of the streaming upload (scans [seg_end[k-1], seg_end[k]) of xy), then the arrival counter's new
// value k + 1, in stream order: the counter changes after the piece it announces has landed.
cudaError_t enqueue_piece(icpb_ctx *h, const double *xy, const int64_t *off, const int64_t *seg_end, int k)
{
    const int64_t o0 = off[k ? seg_end[k - 1] : 0], o1 = off[seg_end[k]];
    cudaError_t e = cudaSuccess;
    if (o1 > o0)
        e = cudaMemcpyAsync((double *)h->own_xy.p + 2 * o0, xy + 2 * o0, sizeof(double) * 2 * (size_t)(o1 - o0),
                            cudaMemcpyHostToDevice, h->stream);
    // (drop_counter, tests only: the kernel must time out and the batch be rerun.)  Without
    // cuStreamWriteValue32, or when it fails, the counter is copied.
    if (e == cudaSuccess && !h->tune_drop_counter &&
        (!h->write32 || h->write32(h->stream, (unsigned long long)(uintptr_t)h->arrived_dev, (unsigned)(k + 1), 0) != 0))
        e = cudaMemcpyAsync(h->arrived_dev, h->seg_vals_pinned + (k + 1), sizeof(int32_t), cudaMemcpyHostToDevice,
                            h->stream);
    return e;
}

// Queue order of a streamed batch: pairs grouped by the piece that completes them (the later of their two
// scans); the pairs, guesses and results themselves stay in the caller's order.  pseg[q]: the piece of the
// pair at queue position q, porder[q]: that pair, unless the batch already comes in arrival order (the
// odometry chain does).  A table whose longest scan does not fit shared memory splits the queue by scan
// length, each part keeping its arrival order.  scratch: B words.
struct QueueOrder {
    bool in_order = true;                               // queue position = pair id
    bool split = false;                                 // porder holds the split queue, sp its parts
    Split sp;
};

QueueOrder order_queue(icpb_ctx *h, const int64_t *off, int64_t n_scans, int64_t longest, const int64_t *seg_end,
                       int nseg, const int32_t *pairs, int64_t B, const icpb_params *p, int32_t *scratch,
                       int32_t *porder, int32_t *pseg)
{
    QueueOrder qo;
    std::vector<int32_t> seg_of_scan((size_t)n_scans);
    for (int64_t sc = 0, k = 0; sc < n_scans; ++sc) { while (sc >= seg_end[k]) ++k; seg_of_scan[sc] = (int32_t)k; }
    int32_t *seg_of_pair = scratch;
    int32_t prev = 0, sorted = 1;
    for (int64_t b = 0; b < B; ++b) {
        const int32_t i = pairs[2 * b], j = pairs[2 * b + 1];
        const int32_t sg = seg_of_scan[i > j ? i : j];
        seg_of_pair[b] = sg;
        sorted &= (int32_t)(sg >= prev);
        prev = sg;
    }
    qo.in_order = sorted != 0;
    if (qo.in_order) {
        memcpy(pseg, seg_of_pair, sizeof(int32_t) * (size_t)B);
    } else {                                                  // stable counting sort
        int64_t start[kMaxSegments + 1] = {0};
        for (int64_t b = 0; b < B; ++b) ++start[seg_of_pair[b] + 1];
        for (int k = 0; k < nseg; ++k) start[k + 1] += start[k];
        for (int64_t b = 0; b < B; ++b) {
            const int64_t q = start[seg_of_pair[b]]++;
            porder[q] = (int32_t)b; pseg[q] = seg_of_pair[b];
        }
    }
    qo.split = needs_split(h, longest, B, p);
    if (qo.split) {
        const std::vector<int32_t> queue(porder, porder + (qo.in_order ? 0 : B));
        qo.sp = split_queue(h, off, pairs, B, qo.in_order ? nullptr : queue.data(), porder, pseg);
        qo.in_order = false;
    }
    return qo;
}

// n transforms of 6 doubles (the top two rows) into rows of ld doubles: 6 (2x3) or 9 (3x3, bottom row [0, 0, 1]).
void put_transforms(double *dst, int32_t ld, const double *t6, int64_t n)
{
    if (ld == 6) { memcpy(dst, t6, sizeof(double) * 6 * (size_t)n); return; }
    for (int64_t b = 0; b < n; ++b) {
        double *m = dst + 9 * b;
        memcpy(m, t6 + 6 * b, 6 * sizeof(double));
        m[6] = 0.0; m[7] = 0.0; m[8] = 1.0;
    }
}

// The inverse of put_transforms: the top two rows of n transforms of ld (6 or 9) doubles, as 6 doubles each.
void get_transforms(double *t6, const double *src, int32_t ld, int64_t n)
{
    if (ld == 6) { memcpy(t6, src, sizeof(double) * 6 * (size_t)n); return; }
    for (int64_t b = 0; b < n; ++b) memcpy(t6 + 6 * b, src + 9 * b, 6 * sizeof(double));
}

// align_impl's two per-pair blocks, each sent in one copy, at the same offsets in the pinned staging and in
// its device mirror:  up = [init | pairs | seg | order],  down = [T | err | passes | timeout word], 8-byte
// members first; after them the accepted count of icpb_align_host_accept.
struct AlignBlocks {
    struct Ptrs {
        double *init; int32_t *pairs, *seg, *order;
        double *T, *err; int32_t *passes, *timeout;
        int64_t *accepted;
    };
    size_t init = 0, pairs, seg, order, up;                  // up: the end of the up block
    size_t T, err, passes, timeout, down, accepted, bytes;   // down: bytes of the down block, T to timeout
    explicit AlignBlocks(int64_t B)
    {
        const size_t n = (size_t)B;
        pairs = init + sizeof(double) * 6 * n; seg = pairs + sizeof(int32_t) * 2 * n;
        order = seg + sizeof(int32_t) * n; up = order + sizeof(int32_t) * n;
        T = up; err = T + sizeof(double) * 6 * n; passes = err + sizeof(double) * n;
        timeout = passes + sizeof(int32_t) * n; down = timeout + sizeof(int32_t) - T;
        accepted = (timeout + sizeof(int32_t) + 7) & ~size_t(7); bytes = accepted + sizeof(int64_t);
    }
    Ptrs ptrs(void *base) const
    {
        unsigned char *b = (unsigned char *)base;
        return {(double *)(b + init), (int32_t *)(b + pairs), (int32_t *)(b + seg), (int32_t *)(b + order),
                (double *)(b + T), (double *)(b + err), (int32_t *)(b + passes), (int32_t *)(b + timeout),
                (int64_t *)(b + accepted)};
    }
};

// icpb_align_host_accept's results: the n records the kernel appended at d_rec as pairs finished (n < 0: more
// pairs passed than the capacity, and -n of them), fetched and put in ascending pair order.
int deliver_accepted(const AcceptHost *acc, const double *d_rec, int64_t n, cudaStream_t st)
{
    *acc->n_out = n < 0 ? -n : n;
    if (n < 0) return fail(ICPB_EINVAL, "icpb_align_host_accept: more pairs accepted than the capacity given%s");
    std::vector<double> rec(8 * (size_t)n);
    if (n > 0) {
        CU(cudaMemcpyAsync(rec.data(), d_rec, sizeof(double) * 8 * (size_t)n, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    std::vector<int64_t> idx((size_t)n);
    for (int64_t k = 0; k < n; ++k) idx[(size_t)k] = k;
    auto tag_of = [&](int64_t k) { int64_t t; memcpy(&t, &rec[8 * (size_t)k + 7], sizeof t); return t; };
    std::sort(idx.begin(), idx.end(), [&](int64_t x, int64_t y) { return (tag_of(x) >> 16) < (tag_of(y) >> 16); });
    for (int64_t q = 0; q < n; ++q) {
        const double *r = &rec[8 * (size_t)idx[(size_t)q]];
        const int64_t tag = tag_of(idx[(size_t)q]);
        acc->rows[q] = tag >> 16;
        acc->passes[q] = (int32_t)(tag & 0xffff);
        acc->err[q] = r[6];
        put_transforms(acc->T + (size_t)acc->T_ld * q, acc->T_ld, r, 1);
    }
    return 0;
}

// Every pair's results, from the pinned down block into the caller's arrays.
void deliver_all(const AlignBlocks::Ptrs &pin, int64_t B, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes)
{
    put_transforms(h_T, T_ld, pin.T, B);
    memcpy(h_err, pin.err, sizeof(double) * (size_t)B);
    memcpy(h_passes, pin.passes, sizeof(int32_t) * (size_t)B);
}

// A call without pairs: the table goes up whole (planned as one piece), and the handle owns it once it has landed.
int upload_only(icpb_ctx *h, const TableSrc &src, ListPacker &packer, const double *up_xy, int64_t n_scans,
                int64_t longest)
{
    if (src.scan_xy) packer.wait_piece(0);
    if (packer.finish())                                      // before the table goes up
        return align_abort(h, fail(ICPB_EINVAL, "scan table holds non-finite coordinates or coordinates beyond ICPB_MAX_COORD%s"));
    const int rc = upload_table(h, up_xy, src.offsets, n_scans, longest);
    return rc ? align_abort(h, rc) : 0;
}

int align_impl(icpb_handle h, const TableSrc &src, int64_t n_scans, int64_t longest,
               const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
               const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes,
               const icpb_epilogue *ep, const AcceptHost *acc = nullptr)
{
    const int64_t *h_offsets = src.offsets;
    int rc;
    ON_DEVICE(h);
    const size_t nb_xy = sizeof(double) * 2 * (size_t)h_offsets[n_scans];
    const size_t nb_off = sizeof(int64_t) * (size_t)(n_scans + 1);
    if (src.scan_xy && (rc = h->stage_xy.reserve(nb_xy))) return rc;
    int nseg = 0;
    int64_t seg_end[kMaxSegments];                            // exclusive scan id
    if ((rc = icpb_plan_upload(h_offsets, n_scans, B == 0 ? 1 : h->tune_segments, seg_end, &nseg))) return rc;
    // the per-pair blocks, pinned and on the device; on the device also the accepted records
    const AlignBlocks blk(B);
    Carve c;
    const size_t o_blk = c(blk.bytes), o_rec = c(acc ? sizeof(double) * 8 * (size_t)acc->cap : 0);
    if ((rc = h->stage.reserve(blk.bytes))) return rc;
    if ((rc = h->arena.reserve(c.used))) return rc;
    unsigned char *pin_base = (unsigned char *)h->stage.p, *dev_base = at<unsigned char>(h->arena, o_blk);
    const AlignBlocks::Ptrs pin = blk.ptrs(pin_base), dev = blk.ptrs(dev_base);
    double *d_rec = at<double>(h->arena, o_rec);
    icpb_epilogue ep_acc;
    if (acc) {
        // acceptance on the device: compact records and their count, fetched at the end
        if (ep) ep_acc = *ep; else memset(&ep_acc, 0, sizeof ep_acc);
        ep_acc.accept_thresh = acc->thresh; ep_acc.accept_cap = acc->cap;
        ep_acc.d_accept_count = dev.accepted;
        ep_acc.d_accept_rec = d_rec;
        ep_acc.d_accept_peer_ptrs = nullptr; ep_acc.d_accept_count_peer_ptrs = nullptr;
        ep = &ep_acc;
    }

    // The packers (list input) start now, so they work while the caller's pairs and initial guesses are checked
    ListPacker packer;
    const double *up_xy = src.scan_xy ? (const double *)h->stage_xy.p : src.xy;
    if (src.scan_xy) packer.start(h, src.scan_xy, h_offsets, (double *)h->stage_xy.p, seg_end, nseg);
    if ((rc = check_align_inputs(h_pairs, h_init, init_ld, B, n_scans))) return rc;
    // ---- from here on the handle's table is being replaced: a failure leaves it without one ----
    drop_table(h);
    if ((rc = h->own_xy.reserve(nb_xy))) return rc;
    if ((rc = h->own_off.reserve(nb_off))) return rc;
    if (B == 0) return upload_only(h, src, packer, up_xy, n_scans, longest);
    cudaStream_t cp = h->stream, cp2 = h->cstream[1], cs = h->cstream[0];
    // The first pieces start NOW, before the per-pair staging below: the copy engine works while the
    // host sorts and packs (everything has been validated above; nothing below can fail on user input).
    CUA(cudaMemsetAsync(h->arrived_dev, 0, sizeof(int32_t), cp));
    CUA(cudaEventRecord(h->counter_zeroed, cp));              // the counter is zero before the kernel may start
    int n_sent = 0;
    if (!src.scan_xy)
        for (; n_sent < (nseg < 4 ? nseg : 4); ++n_sent) CUA(enqueue_piece(h, up_xy, h_offsets, seg_end, n_sent));
    const QueueOrder qo = order_queue(h, h_offsets, n_scans, longest, seg_end, nseg, h_pairs, B, p,
                                      pin.passes /* the down block is free until the end */, pin.order, pin.seg);
    memcpy(pin.pairs, h_pairs, sizeof(int32_t) * 2 * (size_t)B);
    if (h_init) get_transforms(pin.init, h_init, init_ld, B);
    // the up block goes on a second copy stream, beside the pieces already in flight: from the guesses (or the
    // pairs) to the piece numbers (or the queue order)
    CUA(cudaMemsetAsync(dev.timeout, 0, sizeof(int32_t), cp2));
    CUA(cudaMemcpyAsync(h->own_off.p, h_offsets, nb_off, cudaMemcpyHostToDevice, cp2));
    const size_t up0 = h_init ? blk.init : blk.pairs, up1 = qo.in_order ? blk.order : blk.up;
    CUA(cudaMemcpyAsync(dev_base + up0, pin_base + up0, up1 - up0, cudaMemcpyHostToDevice, cp2));
    CUA(cudaEventRecord(h->inputs_up, cp2));
    // ONE launch over all pairs, in arrival order; its CTAs wait on the segment counter
    CUA(cudaStreamWaitEvent(cs, h->inputs_up, 0));
    CUA(cudaStreamWaitEvent(cs, h->counter_zeroed, 0));
    Batch bt;
    bt.xy = (const double *)h->own_xy.p; bt.offsets = (const int64_t *)h->own_off.p; bt.n_scans = n_scans;
    bt.longest = longest; bt.pairs = dev.pairs; bt.init = h_init ? dev.init : nullptr; bt.B = B; bt.p = p;
    bt.T = dev.T; bt.err = dev.err; bt.passes = dev.passes;
    bt.stream = cs; bt.ep = ep; bt.order = qo.in_order ? nullptr : dev.order;
    bt.seg_of_pair = dev.seg; bt.arrived = h->arrived_dev; bt.upload_timeout = dev.timeout;
    bt.split = qo.split ? &qo.sp : nullptr;
    if ((rc = launch(h, bt))) return align_abort(h, rc);
    for (int k = n_sent; k < nseg; ++k) {
        if (src.scan_xy && packer.wait_piece(k)) break;       // a bad scan: no further piece goes up
        CUA(enqueue_piece(h, up_xy, h_offsets, seg_end, k));
    }
    if (packer.finish()) {
        // the kernel is waiting for pieces that will not come: raise its give-up flag, drain, report
        CUA(cudaMemcpyAsync(dev.timeout, h->seg_vals_pinned + 1, sizeof(int32_t), cudaMemcpyHostToDevice, cp));
        return align_abort(h, fail(ICPB_EINVAL, "scan table holds non-finite coordinates or coordinates beyond ICPB_MAX_COORD%s"));
    }
    CUA(cudaEventRecord(h->kernel_done, cs));
    CUA(cudaStreamWaitEvent(cp, h->kernel_done, 0));
    if (!acc) {
        CUA(cudaMemcpyAsync(pin.T, dev.T, blk.down, cudaMemcpyDeviceToHost, cp));
    } else {                                                  // the timeout word and the count, not the results
        CUA(cudaMemcpyAsync(pin.timeout, dev.timeout, sizeof(int32_t), cudaMemcpyDeviceToHost, cp));
        CUA(cudaMemcpyAsync(pin.accepted, dev.accepted, sizeof(int64_t), cudaMemcpyDeviceToHost, cp));
    }
    CUA(cudaStreamSynchronize(cp));
    if (*pin.timeout != 0) {
        // a CTA gave up waiting for its scans (see the kernel): by now the whole table is resident,
        // so run the batch again without the streaming protocol
        Batch again = bt;
        again.seg_of_pair = nullptr; again.arrived = nullptr; again.upload_timeout = nullptr;
        again.stream = cp;
        if ((rc = launch(h, again))) return align_abort(h, rc);
        if (!acc) CUA(cudaMemcpyAsync(pin.T, dev.T, blk.down, cudaMemcpyDeviceToHost, cp));
        else      CUA(cudaMemcpyAsync(pin.accepted, dev.accepted, sizeof(int64_t), cudaMemcpyDeviceToHost, cp));
        CUA(cudaStreamSynchronize(cp));
    }
    // only now does the handle own the new table
    set_table(h, bt.xy, bt.offsets, n_scans, longest, h_offsets);
    if (acc) return deliver_accepted(acc, d_rec, *pin.accepted, cp);
    deliver_all(pin, B, h_T, T_ld, h_err, h_passes);
    return 0;
}

int align_check(icpb_handle h, int64_t n_scans, const int32_t *h_pairs, int32_t init_ld, int64_t B,
                const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes,
                const icpb_epilogue *ep)
{
    if (!h || n_scans <= 0) return fail(ICPB_EINVAL, "icpb_align_host: bad argument%s");
    if ((init_ld != 6 && init_ld != 9) || (T_ld != 6 && T_ld != 9))
        return fail(ICPB_EINVAL, "icpb_align_host: init_ld / T_ld must be 6 (2x3 rows) or 9 (3x3)%s");
    int rc = check_params(p, B);
    if (rc) return rc;
    if ((rc = check_epilogue(ep))) return rc;
    if (p->pair_mode != 0 || p->hist_cap > 0 || p->corr_stride > 0)
        return fail(ICPB_EINVAL, "icpb_align_host: explicit pairs, no history/correspondences (use upload + run)%s");
    if (B >= (int64_t(1) << 31)) return fail(ICPB_EINVAL, "icpb_align_host: at most 2^31 - 1 pairs per call%s");
    if (B > 0 && (!h_pairs || !h_T || !h_err || !h_passes)) return fail(ICPB_EINVAL, "null pointer%s");
    return 0;
}

// The scan table of an icpb_align_host* call, packed (xy + off) or as a list of arrays (scan_xy +
// scan_len; its offsets are computed into `offsets`, which src then points to).
int table_src(const double *xy, const int64_t *off, const double *const *scan_xy, const int64_t *scan_len,
              int64_t n_scans, std::vector<int64_t> &offsets, TableSrc *src, int64_t *longest)
{
    if (xy && off) {
        src->xy = xy; src->offsets = off;
        return validate_offsets(off, n_scans, longest);
    }
    if (!scan_xy || !scan_len) return fail(ICPB_EINVAL, "icpb_align_host: no scans (xy + offsets or a list of arrays)%s");
    offsets.resize((size_t)n_scans + 1);
    offsets[0] = 0;
    *longest = 0;
    for (int64_t s = 0; s < n_scans; ++s) {
        if (!scan_xy[s] || scan_len[s] <= 0)
            return fail(ICPB_EINVAL, "empty scan in the list (the reference's argmin raises on it)%s");
        offsets[(size_t)s + 1] = offsets[(size_t)s] + scan_len[s];
        if (scan_len[s] > *longest) *longest = scan_len[s];
    }
    src->scan_xy = scan_xy; src->offsets = offsets.data();
    return 0;
}

}  // namespace

int icpb_align_host_ex(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans,
                       const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                       const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes,
                       const icpb_epilogue *ep)
{
    int rc = align_check(h, n_scans, h_pairs, init_ld, B, p, h_T, T_ld, h_err, h_passes, ep);
    if (rc) return rc;
    TableSrc src;
    std::vector<int64_t> offsets;
    int64_t longest = 0;
    if ((rc = table_src(h_xy, h_offsets, nullptr, nullptr, n_scans, offsets, &src, &longest))) return rc;
    return align_impl(h, src, n_scans, longest, h_pairs, h_init, init_ld, B, p, h_T, T_ld, h_err, h_passes, ep);
}

int icpb_align_host_scans(icpb_handle h, const double *const *scan_xy, const int64_t *scan_len, int64_t n_scans,
                          const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                          const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes,
                          const icpb_epilogue *ep)
{
    int rc = align_check(h, n_scans, h_pairs, init_ld, B, p, h_T, T_ld, h_err, h_passes, ep);
    if (rc) return rc;
    TableSrc src;
    std::vector<int64_t> offsets;
    int64_t longest = 0;
    if ((rc = table_src(nullptr, nullptr, scan_xy, scan_len, n_scans, offsets, &src, &longest))) return rc;
    return align_impl(h, src, n_scans, longest, h_pairs, h_init, init_ld, B, p, h_T, T_ld, h_err, h_passes, ep);
}

int icpb_align_host_accept(icpb_handle h, const double *h_xy, const int64_t *h_offsets,
                           const double *const *scan_xy, const int64_t *scan_len, int64_t n_scans,
                           const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                           const icpb_params *p, double accept_thresh, int64_t capacity, int64_t *n_accepted,
                           int64_t *h_rows, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes)
{
    int rc = align_check(h, n_scans, h_pairs, init_ld, B, p, h_T, T_ld, h_err, h_passes, nullptr);
    if (rc) return rc;
    if (B == 0) return fail(ICPB_EINVAL, "icpb_align_host_accept: bad argument%s");
    if (capacity < 1 || !n_accepted || !h_rows || isnan(accept_thresh))
        return fail(ICPB_EINVAL, "icpb_align_host_accept: bad output arguments%s");
    TableSrc src;
    std::vector<int64_t> offsets;
    int64_t longest = 0;
    if ((rc = table_src(h_xy, h_offsets, scan_xy, scan_len, n_scans, offsets, &src, &longest))) return rc;
    AcceptHost acc = {accept_thresh, capacity, n_accepted, h_rows, h_T, T_ld, h_err, h_passes};
    return align_impl(h, src, n_scans, longest, h_pairs, h_init, init_ld, B, p, nullptr, T_ld, nullptr, nullptr,
                      nullptr, &acc);
}

int icpb_align_host_ld(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans,
                       const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                       const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes)
{
    return icpb_align_host_ex(h, h_xy, h_offsets, n_scans, h_pairs, h_init, init_ld, B, p, h_T, T_ld, h_err, h_passes,
                              nullptr);
}

int icpb_align_host(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans,
                    const int32_t *h_pairs, const double *h_init, int64_t B, const icpb_params *p,
                    double *h_T, double *h_err, int32_t *h_passes)
{
    return icpb_align_host_ld(h, h_xy, h_offsets, n_scans, h_pairs, h_init, 6, B, p, h_T, 6, h_err, h_passes);
}

int icpb_icp_pair_host(icpb_handle h, const double *h_src_xy, int64_t n_src,
                       const double *h_dst_xy, int64_t n_dst, const double *h_init6,
                       const icpb_params *p, double *h_T6, double *h_err, int32_t *h_passes,
                       double *h_hist, int32_t *h_corr)
{
    if (!h) return fail(ICPB_EINVAL, "handle is null%s");
    if (!h_src_xy || !h_dst_xy || n_src <= 0 || n_dst <= 0)
        return fail(ICPB_EINVAL, "empty point cloud (the reference's argmin raises on it)%s");
    int rc = check_params(p, 1);
    if (rc) return rc;
    if (!h_T6 || !h_err || !h_passes) return fail(ICPB_EINVAL, "output pointer is null%s");
    if (p->hist_cap > 0 && !h_hist) return fail(ICPB_EINVAL, "hist_cap > 0 but hist is null%s");
    if (p->corr_stride > 0 && (!h_corr || p->corr_stride < n_src))
        return fail(ICPB_EINVAL, "corr buffer missing or shorter than the source cloud%s");
    icpb_params q = *p;
    q.pair_mode = 0; q.k_first = 0; q.k_block = 1; q.k_stride = 0;
    ON_DEVICE(h);
    const double *const cloud[2] = {h_src_xy, h_dst_xy};
    const int64_t off[3] = {0, n_src, n_src + n_dst};
    const int32_t pair[2] = {0, 1};
    return run_host_common(h, cloud, off, 2, n_src > n_dst ? n_src : n_dst,
                           pair, h_init6, 1, &q, h_T6, h_err, h_passes, h_hist, h_corr);
}

int icpb_fit_pairs_host(icpb_handle h, const double *h_a_xy, const double *h_b_xy, int64_t n,
                        double *h_T6, double *h_err)
{
    if (!h || !h_a_xy || !h_b_xy || n <= 0 || n > 0x7fffffff || !h_T6 || !h_err)
        return fail(ICPB_EINVAL, "icpb_fit_pairs_host: bad argument%s");
    ON_DEVICE(h);
    int rc;
    const size_t nb = sizeof(double) * 2 * (size_t)n;
    double out[7];                                            // [T (6) | error]
    Carve c;
    const size_t o_a = c(nb), o_b = c(nb), o_out = c(sizeof out);
    if ((rc = h->arena.reserve(c.used))) return rc;
    double *da = at<double>(h->arena, o_a), *db = at<double>(h->arena, o_b), *dout = at<double>(h->arena, o_out);
    CU(cudaMemcpyAsync(da, h_a_xy, nb, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(db, h_b_xy, nb, cudaMemcpyHostToDevice, h->stream));
    icpb::fit_pairs_kernel<<<1, 256, 0, h->stream>>>((const double2 *)da, (const double2 *)db, (int)n,
                                                     dout, dout + 6);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, sizeof out, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    memcpy(h_T6, out, 6 * sizeof(double));
    *h_err = out[6];
    return 0;
}

static int upload_poses(icpb_handle h, const double *h_xy, const double *h_travelled, int64_t n,
                        double *d_xy, double *d_trav)
{
    CU(cudaMemcpyAsync(d_xy, h_xy, sizeof(double) * 2 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_trav, h_travelled, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    return 0;
}

// The input contract of the candidate kernels (include/icpb.h, ICPB_MAX_POSE_COORD): poses within the
// bound (so no squared distance overflows), `travelled` finite and non-decreasing (upper_bound's binary
// search), a min_dist_along_path that is not NaN (np.searchsorted and upper_bound disagree on NaN).
static int proximity_check(const double *h_xy, const double *h_travelled, int64_t n, double min_dist_along_path,
                           const char *who)
{
    if (min_dist_along_path != min_dist_along_path) return fail(ICPB_EINVAL, "%s: min_dist_along_path is NaN", who);
    bool bad = false;
    for (int64_t k = 0; k < 2 * n; ++k) bad |= !(fabs(h_xy[k]) <= ICPB_MAX_POSE_COORD);
    if (bad) return fail(ICPB_EINVAL, "%s: pose coordinates are non-finite or beyond ICPB_MAX_POSE_COORD", who);
    for (int64_t i = 0; i < n; ++i)
        bad |= !isfinite(h_travelled[i]) || (i > 0 && h_travelled[i] < h_travelled[i - 1]);
    if (bad) return fail(ICPB_EINVAL, "%s: travelled must be finite and non-decreasing", who);
    return 0;
}

int icpb_proximity_closest(icpb_handle h, const double *h_xy, const double *h_travelled, int64_t n,
                           double min_dist_along_path, double max_dist, int32_t *h_closest, double *h_dist)
{
    if (!h || !h_xy || !h_travelled || n <= 0 || n > 0x3fffffff || !h_closest || !h_dist)
        return fail(ICPB_EINVAL, "icpb_proximity_closest: bad argument%s");
    int rc = proximity_check(h_xy, h_travelled, n, min_dist_along_path, "icpb_proximity_closest");
    if (rc) return rc;
    ON_DEVICE(h);
    Carve c;
    const size_t o_xy = c(sizeof(double) * 2 * (size_t)n), o_trav = c(sizeof(double) * (size_t)n);
    const size_t o_closest = c(sizeof(int32_t) * (size_t)n), o_dist = c(sizeof(double) * (size_t)n);
    if ((rc = h->arena.reserve(c.used))) return rc;
    double *d_xy = at<double>(h->arena, o_xy), *d_trav = at<double>(h->arena, o_trav);
    int32_t *d_closest = at<int32_t>(h->arena, o_closest);
    double *d_dist = at<double>(h->arena, o_dist);
    if ((rc = upload_poses(h, h_xy, h_travelled, n, d_xy, d_trav))) return rc;
    const unsigned grid = (unsigned)((n * 32 + 255) / 256);
    icpb::proximity_closest_kernel<<<grid, 256, 0, h->stream>>>((const double2 *)d_xy, d_trav, (int)n,
                                                                min_dist_along_path, max_dist, d_closest, d_dist);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h_closest, d_closest, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(h_dist, d_dist, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

int icpb_proximity_pairs(icpb_handle h, const double *h_xy, const double *h_travelled, int64_t n,
                         double min_dist_along_path, double max_dist, int64_t capacity,
                         int32_t *h_pairs, int64_t *n_pairs)
{
    if (!h || !h_xy || !h_travelled || n <= 0 || n > 0x3fffffff || !n_pairs || capacity < 0 ||
        (capacity > 0 && !h_pairs))
        return fail(ICPB_EINVAL, "icpb_proximity_pairs: bad argument%s");
    int rc = proximity_check(h_xy, h_travelled, n, min_dist_along_path, "icpb_proximity_pairs");
    if (rc) return rc;
    ON_DEVICE(h);
    // The pairs are carved at the caller's capacity (the count from a capacity-0 call; n * n bounds any
    // count): the arena is reserved before the count is known, and a later reservation would free the poses.
    const int64_t rows = capacity < n * n ? capacity : n * n;
    Carve c;
    const size_t o_xy = c(sizeof(double) * 2 * (size_t)n), o_trav = c(sizeof(double) * (size_t)n);
    const size_t o_count = c(sizeof(int64_t) * (size_t)n), o_off = c(sizeof(int64_t) * (size_t)n);
    const size_t o_pairs = c(sizeof(int32_t) * 2 * (size_t)rows);
    if ((rc = h->arena.reserve(c.used))) return rc;
    double *d_xy = at<double>(h->arena, o_xy), *d_trav = at<double>(h->arena, o_trav);
    int64_t *d_count = at<int64_t>(h->arena, o_count), *d_off = at<int64_t>(h->arena, o_off);
    int32_t *d_pairs = at<int32_t>(h->arena, o_pairs);
    if ((rc = upload_poses(h, h_xy, h_travelled, n, d_xy, d_trav))) return rc;
    const unsigned grid = (unsigned)((n * 32 + 255) / 256);
    icpb::proximity_pairs_kernel<false><<<grid, 256, 0, h->stream>>>((const double2 *)d_xy, d_trav, (int)n,
                                                                     min_dist_along_path, max_dist,
                                                                     d_count, nullptr, nullptr);
    CU(cudaGetLastError());
    std::vector<int64_t> cnt((size_t)n), off((size_t)n);
    CU(cudaMemcpyAsync(cnt.data(), d_count, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    int64_t total = 0;
    for (int64_t i = 0; i < n; ++i) { off[i] = total; total += cnt[i]; }      // S values: a host scan is enough
    *n_pairs = total;
    if (capacity == 0 || total == 0) return 0;                                // size query
    if (total > capacity) return fail(ICPB_EINVAL, "icpb_proximity_pairs: capacity too small%s");
    CU(cudaMemcpyAsync(d_off, off.data(), sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    icpb::proximity_pairs_kernel<true><<<grid, 256, 0, h->stream>>>((const double2 *)d_xy, d_trav, (int)n,
                                                                    min_dist_along_path, max_dist,
                                                                    nullptr, d_off, d_pairs);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h_pairs, d_pairs, sizeof(int32_t) * 2 * (size_t)total, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

/* Host epilogue of the odometry fan-out: the serial SE(2) prefix product of scripts/main.py:249-256,
 * pose_i = mat_to_pose(pose_to_mat(pose_{i-1}) @ T_{i-1}), with the reference's own sequence of
 * operations (cos/sin of the heading, 3x3 product, atan2) so the poses match it to rounding.  It
 * is a 5,000-step dependency chain of a few flops each: a host loop in C (0.3 ms) beats both the
 * reference's Python loop (~100 ms) and a kernel launch. */
int icpb_compose_chain(const double *pose0, const double *T6, int64_t n, double *poses_out)
{
    if (!pose0 || (n > 0 && !T6) || n < 0 || !poses_out) return fail(ICPB_EINVAL, "icpb_compose_chain: bad argument%s");
    poses_out[0] = pose0[0]; poses_out[1] = pose0[1]; poses_out[2] = pose0[2];
    for (int64_t i = 0; i < n; ++i) {
        const double *p = poses_out + 3 * i, *T = T6 + 6 * i;
        const double c = cos(p[2]), s = sin(p[2]);
        // rows of pose_to_mat(p) @ [T; 0 0 1], summed left to right like a 3-term dot product
        const double m00 = c * T[0] + -s * T[3];
        const double m10 = s * T[0] + c * T[3];
        const double x = c * T[2] + -s * T[5] + p[0];
        const double y = s * T[2] + c * T[5] + p[1];
        double *q = poses_out + 3 * (i + 1);
        q[0] = x; q[1] = y; q[2] = atan2(m10, m00);
    }
    return 0;
}

/* The same prefix product as a parallel scan on the device (csrc/icpb_compose.cuh).  d_T6 may be the
 * d_T output of icpb_run_device: the transforms then never visit the host. */
int icpb_compose_chain_device(icpb_handle h, const double *pose0, const double *d_T6, int64_t n,
                              double *d_poses_out, void *stream)
{
    if (!h || !pose0 || (n > 0 && !d_T6) || n < 0 || !d_poses_out)
        return fail(ICPB_EINVAL, "icpb_compose_chain_device: bad argument%s");
    ON_DEVICE(h);
    icpb::compose_chain_kernel<<<1, icpb::kComposeThreads, 0, (cudaStream_t)stream>>>(d_T6, n, pose0[0], pose0[1], pose0[2],
                                                                                      d_poses_out);
    CU(cudaGetLastError());
    return 0;
}

/* Host buffers in and out, through the device scan (for the comparison with the host loop). */
int icpb_compose_chain_gpu(icpb_handle h, const double *pose0, const double *h_T6, int64_t n, double *h_poses_out)
{
    if (!h || !pose0 || (n > 0 && !h_T6) || n < 0 || !h_poses_out)
        return fail(ICPB_EINVAL, "icpb_compose_chain_gpu: bad argument%s");
    ON_DEVICE(h);
    int rc;
    Carve c;
    const size_t o_T = c(sizeof(double) * 6 * (size_t)n), o_P = c(sizeof(double) * 3 * (size_t)(n + 1));
    if ((rc = h->arena.reserve(c.used))) return rc;
    double *d_T = at<double>(h->arena, o_T), *d_P = at<double>(h->arena, o_P);
    if (n > 0) CU(cudaMemcpyAsync(d_T, h_T6, sizeof(double) * 6 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    if ((rc = icpb_compose_chain_device(h, pose0, d_T, n, d_P, h->stream))) return rc;
    CU(cudaMemcpyAsync(h_poses_out, d_P, sizeof(double) * 3 * (size_t)(n + 1), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

/* Pose-graph SGD (include/icpb.h): n_steps passes of the reference's
 * pose_graph_optimization_step_sgd over the same edge list, poses updated in place. */
int icpb_pose_graph_sgd(icpb_handle h, double *h_poses, int64_t n, const int32_t *h_edges,
                        const double *h_edge_T6, int64_t n_edges, const double *h_learning_rates,
                        int32_t n_steps, double loop_closure_uncertainty)
{
    if (!h || !h_poses || n <= 0 || n > 0x1fffffff || n_edges < 0 || n_edges > 0x1fffffff || n_steps < 0 ||
        (n_edges > 0 && (!h_edges || !h_edge_T6)) || (n_steps > 0 && !h_learning_rates))
        return fail(ICPB_EINVAL, "icpb_pose_graph_sgd: bad argument%s");
    if (!(loop_closure_uncertainty > 0.0)) return fail(ICPB_EINVAL, "icpb_pose_graph_sgd: loop_closure_uncertainty must be > 0%s");
    for (int64_t e = 0; e < 2 * n_edges; ++e)
        if (h_edges[e] < 0 || h_edges[e] >= n) return fail(ICPB_EINVAL, "icpb_pose_graph_sgd: edge endpoint out of range%s");
    // Edges the optimiser ignores (|a - b| == 1, :14-16 and :28-30) or that have an empty node range
    // (b <= a: `range(a+1, b+1)` :20 and `i <= b` :46 never hold) move nothing: they stay on the host.
    std::vector<int32_t> ve;
    std::vector<double> vt;
    for (int64_t e = 0; e < n_edges; ++e) {
        const int32_t ea = h_edges[2 * e], eb = h_edges[2 * e + 1];
        if (eb > ea + 1) {
            ve.push_back(ea); ve.push_back(eb);
            vt.insert(vt.end(), h_edge_T6 + 6 * e, h_edge_T6 + 6 * e + 6);
        }
    }
    if (ve.empty() || n_steps == 0) return 0;
    ON_DEVICE(h);
    const size_t E = ve.size() / 2, N = (size_t)n;
    // (RECA's 80-byte records are read as 16-byte pairs: the 256-byte alignment of a carved array covers it)
    const size_t D = sizeof(double);
    Carve c;
    const size_t o_RECA = c(D * 10 * E), o_tf = c(D * 6 * E), o_dW = c(D * 4 * E), o_REC = c(D * 10 * E);
    const size_t o_ES = c(D * 23 * E), o_poses = c(D * 3 * N), o_M = c(D * 3 * N), o_P = c(D * 3 * N);
    const size_t o_edges = c(sizeof(int32_t) * 2 * E);
    int rc;
    if ((rc = h->arena.reserve(c.used))) return rc;
    double *d_RECA = at<double>(h->arena, o_RECA), *d_tf = at<double>(h->arena, o_tf), *d_dW = at<double>(h->arena, o_dW);
    double *d_REC = at<double>(h->arena, o_REC), *d_ES = at<double>(h->arena, o_ES);
    double *d_poses = at<double>(h->arena, o_poses), *d_M = at<double>(h->arena, o_M), *d_P = at<double>(h->arena, o_P);
    int32_t *d_edges = at<int32_t>(h->arena, o_edges);
    CU(cudaMemcpyAsync(d_poses, h_poses, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_tf, vt.data(), sizeof(double) * 6 * E, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_edges, ve.data(), sizeof(int32_t) * 2 * E, cudaMemcpyHostToDevice, h->stream));
    icpb::SgdArgs a;
    a.poses = d_poses; a.edges = d_edges; a.tf = d_tf; a.n = (int32_t)n; a.E = (int32_t)E;
    a.lcu = loop_closure_uncertainty; a.dW = d_dW; a.REC = d_REC; a.RECA = d_RECA; a.ES = d_ES; a.M = d_M; a.P = d_P;
    // per pass: weights of the edges, their sum per node, the lazy chain over the edges on one SM (the
    // only sequential part), then every record applied to every node on all SMs
    const dim3 node_grid((unsigned)((N + icpb::kSgdNodeThreads - 1) / icpb::kSgdNodeThreads), 3);   // (nodes, dof)
    for (int32_t k = 0; k < n_steps; ++k) {
        a.learning_rate = h_learning_rates[k];
        icpb::sgd_weights_kernel<<<(unsigned)((E + 255) / 256), 256, 0, h->stream>>>(a);
        icpb::sgd_accumulate_kernel<<<node_grid, icpb::kSgdNodeThreads, 0, h->stream>>>(a);
        icpb::sgd_chain_kernel<<<1, icpb::kSgdThreads, 0, h->stream>>>(a);
        icpb::sgd_apply_kernel<<<node_grid, icpb::kSgdNodeThreads, 0, h->stream>>>(a);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(h_poses, d_poses, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

/* ---- occupancy grid (include/icpb.h; reference src/produce_occupancy_grid.py) ---- */
namespace {

int grid_check(icpb_handle h, const double *h_poses, int64_t n, double cell_width, const char *who)
{
    if (!h || !h_poses || n <= 0 || !(cell_width > 0.0 && isfinite(cell_width)))
        return fail(ICPB_EINVAL, "%s: bad argument", who);
    if (!h->xy) return fail(ICPB_ENOSCANS, "%s: no scan table set", who);
    if (n > h->n_scans) return fail(ICPB_EINVAL, "%s: more poses than scans in the table", who);
    bool bad = false;
    for (int64_t k = 0; k < 3 * n; ++k) bad |= !isfinite(h_poses[k]);
    if (bad) return fail(ICPB_EINVAL, "%s: non-finite pose", who);
    return 0;
}

// ICPB_MAX_GRID_CELL (include/icpb.h): every cell coordinate the walk can see -- the pose's and the beam
// end's, |global| <= |pose| + sqrt(2) * ICPB_MAX_COORD -- is bounded from the host's data alone.
int grid_cell_check(const double *h_poses, int64_t n, double min_x, double min_y, double cell_width)
{
    if (!isfinite(min_x) || !isfinite(min_y))
        return fail(ICPB_EINVAL, "icpb_occupancy_grid_update: non-finite grid origin%s");
    double p = 0.0;
    for (int64_t i = 0; i < n; ++i) p = fmax(p, fmax(fabs(h_poses[3 * i]), fabs(h_poses[3 * i + 1])));
    const double reach = (p + fmax(fabs(min_x), fabs(min_y)) + M_SQRT2 * ICPB_MAX_COORD) / cell_width;
    if (!(reach <= ICPB_MAX_GRID_CELL))
        return fail(ICPB_EINVAL, "icpb_occupancy_grid_update: cell coordinates could exceed ICPB_MAX_GRID_CELL "
                                 "(poses or origin too far for this cell width)%s");
    return 0;
}

// (cos theta, sin theta, x, y) per pose: odom_change_to_mat's trigonometry (src/utils.py:8-9) in libm
std::vector<double> pose_records(const double *h_poses, int64_t n)
{
    std::vector<double> r(4 * (size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        r[4 * i] = cos(h_poses[3 * i + 2]); r[4 * i + 1] = sin(h_poses[3 * i + 2]);
        r[4 * i + 2] = h_poses[3 * i]; r[4 * i + 3] = h_poses[3 * i + 1];
    }
    return r;
}

double key_to_double(unsigned long long k)
{
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k;
    double v;
    memcpy(&v, &b, sizeof v);
    return v;
}

}  // namespace

int icpb_occupancy_grid_bounds(icpb_handle h, const double *h_poses, int64_t n, double cell_width,
                               double min_width, double min_height, double *min_x_out, double *min_y_out,
                               int64_t *height, int64_t *width)
{
    int rc = grid_check(h, h_poses, n, cell_width, "icpb_occupancy_grid_bounds");
    if (rc) return rc;
    if (!min_x_out || !min_y_out || !height || !width) return fail(ICPB_EINVAL, "icpb_occupancy_grid_bounds: null output%s");
    if (!isfinite(min_width) || !isfinite(min_height))
        return fail(ICPB_EINVAL, "icpb_occupancy_grid_bounds: non-finite minimum size%s");
    ON_DEVICE(h);
    const unsigned long long init[4] = {~0ULL, ~0ULL, 0ULL, 0ULL};
    Carve c;
    const size_t o_mm = c(sizeof init), o_poses = c(sizeof(double) * 4 * (size_t)n);
    if ((rc = h->arena.reserve(c.used))) return rc;
    unsigned long long *d_mm = at<unsigned long long>(h->arena, o_mm);
    double *d_poses = at<double>(h->arena, o_poses);
    const std::vector<double> rec = pose_records(h_poses, n);
    CU(cudaMemcpyAsync(d_mm, init, sizeof init, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_poses, rec.data(), sizeof(double) * 4 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    icpb::GridArgs a = {};
    a.xy = h->xy; a.offsets = h->offsets; a.poses = d_poses; a.n = (int32_t)n;
    icpb::grid_bounds_kernel<<<(unsigned)n, 256, 0, h->stream>>>(a, d_mm);
    CU(cudaGetLastError());
    unsigned long long mm[4];
    CU(cudaMemcpyAsync(mm, d_mm, sizeof mm, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (mm[0] == ~0ULL) return fail(ICPB_EINVAL, "icpb_occupancy_grid_bounds: the scans hold no points%s");
    // src/produce_occupancy_grid.py:30-51, operation for operation
    double min_x = key_to_double(mm[0]) - (cell_width / 2), max_x = key_to_double(mm[2]) + (cell_width / 2);
    double min_y = key_to_double(mm[1]) - (cell_width / 2), max_y = key_to_double(mm[3]) + (cell_width / 2);
    double width_dist = max_x - min_x, height_dist = max_y - min_y;
    if (width_dist < min_width) { const double off = (min_width - width_dist) / 2; min_x -= off; width_dist = min_width; }
    if (height_dist < min_height) { const double off = (min_height - height_dist) / 2; min_y -= off; height_dist = min_height; }
    const double w_cells = ceil(width_dist / cell_width), h_cells = ceil(height_dist / cell_width);
    if (!(w_cells * h_cells <= (double)ICPB_MAX_GRID_CELLS))                 // NaN and inf too
        return fail(ICPB_EINVAL, "icpb_occupancy_grid_bounds: the grid would exceed ICPB_MAX_GRID_CELLS cells%s");
    *min_x_out = min_x; *min_y_out = min_y;
    *width = (int64_t)w_cells;
    *height = (int64_t)h_cells;
    return 0;
}

int icpb_occupancy_grid_update(icpb_handle h, const double *h_poses, int64_t n, int8_t *h_grid,
                               int64_t height, int64_t width, double min_x, double min_y,
                               double cell_width, int32_t k_hit, int32_t k_miss)
{
    int rc = grid_check(h, h_poses, n, cell_width, "icpb_occupancy_grid_update");
    if (rc) return rc;
    if (!h_grid || height <= 0 || width <= 0 || height > 0x7fffffff || width > 0x7fffffff ||
        height * width > ICPB_MAX_GRID_CELLS)
        return fail(ICPB_EINVAL, "icpb_occupancy_grid_update: bad grid%s");
    // the per-cell closed form needs a miss to leave a cell negative and a hit to leave it positive
    if (k_hit < 1 || k_hit > 127 || k_miss < 1 || k_miss > 127)
        return fail(ICPB_EINVAL, "icpb_occupancy_grid_update: kHitOdds and kMissOdds must be integers in 1..127%s");
    if ((rc = grid_cell_check(h_poses, n, min_x, min_y, cell_width))) return rc;
    ON_DEVICE(h);
    // the beam order keys are 32 bit: 2 * (beam index + 1) + 1 must fit (2^31 - 2 beams)
    int64_t n_points = 0;
    CU(cudaMemcpy(&n_points, h->offsets + n, sizeof n_points, cudaMemcpyDeviceToHost));
    if (n_points >= 0x7ffffffeLL) return fail(ICPB_EINVAL, "icpb_occupancy_grid_update: more than 2^31 - 2 beams in one call%s");
    const size_t cells = (size_t)height * (size_t)width;
    const size_t words = 4 * cells;                          // [last_hit | n_miss | n_hit | miss_after], per cell
    Carve c;
    const size_t o_poses = c(sizeof(double) * 4 * (size_t)n), o_words = c(sizeof(uint32_t) * words), o_grid = c(cells);
    if ((rc = h->arena.reserve(c.used))) return rc;
    double *d_poses = at<double>(h->arena, o_poses);
    uint32_t *d_words = at<uint32_t>(h->arena, o_words);
    int8_t *d_grid = at<int8_t>(h->arena, o_grid);
    const std::vector<double> rec = pose_records(h_poses, n);
    CU(cudaMemcpyAsync(d_poses, rec.data(), sizeof(double) * 4 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_grid, h_grid, cells, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(d_words, 0, sizeof(uint32_t) * words, h->stream));
    icpb::GridArgs a = {};
    a.xy = h->xy; a.offsets = h->offsets; a.poses = d_poses; a.n = (int32_t)n;
    a.min_x = min_x; a.min_y = min_y; a.cell = cell_width; a.h = (int32_t)height; a.w = (int32_t)width;
    a.last_hit = d_words; a.n_miss = d_words + cells; a.n_hit = d_words + 2 * cells; a.miss_after = d_words + 3 * cells;
    icpb::grid_hits_kernel<<<(unsigned)n, 256, 0, h->stream>>>(a);
    CU(cudaGetLastError());
    icpb::grid_misses_kernel<<<(unsigned)n, 256, 0, h->stream>>>(a);
    CU(cudaGetLastError());
    icpb::grid_finalize_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, h->stream>>>(a, d_grid, k_hit, k_miss);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h_grid, d_grid, cells, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return 0;
}

int icpb_get_kernel_info(icpb_handle h, int64_t B, icpb_kernel_info *out)
{
    if (!h || !out) return fail(ICPB_EINVAL, "icpb_get_kernel_info: bad argument%s");
    if (!h->xy) return fail(ICPB_ENOSCANS, "no scan table set%s");
    ON_DEVICE(h);
    LaunchCfg cfg;
    int rc = make_cfg(h, h->longest, B > 0 ? B : (int64_t)1 << 40, &cfg, nullptr, h->tune_large == 1);
    if (rc) return rc;
    cudaFuncAttributes fa;
    CU(cudaFuncGetAttributes(&fa, align_kernel(cfg.big, false, false)));
    int64_t grid = (int64_t)cfg.ctas_per_sm * h->sm_count;
    if (B > 0 && grid > B) grid = B;
    out->threads_per_cta = cfg.threads; out->ctas_per_sm = cfg.ctas_per_sm; out->sm_count = h->sm_count;
    out->grid = (int32_t)grid; out->regs_per_thread = fa.numRegs; out->smem_bytes = cfg.smem;
    out->points_per_thread = kPointsPerThread; out->variant = 2;
    return 0;
}

int64_t icpb_launch_count(icpb_handle h) { return h ? h->launches : 0; }

int64_t icpb_scan_count(icpb_handle h) { return h && h->xy ? h->n_scans : 0; }

int icpb_count_work(icpb_handle h, int enable)
{
    if (!h) return fail(ICPB_EINVAL, "handle is null%s");
    ON_DEVICE(h);
    if (enable) {
        CU(cudaMemset(h->queue + kQueueRing, 0, sizeof(unsigned long long)));
        h->executed = h->queue + kQueueRing;
    } else {
        h->executed = nullptr;
    }
    return 0;
}

int icpb_read_work(icpb_handle h, uint64_t *executed_pde)
{
    if (!h || !executed_pde) return fail(ICPB_EINVAL, "icpb_read_work: bad argument%s");
    ON_DEVICE(h);
    CU(cudaDeviceSynchronize());
    unsigned long long v = 0;
    CU(cudaMemcpy(&v, h->queue + kQueueRing, sizeof v, cudaMemcpyDeviceToHost));
    *executed_pde = v;
    return 0;
}

}  // extern "C"
