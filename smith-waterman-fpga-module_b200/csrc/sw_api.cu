/*
 * sw_api.cu -- host side of libsw_b200.so: the C ABI declared in include/sw_b200.h.
 *
 * Replaces the reference's job path (main_test.c:290-477: build sequence records, attach the
 * AFU, poll the WED) and the bank-level dispatch (ScoreBank_v2.v:142-169 + PrioEncoder.v +
 * SM_Feeder2.v): subjects are length-sorted and paired on the host (the "first free module"
 * arbitration becomes a length-bucketed work queue drained by persistent blocks), sharded
 * over the handle's GPUs as contiguous input ranges, and moved with cudaMemcpyAsync from
 * pinned staging on per-GPU streams.  No CPU scoring path exists in this library.
 *
 * Two submit paths:
 *   regular  -- length sort + pairing on the host, code stream built on the GPU (build_tp_kernel),
 *               a launch plan of strip-kernel launches (per query group / query chunk), results
 *               in an HBM matrix (int32 / int16) or fused per-query top-k lists;
 *   small    -- latency path for small batches: ONE pinned staging buffer, ONE H2D copy, ONE
 *               kernel (a DIRECT strip instance that forms the column codes on the fly), scores
 *               written straight into mapped pinned host memory.  No memsets, no event creation,
 *               no heap allocation per call.
 */
#include "../../include/sw_b200.h"
#include "sw_jit.h"
#include "sw_kernels.h"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <thread>
#include <vector>

namespace {

#ifdef SW_BOUNDS_CHECK
constexpr size_t kGuard = 256;           // canary bytes on both sides of every device buffer
constexpr int kGuardByte = 0xA5;
#else
constexpr size_t kGuard = 0;
#endif

struct PinnedBuf {
    void *p = nullptr;
    void *dptr = nullptr;                // device view (mapped allocations)
    size_t cap = 0;
    cudaError_t reserve(size_t bytes, bool mapped = false) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; dptr = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, mapped ? (cudaHostAllocMapped | cudaHostAllocPortable) : cudaHostAllocDefault);
        if (e != cudaSuccess) return e;
        if (mapped) {
            e = cudaHostGetDevicePointer(&dptr, p, 0);
            if (e != cudaSuccess) { cudaFreeHost(p); p = nullptr; return e; }
        }
        cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; dptr = nullptr; cap = 0; }
};

struct DevBuf {
    void *p = nullptr;                   // usable region
    void *base = nullptr;                // allocation (p - kGuard)
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap && p) return cudaSuccess;
        if (base) cudaFree(base);
        p = base = nullptr; cap = 0;
        size_t want = bytes ? bytes : 16;
        want = (want + 255) & ~(size_t)255;
        cudaError_t e = cudaMalloc(&base, want + 2 * kGuard);
        if (e != cudaSuccess) { base = nullptr; return e; }
        p = (char *)base + kGuard;
        cap = want;
#ifdef SW_BOUNDS_CHECK
        e = cudaMemset(base, kGuardByte, kGuard);
        if (e == cudaSuccess) e = cudaMemset((char *)p + cap, kGuardByte, kGuard);
#endif
        return e;
    }
    void release() { if (base) cudaFree(base); p = base = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    // true if both canaries are intact (always true in regular builds)
    bool canaries_ok() const {
#ifdef SW_BOUNDS_CHECK
        if (!base) return true;
        unsigned char g[2 * kGuard];
        if (cudaMemcpy(g, base, kGuard, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
        if (cudaMemcpy(g + kGuard, (char *)p + cap, kGuard, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
        for (size_t i = 0; i < 2 * kGuard; ++i) if (g[i] != kGuardByte) return false;
#endif
        return true;
    }
};

struct QueryChunk { int q0, q1; cudaEvent_t done; };

// A length group of the sorted pair list: pairs [p0, p1) (p0 a multiple of 32), subjects at most
// max_len long.  The bank's arbitration (PrioEncoder.v:18-21 + SM_Feeder2.v:104-205) hands every
// target to the first free module; here every length group gets its own launch, kernel variant and
// pass-boundary scratch, so one very long subject does not size the scratch of every block.
struct Seg { uint32_t p0, p1, max_len; uint64_t sum_len; };

constexpr int kStreams = 4;              // concurrent launch streams per GPU (the compute stream + 3)

constexpr unsigned kOvfCap = 1u << 20;   // entries of the 16-bit-overflow side list

// Everything that belongs to one database batch on one GPU.  Two slots per GPU: while the
// kernels of batch k run, batch k+1 can be sorted, uploaded and enqueued, and batch k-1 copied
// back (the feeder's double buffering, SM_Feeder2.v:104-205, at batch granularity).
struct Slot {
    size_t s0 = 0, s1 = 0;            // global subject range [s0, s1) of this GPU's shard
    DevBuf d_raw, d_off, d_len, d_pair_subj, d_pair_len, d_tile_woff, d_tp, d_out;
    DevBuf d_ovf_count, d_ovf_list, d_ovf_score, d_topk_out;
    DevBuf d_hits_key, d_hits_score, d_hits_count;   // hit list of the last scoring (reserved at the first one in hits mode)
    uint32_t npairs = 0, max_len = 0;
    uint64_t sum_len = 0, tp_words = 0;
    PinnedBuf h_stage_a, h_stage_b, h_stage_c, h_stage_d, h_topk, h_ovf, h_hits;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_upload = nullptr;
    std::vector<cudaEvent_t> ev_pool;  // chunk-done events, created once
    std::vector<QueryChunk> chunks;
    std::vector<uint32_t> order, hist; // host scratch of the length sort (capacity is kept)
    std::vector<uint32_t> empties;     // first few zero-length subjects (they score 0; top-k fill)
    std::vector<Seg> segs;             // length groups of the sorted pair list (launch planning)
    std::vector<int> qidx_host;        // query lists of the last launch plan (source of an async upload)
    std::vector<uint32_t> pair_tmp;    // latency path: pairing scratch before the descriptors are written
    bool scored = false;
    bool ovf_used = false;
    int out_mode = SW_OUT_I32;         // of the last scoring
    int topk_k = 0;
    int hits_shift = 0;                // hit keys: row << hits_shift | shard-local subject
    // small (latency) path: one staging buffer in, mapped scores out
    bool is_small = false;
    PinnedBuf h_small_in, h_small_out, h_small_flag;
    DevBuf d_small_in, d_small_done;
    unsigned small_seq = 0;            // value the kernel writes to the completion flag
    bool ev_stop_deferred = false;     // latency path without timing: ev_stop is recorded only when somebody needs it
    bool small_by_flag = false;        // this batch completes by flag (else: every result word replaces a sentinel)
    bool small_timed = false;          // events were recorded around the kernel
};

struct GpuCtx {
    int dev = 0;
    int num_sms = 0;
    cudaStream_t st_compute = nullptr, st_copy = nullptr;
    cudaStream_t st_aux[kStreams - 1] = {nullptr, nullptr, nullptr};   // launches of a plan run concurrently
    cudaEvent_t ev_fork = nullptr, ev_join[kStreams - 1] = {nullptr, nullptr, nullptr};
    DevBuf d_bnd_aux[kStreams - 1];
    // queries
    DevBuf d_qpacked, d_qoff, d_qlen, d_qidx;
    Slot slot[2];
    // scratch shared by both slots (kernels of one GPU run in stream order)
    DevBuf d_bnd, d_counters, d_scratch32, d_best_score, d_best_index, d_topk_keys, d_err;
    DevBuf d_part_done, d_part_best;  // pass split: progress words and parked running maxima per (pair block, query) chain
    DevBuf d_wave_bnd, d_wave_state;  // band-pipelined kernel: boundary rows; progress / best / done words
    int wave_bps[16] = {0};           // resident blocks per SM of its instances (0 = not asked yet)
    DevBuf d_wave32_bnd, d_wave32_state;   // 32-bit band-pipelined scorer of the overflow list
    DevBuf d_wave_rows;               // top-k / hits mode: one scratch score row per band-pipelined query
    DevBuf d_hits_key2, d_hits_score2, d_sort_tmp;   // fetch of a hit list: radix-sort output and temp storage (copy stream)
    uint32_t wave32_epoch = 0;        // 8-bit tag field: 1 .. 255, boundary rows zeroed when it restarts
    int wave32_bps = 0;
    uint32_t wave_epoch = 0;          // launches so far: the tag of the boundary elements (20 bits)
    unsigned counter_next = 0;        // next unused work-queue counter
    // autotune: timing events and the cached decision, per GPU (shards differ in shape)
    cudaEvent_t ev_tune0 = nullptr, ev_tune1 = nullptr;
    uint64_t tune_key = 0;            // workload signature of the cached decision
    int tune_choice = -1;
    std::map<std::pair<int, int>, int> occ_cache;   // (variant, chunk_passes) -> resident blocks / SM
};

// Host-side description of one batch (all GPUs).
struct Batch {
    size_t ns = 0;
    int nq = 0;                       // query rows the scores of this batch have
    bool loaded = false, scored = false, small = false;
    int out_mode = SW_OUT_I32, topk_k = 0;
    int32_t hits_min = 0;             // > 0: scored in hits mode with this threshold
    size_t hits_max = 0;
    bool hits_staged = false;         // the stitched list below waits for a fetch with enough room
    std::vector<uint32_t> hits_row;
    std::vector<uint64_t> hits_index;
    std::vector<int32_t> hits_score;
    std::vector<uint64_t> ids;
    bool have_ids = false;
    uint64_t cells = 0;
    std::vector<uint64_t> ovf_index;  // I16 mode: entries above 32767 of the batch fetched last
    std::vector<int32_t> ovf_score;
};

}  // namespace

struct sw_handle {
    sw_params_t params;
    std::vector<GpuCtx> gpus;
    // host copy of the queries
    std::vector<uint8_t> q_packed;
    std::vector<uint32_t> q_off, q_len;
    uint32_t q_max_len = 0;
    uint64_t q_sum_len = 0;
    bool both_strands = false;
    int nq_user = 0;                  // queries given by the caller (rows = nq_user * strands)
    // database batches: slot 0 doubles as the resident database of sw_load_db
    Batch batch[2];
    int fifo[2] = {0, 0};             // slots in flight, oldest first
    int n_inflight = 0;
    int last_slot = 0;                // slot of the most recent load / fetch (ids, cells, overflow list)
    int out_mode = SW_OUT_I32;        // SW_OUTPUT_I32 / SW_OUTPUT_I16 for the next scoring
    int topk_k = 0;                   // > 0: fused top-k instead of a matrix
    int32_t hits_min = 0;             // > 0: hit list (scores >= hits_min) instead of a matrix
    size_t hits_max = 0;              // entries of each GPU's hit list
    bool small_path = true;
    bool small_timing = true;         // record CUDA events around the latency path's kernel (sw_last_kernel_ms)
    int jit = 1;                      // run-time specialisation of gap penalties: 0 off, 1 large jobs, 2 always
    int wave = 1;                     // band-pipelined kernel for few long pairs: 0 off, 1 automatic, 2 whenever possible
    int wave32 = 1;                   // overflow list: long entries go to the band-pipelined 32-bit scorer
    bool trace_small = false;         // SW_B200_TRACE_SMALL=1: phase times of the latency path, printed by sw_destroy
    double tr_prep = 0, tr_launch = 0, tr_wait = 0, tr_copy = 0; long tr_n = 0;
    bool small_sentinel = true;       // latency path: completion seen in the result words themselves (no fence, no flag)
    bool small_zero_copy = true;      // latency path: staging buffers of <= 64 KB are read by the kernel from mapped host memory (no H2D copy)
    unsigned long long wave32_min_cells = 1000000ull;
    // launch-planner knobs (environment SW_B200_PLAN_SEGS / _QGROUPS / _STREAMS / _TAU): experiments
    int plan_segs = 2;                // 0 never, 1 always, 2 when one launch would need a huge pass-boundary scratch
    bool plan_qgroups = false;        // per-query variant choice (measured: the extra launches cost more than they gain)
    int plan_streams = kStreams;
    double plan_tau = 0.5;
    // work order of a strip launch (sw_strip.cuh; environment SW_B200_STICKY / SW_B200_SUPERBLOCK_MB)
    int sticky = -1;                  // 0 = super-block order; > 0 = sticky order with this drift bound in pair blocks;
                                      // -1 = sticky order, drift bound of about 1 MB of code stream (4 .. 32 pair blocks)
    double superblock_mb = 24.0;      // code-stream bytes of one super-block
    int pass_split = -1;              // pass split of long queries with few work items: 0 never, -1 automatic,
                                      // n > 1 = about n parts whenever the query has that many profile chunks (A/B, tests)
    // bookkeeping
    int last_parts = 1;               // parts per work item of the last strip plan (pass split), 1 = not split
    std::atomic<int> last_cuda{0};    // written by the per-GPU worker threads as well
    std::atomic<uint64_t> launches{0};
    uint64_t last_cells = 0;
    double last_ms = 0.0;
    sw_stats_t stats{};               // host-visible phase times of the last submit / fetch
    char last_kernel[96] = "none";
    int force_R = 0, force_G = 0, force32 = 0, force_arith = -1;
    int force_variant = -1;
    bool autotune = true;             // time the model's top candidates on a sample of large jobs
};

namespace {

const int kMaxCounters = 4096;

#define SW_CUDA(h, call)                                                        \
    do {                                                                        \
        cudaError_t e__ = (call);                                               \
        if (e__ != cudaSuccess) { (h)->last_cuda.store((int)e__); return (e__ == cudaErrorMemoryAllocation) ? SW_ENOMEM : SW_ECUDA; } \
    } while (0)

int validate_params(const sw_params_t *p)
{
    if (p->match <= 0 || p->match > 255) return SW_EINVAL;
    if (p->mismatch > p->match || p->mismatch < -255) return SW_EINVAL;
    if (p->gap_extend > 0 || p->gap_extend < -255) return SW_EINVAL;
    const int goe = (int)p->gap_open + (int)p->gap_extend;
    if (goe > 0 || p->gap_open < -2040) return SW_EINVAL;
    if (p->score_width != 0) {
        if (p->score_width < 6 || p->score_width > 15) return SW_EINVAL;
        const int half = 1 << (p->score_width - 1);
        /* keep every intermediate of the W-bit machine inside its range except the
           M overflow the mode exists to reproduce (SURVEY A.3) */
        if (p->match >= half || goe + p->gap_extend < -half || p->mismatch < -half) return SW_EINVAL;
    }
    return SW_OK;
}

SwScoring scoring_of(const sw_handle *h)
{
    SwScoring sc;
    sc.match = h->params.match; sc.mismatch = h->params.mismatch;
    sc.goe = (int)h->params.gap_open + (int)h->params.gap_extend; sc.ge = h->params.gap_extend;
    sc.limit = h->params.score_width ? (1 << (h->params.score_width - 1)) - 1 : 0;
    return sc;
}

std::vector<DevBuf *> all_devbufs(GpuCtx &g)
{
    std::vector<DevBuf *> v = {&g.d_qpacked, &g.d_qoff, &g.d_qlen, &g.d_qidx, &g.d_bnd, &g.d_counters, &g.d_scratch32,
                               &g.d_best_score, &g.d_best_index, &g.d_topk_keys, &g.d_err, &g.d_wave_bnd, &g.d_wave_state, &g.d_wave32_bnd, &g.d_wave32_state, &g.d_wave_rows,
                               &g.d_bnd_aux[0], &g.d_bnd_aux[1], &g.d_bnd_aux[2], &g.d_part_done, &g.d_part_best,
                               &g.d_hits_key2, &g.d_hits_score2, &g.d_sort_tmp};
    for (Slot &b : g.slot) {
        DevBuf *bufs[] = {&b.d_raw, &b.d_off, &b.d_len, &b.d_pair_subj, &b.d_pair_len, &b.d_tile_woff, &b.d_tp, &b.d_out,
                          &b.d_ovf_count, &b.d_ovf_list, &b.d_ovf_score, &b.d_topk_out, &b.d_small_in, &b.d_small_done,
                          &b.d_hits_key, &b.d_hits_score, &b.d_hits_count};
        v.insert(v.end(), std::begin(bufs), std::end(bufs));
    }
    return v;
}

void free_gpu(GpuCtx &g)
{
    cudaSetDevice(g.dev);
    for (DevBuf *d : all_devbufs(g)) d->release();
    for (Slot &b : g.slot) {
        for (cudaEvent_t e : b.ev_pool) cudaEventDestroy(e);
        b.ev_pool.clear();
        b.chunks.clear();
        PinnedBuf *pins[] = {&b.h_stage_a, &b.h_stage_b, &b.h_stage_c, &b.h_stage_d, &b.h_topk, &b.h_ovf, &b.h_hits, &b.h_small_in, &b.h_small_out,
                             &b.h_small_flag};
        for (PinnedBuf *p : pins) p->release();
        if (b.ev_start) cudaEventDestroy(b.ev_start);
        if (b.ev_stop) cudaEventDestroy(b.ev_stop);
        if (b.ev_upload) cudaEventDestroy(b.ev_upload);
    }
    for (cudaStream_t st : g.st_aux) if (st) cudaStreamDestroy(st);
    if (g.ev_fork) cudaEventDestroy(g.ev_fork);
    for (cudaEvent_t e : g.ev_join) if (e) cudaEventDestroy(e);
    if (g.ev_tune0) cudaEventDestroy(g.ev_tune0);
    if (g.ev_tune1) cudaEventDestroy(g.ev_tune1);
    if (g.st_compute) cudaStreamDestroy(g.st_compute);
    if (g.st_copy) cudaStreamDestroy(g.st_copy);
}

int upload_queries(sw_handle *h, GpuCtx &g)
{
    SW_CUDA(h, cudaSetDevice(g.dev));
    const size_t nq = h->q_len.size();
    SW_CUDA(h, g.d_qpacked.reserve(h->q_packed.size() + 16));
    SW_CUDA(h, g.d_qoff.reserve(nq * sizeof(uint32_t)));
    SW_CUDA(h, g.d_qlen.reserve(nq * sizeof(uint32_t)));
    // the compute stream orders these copies before any later kernel
    SW_CUDA(h, cudaMemcpyAsync(g.d_qpacked.p, h->q_packed.data(), h->q_packed.size(), cudaMemcpyHostToDevice, g.st_compute));
    SW_CUDA(h, cudaMemcpyAsync(g.d_qoff.p, h->q_off.data(), nq * sizeof(uint32_t), cudaMemcpyHostToDevice, g.st_compute));
    SW_CUDA(h, cudaMemcpyAsync(g.d_qlen.p, h->q_len.data(), nq * sizeof(uint32_t), cudaMemcpyHostToDevice, g.st_compute));
    SW_CUDA(h, cudaStreamSynchronize(g.st_compute));
    return SW_OK;
}

// Orders the subjects [0, n) by ascending length into g.order (counting sort when the range is
// small, else comparison sort) and records the first few empty ones.
void sort_by_length(Slot &g, const uint32_t *ln, size_t n, uint32_t maxlen)
{
    g.order.resize(n);
    if (maxlen <= (1u << 22) && (size_t)maxlen <= 4 * n + 4096) {
        g.hist.assign((size_t)maxlen + 2, 0);
        for (size_t i = 0; i < n; ++i) g.hist[ln[i] + 1]++;
        for (size_t l = 1; l < g.hist.size(); ++l) g.hist[l] += g.hist[l - 1];
        for (size_t i = 0; i < n; ++i) g.order[g.hist[ln[i]]++] = (uint32_t)i;
    } else {
        for (size_t i = 0; i < n; ++i) g.order[i] = (uint32_t)i;
        std::stable_sort(g.order.begin(), g.order.end(), [&](uint32_t a, uint32_t b) { return ln[a] < ln[b]; });
    }
    g.empties.clear();
    for (size_t i = 0; i < n && ln[g.order[i]] == 0 && g.empties.size() < SW_MAX_TOPK; ++i) g.empties.push_back(g.order[i]);
    std::sort(g.empties.begin(), g.empties.end());
}

// Pairs neighbours in length order: the longer member drives the column loop (low lane), the
// shorter one (high lane) sees PAD columns once it has ended.  Returns the number of pairs;
// pair_subj / pair_len are padded to a multiple of 32 pairs.
size_t make_pairs(const Slot &g, const uint32_t *ln, size_t n, uint32_t *pair_subj, uint32_t *pair_len)
{
    size_t np = 0, i = 0;
    while (i < n && ln[g.order[i]] == 0) ++i;           // empty subjects score 0 (output is pre-zeroed)
    if ((n - i) & 1) {                                  // odd count: the shortest one stays single
        pair_subj[0] = g.order[i]; pair_subj[1] = SW_NO_SUBJECT;
        pair_len[0] = ln[g.order[i]]; pair_len[1] = 0;
        ++i; ++np;
    }
    for (; i + 1 < n; i += 2, ++np) {
        const uint32_t shorter = g.order[i], longer = g.order[i + 1];
        pair_subj[2 * np] = longer; pair_subj[2 * np + 1] = shorter;
        pair_len[2 * np] = ln[longer]; pair_len[2 * np + 1] = ln[shorter];
    }
    const size_t ntiles = (np + 31) / 32;
    for (size_t p = np; p < ntiles * 32; ++p) {
        pair_subj[2 * p] = SW_NO_SUBJECT; pair_subj[2 * p + 1] = SW_NO_SUBJECT;
        pair_len[2 * p] = 0; pair_len[2 * p + 1] = 0;
    }
    return np;
}

// Length groups: from the longest pair down, a group ends where the length has halved (boundaries on
// 32-pair tiles); at most 16 groups.
void build_segments(Slot &g, const uint32_t *pair_len, size_t np)
{
    g.segs.clear();
    size_t hi = np;
    while (hi > 0 && g.segs.size() < 15) {
        const uint32_t lmax = pair_len[2 * (hi - 1)];
        size_t lo = hi;
        // first pair (ascending order) longer than lmax / 2, by binary search
        size_t a = 0, b = hi;
        while (a < b) { const size_t mid = (a + b) / 2; if (pair_len[2 * mid] * 2u > lmax) b = mid; else a = mid + 1; }
        lo = a & ~(size_t)31;
        Seg sg{(uint32_t)lo, (uint32_t)hi, lmax, 0};
        for (size_t p = lo; p < hi; ++p) sg.sum_len += (uint64_t)pair_len[2 * p] + pair_len[2 * p + 1];
        g.segs.push_back(sg);
        hi = lo;
    }
    if (hi > 0) {
        Seg sg{0, (uint32_t)hi, pair_len[2 * (hi - 1)], 0};
        for (size_t p = 0; p < hi; ++p) sg.sum_len += (uint64_t)pair_len[2 * p] + pair_len[2 * p + 1];
        g.segs.push_back(sg);
    }
}

// Length-sorts the shard's subjects, pairs neighbours in length order, lays out 32-pair tiles, uploads.
int load_shard(sw_handle *h, GpuCtx &gc, Slot &g, const uint8_t *packed, const uint32_t *len, const uint64_t *off)
{
    SW_CUDA(h, cudaSetDevice(gc.dev));
    const size_t n = g.s1 - g.s0;
    g.npairs = 0; g.max_len = 0; g.sum_len = 0; g.tp_words = 0; g.is_small = false;
    g.empties.clear();
    if (n == 0) { g.scored = false; return SW_OK; }
    if (n >= 0xFFFFFFF0ull) return SW_EINVAL;
    const uint32_t *ln = len + g.s0;
    const uint64_t *of = off + g.s0;

    uint64_t bmin = ~0ull, bmax = 0;
    uint32_t maxlen = 0;
    uint64_t sum = 0;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t b = (ln[i] + 3ull) >> 2;
        if (ln[i] == 0) continue;
        bmin = std::min(bmin, of[i]);
        bmax = std::max(bmax, of[i] + b);
        maxlen = std::max(maxlen, ln[i]);
        sum += ln[i];
    }
    g.max_len = maxlen; g.sum_len = sum;
    sort_by_length(g, ln, n, maxlen);
    if (maxlen == 0) { g.scored = false; return SW_OK; }

    SW_CUDA(h, g.h_stage_a.reserve((n + 64) * 2 * sizeof(uint32_t)));      // pair_subj
    SW_CUDA(h, g.h_stage_b.reserve((n + 128) * sizeof(uint32_t)));         // pair_len (2 per pair)
    uint32_t *pair_subj = (uint32_t *)g.h_stage_a.p;
    uint32_t *pair_len = (uint32_t *)g.h_stage_b.p;
    const size_t np = make_pairs(g, ln, n, pair_subj, pair_len);
    const size_t ntiles = (np + 31) / 32;
    SW_CUDA(h, g.h_stage_c.reserve((ntiles + 1) * sizeof(uint64_t)));
    uint64_t *tile_woff = (uint64_t *)g.h_stage_c.p;
    uint64_t w = 0;
    for (size_t t = 0; t < ntiles; ++t) {
        tile_woff[t] = w;
        const size_t last = std::min(np, (t + 1) * 32) - 1;     // lengths ascend: last valid pair is longest
        w += 32ull * ((pair_len[2 * last] + 3) / 4);        // one byte per column, 4 per word
    }
    tile_woff[ntiles] = w;
    g.npairs = (uint32_t)np;
    g.tp_words = w;
    build_segments(g, pair_len, np);

    // --- local byte offsets
    SW_CUDA(h, g.h_stage_d.reserve(n * sizeof(uint64_t)));
    uint64_t *loc_off = (uint64_t *)g.h_stage_d.p;
    for (size_t k = 0; k < n; ++k) loc_off[k] = ln[k] ? of[k] - bmin : 0;

    // --- device buffers + uploads (copy stream), then the code-stream build (compute stream)
    const size_t raw_bytes = bmax - bmin;
    SW_CUDA(h, g.d_raw.reserve(raw_bytes + 16));
    SW_CUDA(h, g.d_off.reserve(n * sizeof(uint64_t)));
    SW_CUDA(h, g.d_len.reserve(n * sizeof(uint32_t)));
    SW_CUDA(h, g.d_pair_subj.reserve(ntiles * 32 * 2 * sizeof(uint32_t)));
    SW_CUDA(h, g.d_pair_len.reserve(ntiles * 32 * 2 * sizeof(uint32_t)));
    SW_CUDA(h, g.d_tile_woff.reserve((ntiles + 1) * sizeof(uint64_t)));
    SW_CUDA(h, g.d_tp.reserve((w + 32) * sizeof(uint32_t)));
    cudaStream_t cs = gc.st_copy;
    // the slot's buffers may still be read by scoring kernels queued on the compute stream (sw_score_db
    // is asynchronous): the uploads wait for the tail of that work.  Only this slot's event is waited
    // for, so the other slot's kernels keep overlapping with these copies.
    if (g.scored) {
        if (g.ev_stop_deferred) {                      // an event recorded now still follows that kernel in stream order
            SW_CUDA(h, cudaEventRecord(g.ev_stop, gc.st_compute));
            g.ev_stop_deferred = false;
        }
        SW_CUDA(h, cudaStreamWaitEvent(cs, g.ev_stop, 0));
    }
    g.scored = false;
    SW_CUDA(h, cudaMemcpyAsync(g.d_raw.p, packed + bmin, raw_bytes, cudaMemcpyHostToDevice, cs));
    SW_CUDA(h, cudaMemcpyAsync(g.d_len.p, ln, n * sizeof(uint32_t), cudaMemcpyHostToDevice, cs));
    SW_CUDA(h, cudaMemcpyAsync(g.d_off.p, loc_off, n * sizeof(uint64_t), cudaMemcpyHostToDevice, cs));
    SW_CUDA(h, cudaMemcpyAsync(g.d_pair_subj.p, pair_subj, ntiles * 32 * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, cs));
    SW_CUDA(h, cudaMemcpyAsync(g.d_pair_len.p, pair_len, ntiles * 32 * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, cs));
    SW_CUDA(h, cudaMemcpyAsync(g.d_tile_woff.p, tile_woff, (ntiles + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, cs));
    SW_CUDA(h, cudaEventRecord(g.ev_upload, cs));
    SW_CUDA(h, cudaStreamWaitEvent(gc.st_compute, g.ev_upload, 0));

    SwDevDb db{};
    db.raw = g.d_raw.as<uint8_t>(); db.off = g.d_off.as<uint64_t>(); db.len = g.d_len.as<uint32_t>();
    db.ns = (uint32_t)n; db.pair_subj = g.d_pair_subj.as<uint32_t>(); db.pair_len = g.d_pair_len.as<uint32_t>();
    db.tile_woff = g.d_tile_woff.as<uint64_t>(); db.tp = g.d_tp.as<uint32_t>(); db.tp_words = g.tp_words;
    db.npairs = g.npairs; db.max_len = g.max_len;
    SW_CUDA(h, sw_launch_build_tp(gc.st_compute, db));
    h->launches++;
    return SW_OK;
}

SwDevDb dev_db(const Slot &g)
{
    SwDevDb db{};
    db.raw = g.d_raw.as<uint8_t>(); db.off = g.d_off.as<uint64_t>(); db.len = g.d_len.as<uint32_t>();
    db.ns = (uint32_t)(g.s1 - g.s0); db.pair_subj = g.d_pair_subj.as<uint32_t>();
    db.pair_len = g.d_pair_len.as<uint32_t>(); db.tile_woff = g.d_tile_woff.as<uint64_t>();
    db.tp = g.d_tp.as<uint32_t>(); db.tp_words = g.tp_words; db.npairs = g.npairs; db.max_len = g.max_len;
    return db;
}

SwDevQueries dev_queries(const sw_handle *h, const GpuCtx &gc)
{
    SwDevQueries dq{};
    dq.packed = gc.d_qpacked.as<uint8_t>(); dq.off = gc.d_qoff.as<uint32_t>(); dq.len = gc.d_qlen.as<uint32_t>();
    dq.nq = (int)h->q_len.size(); dq.max_len = h->q_max_len;
    return dq;
}

// Measured steady-state speed of each variant in GCUPS over PADDED cells (150-nt reads,
// profiles/r01_variant_sweep.txt); only the ratios matter for the choice below.
double variant_speed(const SwStripVariant *v)
{
    struct { const char *name; double gcups; } tab[] = {
        {"strip_s16x2_R30x1_G1", 8220}, {"strip_s16x2_R38x1_G1", 8310}, {"strip_s16x2_R75x1_G1", 8040},
        {"strip_s16x2_R32x1_G1", 8230}, {"strip_s16x2_R50x1_G1", 8180}, {"strip_s16x2_R25x2_G1", 8700},
        {"strip_s16x2_R19x2_G1", 7810}, {"strip_s16x2_R15x3_G1", 7590}, {"strip_s16x2_R30x2_G1", 8040},
        {"strip_s16x2_R64x1_G1", 7910}, {"strip_s16x2_R32x2_G1", 8320}, {"strip_s16x2_R25x3_G1", 8620},
        {"strip_s16x2_R38x2_G1", 8600}, {"strip_s16x2_R25x4_G1", 7200}, {"strip_s16x2_R25x1_G2", 7345},
        {"strip_s16x2_R75x1_G2", 7380}, {"strip_s16x2_R25x3_G2", 7480}, {"strip_s16x2_R38x1_G4", 7325},
        {"strip_s16x2_R19x2_G4", 7220}, {"strip_s16x2_R32x1_G4", 7180}, {"strip_s16x2_R16x1_G32", 5980},
        {"strip_s16x2_R8x2_G32", 6320},
        // (R32x2: re-measured on long queries, where its 64-row passes leave no padding: 7 655 vs R38x2 7 653 GCUPS on
        // 200 k x 1 kb x 10 kb, 8 310 vs 8 199 on the mixed-length config 5 -- profiles/r02_variant_ab_long_queries.txt;
        // on the final build ptxas' schedule of R32x2 is the slower one: 8 146 vs R38x2 8 276 on config 5,
        // profiles/r02_pass_split_ab.txt -- launches of one length group still time both, see autotune_variant)
        // small-R latency variants: estimates (shuffle-bound), they are chosen for latency, not throughput
        {"strip_s16x2_R1x1_G32", 900}, {"strip_s16x2_R2x1_G32", 1700}, {"strip_s16x2_R4x1_G32", 3000},
        {"strip_s16x2_R8x1_G32", 4500}, {"strip_s16x2_R8x1_G16", 4600}, {"strip_s16x2_R16x1_G8", 5900},
        {"strip_s16x2_R2x2_G32", 2900},
        // 8 columns per trip: measured +1.6 % on 150-nt reads (profiles/r02_variant_ab_u8.jsonl); the
        // R25x3 / R38x2 counterparts lose 15 % (their loop bodies outgrow the instruction cache)
        {"strip_s16x2_R25x2_G1_U8", 8840}, {"strip_s16x2_R25x3_G1_U8", 7320}, {"strip_s16x2_R38x2_G1_U8", 7390},
        // interior trips: +1.6 % over the 8-column instance (profiles/r02_variant_ab_interior.jsonl)
        {"strip_s16x2_R25x2_G1_U4_F31", 8975},
    };
    for (auto &t : tab) if (std::strcmp(t.name, v->name) == 0) return t.gcups;
    return 5000.0;
}

// Instances whose interior trips drop the L1 prefetch of the boundary row (FL bit 2) are only fast while
// the pass-boundary scratch of all resident blocks stays in L2 (150-nt reads: 68 MB, 8 973 vs 8 833 GCUPS);
// with 1 kb subjects (454 MB of scratch) they lose 5 % to the prefetching instances
// (profiles/r02_variant_ab_interior.jsonl).
double variant_speed_at(const GpuCtx &gc, const SwStripVariant *v, uint32_t max_len)
{
    double sp = variant_speed(v);
    if (v->FL & 4) {
        const double scratch = (double)gc.num_sms * v->min_blocks * (v->block_threads / v->G) * (double)max_len * sizeof(uint2);
        if (scratch > 96.0e6) sp *= 0.9;
    }
    return sp;
}

// Estimated time (arbitrary units) of scoring queries of the given lengths against the shard with
// variant v = padded rows x (columns + pipeline fill) / measured speed / fraction of the GPU the
// pairs can keep busy, plus half the time of the longest work item running at its share of an SM:
// with few, long items the tail of the launch is what matters.
// split: the launch may use the pass split (plan_pass_split), which cuts the item -- and the tail -- into parts.
double variant_cost(const GpuCtx &gc, const Slot &g, const SwStripVariant *v, const uint32_t *qlens, size_t nql, uint32_t maxq,
                    bool split = false)
{
    const int P = v->R * v->G;
    double rows = 0;                      // padded rows over all queries
    for (size_t i = 0; i < nql; ++i) rows += (double)((qlens[i] + P - 1) / P) * P;
    if (rows == 0) rows = (double)((maxq + P - 1) / P) * P;
    // parallel work = lanes of all (pair, query) items of a launch
    const double lanes = (double)g.npairs * v->G * (double)std::max<size_t>(nql, 1);
    const double fill = (double)gc.num_sms * v->min_blocks * v->block_threads;
    const double util = std::min(1.0, lanes / fill);
    const double cols = (double)std::max<uint32_t>(g.max_len, 1);
    const double speed = variant_speed_at(gc, v, g.max_len);
    const double job = rows * (cols + v->G * v->S - 1) / cols * (double)g.sum_len / speed / util;
    const int ppb = v->block_threads / v->G;
    const double qrows = (double)((maxq + P - 1) / P) * P;
    double item = qrows * cols * 2.0 * ppb * ((double)gc.num_sms * v->min_blocks) / speed;
    if (split) {
        // the same arithmetic as plan_pass_split: parts of whole profile chunks, about 20 rounds of items
        const size_t pass_bytes = (size_t)v->G * v->S * ((v->R / v->S + 1) / 2) * 32 * sizeof(uint2);
        const double chunk_rows = (double)std::max<size_t>(1, (48 * 1024) / pass_bytes) * P;
        const double chunks = std::ceil(qrows / chunk_rows);
        const double rounds = std::ceil((double)g.npairs / ppb) * (double)std::max<size_t>(nql, 1) / ((double)gc.num_sms * v->min_blocks);
        if (chunks >= 2.0 && rounds >= 1.0 && rounds < 16.0) item /= std::min(chunks, std::ceil(20.0 / rounds));
    }
    return job + 0.5 * item;
}

// From this many rounds of ONE query's 128-pair items on (2 x SMs) resident blocks the strip kernel with the
// pass split takes partly filled rounds; below it the band-pipelined kernel keeps them.
constexpr double kSplitMinRounds = 1.1;

// launches of the 32-bit band scorer per call (4 096 overflow-list entries each)
constexpr unsigned kWave32Parts = 4;

bool variant_forced(const sw_handle *h) { return h->force_variant >= 0 || h->force_R || h->force_G; }

// Picks the strip variant for a set of queries (least estimated time); ranked = all candidates, best first.
int choose_variant(const sw_handle *h, const GpuCtx &gc, const Slot &g, const uint32_t *qlens, size_t nql, uint32_t maxq,
                   std::vector<int> *ranked = nullptr, bool split = false)
{
    const int nv = sw_strip_variant_count();
    if (h->force_variant >= 0) return h->force_variant;
    if (h->force_R || h->force_G) {
        for (int i = 0; i < nv; ++i) {
            const SwStripVariant *v = sw_strip_variant(i);
            if ((!h->force_R || v->R == h->force_R) && (!h->force_G || v->G == h->force_G))
                return i;
        }
        return -1;
    }
    int best = -1;
    double best_cost = 0;
    std::vector<std::pair<double, int>> costs;
    for (int i = 0; i < nv; ++i) {
        const double cost = variant_cost(gc, g, sw_strip_variant(i), qlens, nql, maxq, split);
        if (best < 0 || cost < best_cost) { best = i; best_cost = cost; }
        costs.emplace_back(cost, i);
    }
    if (ranked) {
        std::sort(costs.begin(), costs.end());
        for (auto &c : costs) ranked->push_back(c.second);
    }
    return best;
}

int cached_occupancy(sw_handle *h, GpuCtx &gc, int vidx, int chunk_passes, int *bps)
{
    auto key = std::make_pair(vidx, chunk_passes);
    auto it = gc.occ_cache.find(key);
    if (it != gc.occ_cache.end()) { *bps = it->second; return SW_OK; }
    SW_CUDA(h, sw_strip_occupancy(vidx, sw_strip_smem_bytes(vidx, chunk_passes), bps));
    gc.occ_cache[key] = *bps;
    return SW_OK;
}

// Launch geometry of a strip variant for `npairs` pairs with subjects up to max_len and queries up to
// maxq rows; also grows the pass-boundary scratch.
int strip_setup(sw_handle *h, GpuCtx &gc, DevBuf &bnd_buf, uint32_t npairs, uint32_t max_len, uint32_t maxq, int nql, int vidx,
                int *grid, int *chunk_passes, size_t *bnd_elems)
{
    const SwStripVariant *v = sw_strip_variant(vidx);
    const int P = v->R * v->G;
    const int need_passes = (int)((maxq + P - 1) / P);
    const size_t pass_bytes = sw_strip_smem_bytes(vidx, 1);
    const int budget_passes = std::max<int>(1, (int)((48 * 1024) / pass_bytes));
    *chunk_passes = std::max(1, std::min(need_passes, budget_passes));
    int bps = 0;
    int rc = cached_occupancy(h, gc, vidx, *chunk_passes, &bps);
    if (rc != SW_OK) return rc;
    if (bps < 1) return SW_ECUDA;
    const int ppb = v->block_threads / v->G;
    const uint32_t npb = (npairs + ppb - 1) / ppb;
    // persistent blocks: as many as there are work items (pair blocks x queries), at most a full GPU
    *grid = (int)std::min<uint64_t>(std::max<uint64_t>((uint64_t)npb * (uint64_t)std::max(nql, 1), 1), (uint64_t)gc.num_sms * bps);
    *bnd_elems = 0;
    if (need_passes > 1) {
        // pass-boundary scratch: one (H, G) per column of the longest subject, per pair slot, per
        // resident block.  A very long subject would make that huge, so the grid shrinks to keep
        // the scratch within a budget.
        const size_t per_block = (size_t)max_len * ppb * sizeof(uint2);
        const size_t budget = (size_t)16 << 30;
        if (per_block > budget) return SW_ENOMEM;
        *grid = (int)std::min<size_t>((size_t)*grid, std::max<size_t>(1, budget / per_block));
        // (a buffer shared by the launches of one stream only ever grows: earlier launches keep fitting)
        if (bnd_buf.cap < (size_t)*grid * per_block) {
            SW_CUDA(h, cudaStreamSynchronize(gc.st_compute));
            for (cudaStream_t st : gc.st_aux) if (st) SW_CUDA(h, cudaStreamSynchronize(st));
            SW_CUDA(h, bnd_buf.reserve((size_t)*grid * per_block));
        }
        *bnd_elems = (size_t)*grid * per_block / sizeof(uint2);
    }
    return SW_OK;
}

// The arithmetic of the pass split, free of any device state (exported for the CPU tests): npass passes in
// profile chunks of chunk_passes, `chains` (pair block, query) chains on `grid` resident blocks (ABI: sw_plan_pass_parts).  mode -1:
// only for 1 <= chains / grid < 16 rounds, aiming at about 20 rounds of part-items; mode n >= 2: about n
// parts.  A part is a whole number of profile chunks.  Returns 1 and the plan, or 0 = do not split.
int plan_pass_parts(int npass, int chunk_passes, unsigned long long chains, int grid, int mode, int *nparts, int *part_passes)
{
    if (nparts) *nparts = 1;
    if (part_passes) *part_passes = npass;
    if (mode == 0 || mode == 1 || mode < -1 || npass < 1 || chunk_passes < 1 || chains < 1) return 0;
    const int chunks = (npass + chunk_passes - 1) / chunk_passes;
    if (chunks < 2) return 0;
    int want = mode;
    if (mode < 0) {
        const double rounds = (double)chains / (double)std::max(grid, 1);
        if (rounds < 1.0 || rounds >= 16.0) return 0;          // under-filled GPU (other kernels' job) / tail already short
        want = (int)std::ceil(20.0 / rounds);
    }
    const int chunks_per_part = std::max(1, chunks / std::max(1, std::min(want, chunks)));
    const int pp = chunks_per_part * chunk_passes;
    const int np = (npass + pp - 1) / pp;
    if (np < 2 || chains * (unsigned long long)np >= (1ull << 31)) return 0;
    if (nparts) *nparts = np;
    if (part_passes) *part_passes = pp;
    return 1;
}

// Pass split (sw_strip.cuh) of a one-launch plan: decides the number of parts, grows the per-chain scratch
// and fills L.nparts / part_passes / part_done / part_best.  Used when the launch is a few rounds of long,
// equally long work items -- rounds = items / resident blocks < 16 -- so that the last, partly filled
// round costs a fraction of a part instead of a whole item: 200 k x 1 kb subjects x one 10 kb query is
// 781 items on 296 blocks = 2.64 rounds (12 % of the GPU-time idle), 8 parts make it 21.1 rounds.
int plan_pass_split(sw_handle *h, GpuCtx &gc, SwStripLaunch &L, uint32_t npairs, uint32_t max_len, uint32_t maxq, int nql_max)
{
    L.nparts = 0; L.part_passes = 0; L.part_done = nullptr; L.part_best = nullptr;
    if (h->pass_split == 0 || L.direct) return SW_OK;
    const SwStripVariant *v = sw_strip_variant(L.vidx);
    const int P = v->R * v->G;
    const int npass = (int)((maxq + P - 1) / P);
    const int chunks = (npass + L.chunk_passes - 1) / L.chunk_passes;       // a part is whole profile chunks
    if (chunks < 2) return SW_OK;
    const int ppb = v->block_threads / v->G;
    const uint64_t npb = (npairs + ppb - 1) / ppb;
    const uint64_t chains = npb * (uint64_t)std::max(nql_max, 1);
    int nparts = 0, part_passes = 0;
    if (!plan_pass_parts(npass, L.chunk_passes, chains, L.grid, h->pass_split, &nparts, &part_passes)) return SW_OK;
    const size_t bnd_bytes = (size_t)chains * (size_t)max_len * ppb * sizeof(uint2);
    size_t free_b = 0, total_b = 0;
    SW_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    if (bnd_bytes > ((size_t)16 << 30) || (gc.d_bnd.cap < bnd_bytes && bnd_bytes - gc.d_bnd.cap > free_b / 2)) return SW_OK;
    if (gc.d_bnd.cap < bnd_bytes || gc.d_part_done.cap < chains * sizeof(unsigned) || gc.d_part_best.cap < chains * v->block_threads * sizeof(uint32_t)) {
        SW_CUDA(h, cudaStreamSynchronize(gc.st_compute));
        for (cudaStream_t st : gc.st_aux) if (st) SW_CUDA(h, cudaStreamSynchronize(st));
        SW_CUDA(h, gc.d_bnd.reserve(bnd_bytes));
        SW_CUDA(h, gc.d_part_done.reserve(chains * sizeof(unsigned)));
        SW_CUDA(h, gc.d_part_best.reserve(chains * v->block_threads * sizeof(uint32_t)));
    }
    L.nparts = nparts; L.part_passes = part_passes;
    L.part_done = gc.d_part_done.as<unsigned>(); L.part_best = gc.d_part_best.as<uint32_t>();
    L.bnd_elems = bnd_bytes / sizeof(uint2);
    return SW_OK;
}

// Pair blocks per super-block of the work order: inside a super-block the queries of a launch pass
// over the same pair blocks one after the other, so its code stream should stay in L2 (about a
// quarter of it: the pass-boundary scratch and the scores live there too) -- but not fewer blocks
// than two full grids, or consecutive items of a thread block stop sharing the query profile.
uint32_t superblock_for(const SwStripVariant *v, uint32_t npairs, uint64_t tp_words, int grid, double sb_mb)
{
    const uint32_t ppb = (uint32_t)(v->block_threads / v->G);
    const uint32_t npb = (npairs + ppb - 1) / ppb;
    if (npb == 0 || tp_words == 0) return 0;
    const double bytes_per_block = (double)tp_words * 4.0 / (double)npb;
    uint32_t b = (uint32_t)std::max(1.0, (sb_mb * 1024 * 1024) / std::max(bytes_per_block, 1.0));
    if (sb_mb >= 8.0) b = std::max<uint32_t>(b, 2u * (uint32_t)std::max(grid, 1));
    b = std::min<uint32_t>(b, std::max<uint32_t>(1u, npb >> 3));
    return std::max<uint32_t>(b, 1u);
}

unsigned *next_counter(GpuCtx &gc)
{
    unsigned *c = gc.d_counters.as<unsigned>() + (gc.counter_next % kMaxCounters);
    gc.counter_next++;
    return c;
}

// Work queue(s) of one strip launch, zeroed on `st`: one counter per query of the launch ("sticky"
// order, sw_strip.cuh) when the launch has 2 .. kMaxStickyQueries queries, else one counter.
const int kMaxStickyQueries = 256;
// Drift bound `sticky` (sw_handle::sticky), measured on config 3 (profiles/r02_traffic.json): 32: 9 000 GCUPS,
// 3.7 GB of DRAM traffic per launch; 96: 8 998, 4.4 GB; none: 9 001, 14.9 GB; super-block order: 8 971, 19.2 GB.
cudaError_t assign_counters(GpuCtx &gc, SwStripLaunch &L, cudaStream_t st, int sticky_mode, bool equal_queries, uint64_t tp_words)
{
    // (queries of different lengths: the blocks of the short ones finish early and pile onto the long
    // ones' queues -- config 5: 7 799 vs 8 302 GCUPS -- so only launches of equally long queries)
    const bool sticky = sticky_mode && equal_queries && L.nql >= 2 && L.nql <= kMaxStickyQueries;
    const unsigned n = sticky ? (unsigned)L.nql : 1u;
    if (gc.counter_next % kMaxCounters + n > (unsigned)kMaxCounters) gc.counter_next += kMaxCounters - gc.counter_next % kMaxCounters;
    L.counter = gc.d_counters.as<unsigned>() + (gc.counter_next % kMaxCounters);
    gc.counter_next += n;
    if (sticky && sticky_mode < 0) {
        const double bytes_per_block = L.db.npairs ? (double)tp_words * 4.0 * 128.0 / (double)L.db.npairs : 1.0;
        L.sticky = (int)std::min(32.0, std::max(4.0, 1048576.0 / std::max(bytes_per_block, 1.0)));
    } else {
        L.sticky = sticky ? sticky_mode : 0;
    }
    return cudaMemsetAsync(L.counter, 0, n * sizeof(unsigned), st);
}

// Times the model's best candidates on a window of the pair list (middle of the length order)
// and a few queries; *choice = the fastest.  Every variant produces identical scores, so the
// sample launches may write into the real output buffer.  Returns a status; the events live in
// the GpuCtx, so no exit path leaks them.
int autotune_variant(sw_handle *h, GpuCtx &gc, Slot &g, SwStripLaunch base, const std::vector<int> &ranked, int nq, bool equal_queries, int *choice)
{
    *choice = ranked[0];
    const int ncand = std::min<int>(3, (int)ranked.size());
    const int nqs = std::min(nq, 8);
    uint64_t qrows = 0;
    for (int q = 0; q < nqs; ++q) qrows += h->q_len[q];
    const double mean_len = (double)g.sum_len / (double)std::max<size_t>(g.s1 - g.s0, 1);
    const double cells_per_pair = 2.0 * mean_len * (double)std::max<uint64_t>(qrows, 1);
    uint64_t pairs_s = (uint64_t)(1.5e11 / cells_per_pair);                      // ~20 ms of work
    pairs_s = std::max<uint64_t>(pairs_s, (uint64_t)gc.num_sms * 4 * 128 * 4);   // >= 4 waves of blocks
    pairs_s = std::min<uint64_t>(pairs_s, g.npairs) & ~31ull;
    if (pairs_s < 1024) return SW_OK;
    const uint64_t p0 = ((g.npairs - pairs_s) / 2) & ~31ull;
    base.db.pair_subj += 2 * p0;
    base.db.pair_len += 2 * p0;
    base.db.tile_woff += p0 / 32;
    base.db.npairs = (uint32_t)pairs_s;
    base.q0 = 0; base.nql = nqs; base.qidx = nullptr;
    if (!gc.ev_tune0) SW_CUDA(h, cudaEventCreate(&gc.ev_tune0));
    if (!gc.ev_tune1) SW_CUDA(h, cudaEventCreate(&gc.ev_tune1));
    float best_ms = 0.f;
    for (int c = 0; c < ncand; ++c) {
        base.vidx = ranked[c];
        int rc = strip_setup(h, gc, gc.d_bnd, base.db.npairs, g.max_len, h->q_max_len, nqs, base.vidx, &base.grid, &base.chunk_passes, &base.bnd_elems);
        if (rc != SW_OK) return rc;
        base.bnd = gc.d_bnd.as<uint2>();
        float ms = 0.f;
        for (int rep = 0; rep < 2; ++rep) {  // first run warms caches and the instruction cache
            SW_CUDA(h, assign_counters(gc, base, gc.st_compute, h->sticky, equal_queries, g.tp_words * (uint64_t)base.db.npairs / std::max<uint32_t>(g.npairs, 1)));
            SW_CUDA(h, cudaEventRecord(gc.ev_tune0, gc.st_compute));
            SW_CUDA(h, sw_launch_strip(gc.st_compute, base));
            h->launches++;
            SW_CUDA(h, cudaEventRecord(gc.ev_tune1, gc.st_compute));
            SW_CUDA(h, cudaEventSynchronize(gc.ev_tune1));
            SW_CUDA(h, cudaEventElapsedTime(&ms, gc.ev_tune0, gc.ev_tune1));
        }
        if (c == 0 || ms < best_ms) { *choice = base.vidx; best_ms = ms; }
    }
    return SW_OK;
}

cudaEvent_t pool_event(sw_handle *h, Slot &g, size_t i, int *rc)
{
    *rc = SW_OK;
    while (g.ev_pool.size() <= i) {
        cudaEvent_t e = nullptr;
        cudaError_t ce = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        if (ce != cudaSuccess) { h->last_cuda.store((int)ce); *rc = SW_ECUDA; return nullptr; }
        g.ev_pool.push_back(e);
    }
    return g.ev_pool[i];
}

// One group of queries that run with the same variant (q empty = all queries, contiguous).
struct QueryGroup { int vidx; std::vector<int> q; uint64_t rows; };

int score_gpu(sw_handle *h, GpuCtx &gc, Slot &g)
{
    if (&gc == &h->gpus[0]) h->last_parts = 1;
    SW_CUDA(h, cudaSetDevice(gc.dev));
    const int nq = (int)h->q_len.size();
    const size_t n = g.s1 - g.s0;
    g.chunks.clear();
    g.scored = true;
    g.ovf_used = false;
    g.out_mode = h->topk_k > 0 ? SW_OUT_TOPK : h->hits_min > 0 ? SW_OUT_HITS : h->out_mode;
    g.topk_k = h->topk_k;
    if (n == 0 || nq == 0) return SW_OK;
    const bool topk = g.out_mode == SW_OUT_TOPK;
    const bool hits = g.out_mode == SW_OUT_HITS;
    const size_t esz = g.out_mode == SW_OUT_I16 ? sizeof(int16_t) : sizeof(int32_t);

    // hit list: keys row << hits_shift | shard-local subject (the fetch sorts them: row-major order)
    SwHitList hl;
    if (hits) {
        int sb = 0;
        while ((1ull << sb) < (uint64_t)n) ++sb;
        g.hits_shift = sb;
        SW_CUDA(h, g.d_hits_count.reserve(sizeof(unsigned long long)));
        SW_CUDA(h, g.d_hits_key.reserve(h->hits_max * sizeof(unsigned long long)));
        SW_CUDA(h, g.d_hits_score.reserve(h->hits_max * sizeof(int32_t)));
        SW_CUDA(h, cudaMemsetAsync(g.d_hits_count.p, 0, sizeof(unsigned long long), gc.st_compute));
        hl.keys = g.d_hits_key.as<unsigned long long>(); hl.score = g.d_hits_score.as<int32_t>();
        hl.count = g.d_hits_count.as<unsigned long long>(); hl.cap = (unsigned)h->hits_max;
        hl.min_score = h->hits_min; hl.shift = sb;
    } else if (!topk) {
        SW_CUDA(h, g.d_out.reserve((size_t)nq * n * esz));
        SW_CUDA(h, cudaMemsetAsync(g.d_out.p, 0, (size_t)nq * n * esz, gc.st_compute));
    } else {
        SW_CUDA(h, g.d_topk_out.reserve((size_t)nq * g.topk_k * sizeof(unsigned long long)));
        SW_CUDA(h, cudaMemsetAsync(g.d_topk_out.p, 0, (size_t)nq * g.topk_k * sizeof(unsigned long long), gc.st_compute));
    }
    SW_CUDA(h, cudaEventRecord(g.ev_start, gc.st_compute));
    int rc = SW_OK;
    if (g.npairs == 0) {
        SW_CUDA(h, cudaEventRecord(g.ev_stop, gc.st_compute));
        g.ev_stop_deferred = false;
        QueryChunk c{0, nq, pool_event(h, g, 0, &rc)};
        if (rc != SW_OK) return rc;
        SW_CUDA(h, cudaEventRecord(c.done, gc.st_compute));
        g.chunks.push_back(c);
        return SW_OK;
    }

    const SwScoring sc = scoring_of(h);
    const SwDevDb db = dev_db(g);
    const SwDevQueries dq = dev_queries(h, gc);

    // Value range: the packed 16-bit kernel is always used; when match * min(m, n) could exceed
    // the 16-bit range it flags the (rare) pairs whose running maximum got near 32767: they go to
    // the overflow list and the 32-bit kernel recomputes exactly those.
    const uint64_t smax = (uint64_t)sc.match * std::min<uint64_t>(h->q_max_len, g.max_len);
    const bool may_overflow = !sc.limit && (smax + (uint64_t)sc.match >= 32000ull);
    SW_CUDA(h, gc.d_counters.reserve(kMaxCounters * sizeof(unsigned)));

    // ---- few, long pairs: the bands of a long query become concurrent work items (sw_wave.cuh) ----
    std::vector<int> wave_q, strip_q;
    {
        // (top-k: the band-pipelined kernel fills a scratch row per query, whose top k then join the key lists)
        const bool wave_ok = h->wave && !sc.limit && !h->force32 && !variant_forced(h);
        // Besides "few pairs": whenever the long queries' work items (128 pairs x all passes) would
        // leave the strip kernel's last round mostly empty.  Measured (profiles/r02_wave_vs_strip_mid.txt):
        // the band-pipelined kernel holds 7.2-7.5 TCUPS from 3 000 to 100 000 pairs, the strip kernel
        // 8.1 TCUPS at exactly two full rounds but 4.9-6.9 below and between whole rounds.
        size_t n_long = 0;
        for (int q = 0; q < nq; ++q) n_long += (h->q_len[q] >= 2 * SW_WAVE_ROWS_PER_BAND && h->q_len[q] <= 4000u * 256u) ? 1 : 0;
        const double rounds = (double)((g.npairs + 127) / 128) * (double)n_long / ((double)gc.num_sms * 2.0);
        // (only when every query is long: shorter ones in the same launch fill the strip kernel's rounds)
        // With the pass split (one launch, equally long queries) the strip kernel no longer pays for a
        // partly filled last round, so from one full round on it is the faster one
        // (profiles/r02_pass_split_ab.txt: 8.4-8.8 TCUPS against the band-pipelined 7.2-7.6).
        // -- when ONE query's items fill kSplitMinRounds rounds (the queries of a call may go out as separate
        // launches: 3 x 4 kb queries x 60 000 x 2 kb, 0.79 rounds per query, strip + split 6 160 vs 7 794 GCUPS).
        // scripts/split_ab.py, profiles/r02_pass_split_ab.txt: 10 kb x 100 000 x 1 kb (1.32 rounds) 7 340 -> 8 492,
        // x 120 000 (1.58) 7 343 -> 8 660, x 151 552 (2.00) 8 327 -> 8 758, x 260 000 (3.43) 8 417 -> 8 756.
        bool split_possible = h->pass_split != 0 && n_long > 0 && rounds / (double)std::max<size_t>(n_long, 1) >= kSplitMinRounds;
        for (int q = 1; q < nq; ++q) split_possible = split_possible && h->q_len[q] == h->q_len[0];
        const bool underfilled = n_long == (size_t)nq &&
                                 (rounds < 1.05 || (!split_possible && rounds < 4.0 && rounds / std::ceil(rounds) < 0.85));
        const double bnd_bytes = (double)g.npairs * 2.0 * ((double)g.max_len + 64.0) * 16.0;      // tagged boundary rows of all pairs
        const bool bnd_fits = bnd_bytes <= 4.0e9, bnd_fits_few = bnd_bytes <= 16.0e9;
        for (int q = 0; q < nq; ++q) {
            const uint32_t ql = h->q_len[q];
            bool w = false;
            if (wave_ok && ql > SW_WAVE_ROWS_PER_BAND && ql <= 4000u * 256u) {
                if (h->wave >= 2) w = true;
                else w = (bnd_fits_few && ((g.npairs <= 1536 && ql >= 2 * SW_WAVE_ROWS_PER_BAND) || g.npairs <= 64)) ||
                         (ql >= 2 * SW_WAVE_ROWS_PER_BAND && underfilled && bnd_fits);
            }
            (w ? wave_q : strip_q).push_back(q);
        }
    }

    // ---- launch plan ---------------------------------------------------------------------------
    // Simple case (one length group, every query on one variant -- the bulk case, config 3): query
    // chunks on the compute stream, D2H of finished rows overlapping the next chunk, the model's top
    // candidates timed on a sample.  General case: every (length group, query group) gets its own
    // launch and variant; launches run on several streams so that the tail of one overlaps the
    // start of the next, longest work items first.
    struct Planned { SwStripLaunch L; int q0, q1; int stream; double item_s; };
    std::vector<Planned> plan;
    std::vector<int> &qidx_host = g.qidx_host;     // stays alive until this slot is scored again
    qidx_host.clear();
    std::vector<int> ranked;
    int max_grid = 0;
    bool simple = false, jit_used = false, sticky_ok = false;
    int label_v = -1;
    size_t n_groups_total = 0;

    SwStripLaunch base;
    base.db = db; base.q = dq; base.sc = sc;
    base.out = (topk || hits) ? nullptr : g.d_out.p; base.out_stride = n; base.out_elems = hits ? h->hits_max : (size_t)nq * n;
    base.out_mode = g.out_mode;
    base.hits = hl;
    base.dev_err = gc.d_err.as<unsigned>();
    if (may_overflow) {
        SW_CUDA(h, g.d_ovf_count.reserve(sizeof(unsigned)));
        SW_CUDA(h, g.d_ovf_list.reserve((size_t)kOvfCap * sizeof(uint2)));
        SW_CUDA(h, g.d_ovf_score.reserve((size_t)kOvfCap * sizeof(int32_t)));
        SW_CUDA(h, cudaMemsetAsync(g.d_ovf_count.p, 0, sizeof(unsigned), gc.st_compute));
        base.ovf_count = g.d_ovf_count.as<unsigned>(); base.ovf_list = g.d_ovf_list.as<uint2>(); base.ovf_cap = kOvfCap;
        g.ovf_used = true;
    }

    if (!h->force32 && !strip_q.empty()) {
        std::vector<uint32_t> sl;
        uint32_t smaxq = 0;
        uint64_t srows = 0;
        for (int q : strip_q) { sl.push_back(h->q_len[q]); smaxq = std::max(smaxq, h->q_len[q]); srows += h->q_len[q]; }
        const bool all_strip = (int)strip_q.size() == nq;
        const bool same_len = std::all_of(sl.begin(), sl.end(), [&](uint32_t x) { return x == sl[0]; });
        std::vector<Seg> segs = g.segs;
        bool use_segs = h->plan_segs == 1;
        if (h->plan_segs == 2 && segs.size() > 1) {
            // one launch over everything sizes every block's pass-boundary scratch by the longest subject
            const size_t worst = (size_t)gc.num_sms * 4 * 128 * (size_t)g.max_len * sizeof(uint2);
            use_segs = smaxq > 64 && worst > ((size_t)4 << 30);
        }
        if (segs.empty() || variant_forced(h) || !use_segs) segs.assign(1, Seg{0, g.npairs, g.max_len, g.sum_len});
        simple = all_strip && segs.size() == 1 && (variant_forced(h) || same_len || strip_q.size() == 1);
        sticky_ok = same_len;

        if (simple) {
            // (the split-aware tail term of variant_cost stays off: with it the model prefers the 3-blocks-per-SM
            // R25x2 instances for 10 kb queries, whose table speed was measured on single-chunk 150-nt reads --
            // scripts/split_ab.py: 8 059 vs 8 752 GCUPS with R38x2 at two rounds, 8 362 vs 8 780 on 200 k x 1 kb)
            int vidx = choose_variant(h, gc, g, sl.data(), sl.size(), smaxq, &ranked, false);
            if (vidx < 0) return SW_EINVAL;
            const double est_ms_all = (double)g.sum_len * (double)srows / 6.0e9;
            if (h->pass_split != 0 && !variant_forced(h) && sw_strip_variant(vidx)->G > 1) {
                // The model asks for more lanes per pair because whole items of a one-lane variant would leave
                // the last round partly empty.  With the pass split that round costs a fraction of a part, so a
                // one-lane variant is the faster one as soon as its chains fill the GPU once
                // (scripts/split_ab.py: 10 kb x 120 000 x 1 kb: R38x1_G4 7 014, band-pipelined 7 340, R32x2_G1 8 390 GCUPS).
                const int nchunks_est = (topk || hits || may_overflow || !wave_q.empty()) ? 1 : std::max(1, std::min(std::min(nq, 8), (int)(est_ms_all / 50.0)));
                const uint64_t nql_launch = (uint64_t)std::max(1, nq / nchunks_est);
                for (int cand : ranked) {
                    const SwStripVariant *cv = sw_strip_variant(cand);
                    if (cv->G != 1) continue;
                    const int P = cv->R;
                    const int npass = (int)((smaxq + P - 1) / P);
                    const int cp = std::max(1, std::min<int>(npass, (int)((48 * 1024) / sw_strip_smem_bytes(cand, 1))));
                    const uint64_t chains = (uint64_t)((g.npairs + cv->block_threads - 1) / cv->block_threads) * nql_launch;
                    if ((npass + cp - 1) / cp >= 2 && (double)chains >= 1.05 * (double)gc.num_sms * cv->min_blocks) { vidx = cand; break; }
                }
            }
            // large jobs: let the GPU pick among the model's top candidates (decision cached per workload shape)
            base.bnd_cols = g.max_len;
            if (!topk && h->autotune && !variant_forced(h) && est_ms_all >= 400.0 && ranked.size() > 1) {
                uint64_t key = 1469598103934665603ull;
                auto log2b = [](uint64_t x) { uint64_t b = 0; while (x >>= 1) ++b; return b; };
                const uint64_t parts[] = {h->q_max_len, h->q_sum_len, (uint64_t)nq, g.max_len, log2b(g.npairs), log2b(g.sum_len),
                                          (uint64_t)(uint16_t)h->params.match, (uint64_t)(uint16_t)h->params.mismatch,
                                          (uint64_t)(uint16_t)h->params.gap_open, (uint64_t)(uint16_t)h->params.gap_extend,
                                          (uint64_t)h->params.score_width, (uint64_t)g.out_mode};
                for (uint64_t x : parts) { key ^= x; key *= 1099511628211ull; }
                if (gc.tune_key != key || gc.tune_choice < 0) {
                    int choice = vidx;
                    // the sample launches append nothing: a pair they score is scored again by the real launch
                    SwStripLaunch sample = base;
                    if (hits) { sample.hits.keys = nullptr; sample.ovf_list = nullptr; sample.ovf_count = nullptr; }
                    rc = autotune_variant(h, gc, g, sample, ranked, nq, same_len, &choice);
                    if (rc != SW_OK) return rc;
                    gc.tune_choice = choice;
                    gc.tune_key = key;
                }
                vidx = gc.tune_choice;
            }
            // query chunks: a handful of launches so that D2H of finished rows overlaps compute
            // (each launch has its own tail: aim for >= ~50 ms of work per launch, at ~6 TCUPS)
            int nchunks = std::max(1, std::min(std::min(nq, 8), (int)(est_ms_all / 50.0)));
            if (topk || hits || may_overflow || !wave_q.empty()) nchunks = 1;
            // the device work counter is 32-bit: (pair blocks) x (queries per launch) must stay below 2^31
            while (nchunks < nq && (uint64_t)(g.npairs / 4 + 1) * (uint64_t)((nq + nchunks - 1) / nchunks) >= (1ull << 31)) nchunks *= 2;
            nchunks = std::min(nchunks, nq);
            SwStripLaunch L = base;
            L.vidx = vidx;
            rc = strip_setup(h, gc, gc.d_bnd, g.npairs, g.max_len, smaxq, nq / nchunks, vidx, &L.grid, &L.chunk_passes, &L.bnd_elems);
            if (rc != SW_OK) return rc;
            L.superblock = superblock_for(sw_strip_variant(vidx), g.npairs, g.tp_words, L.grid, h->superblock_mb);
            rc = plan_pass_split(h, gc, L, g.npairs, g.max_len, smaxq, (nq + nchunks - 1) / nchunks);
            if (rc != SW_OK) return rc;
            if (&gc == &h->gpus[0]) h->last_parts = std::max(1, L.nparts);
            max_grid = L.grid;
            label_v = vidx;
            n_groups_total = 1;
            if (h->jit && !sc.limit && (est_ms_all >= 2000.0 || h->jit >= 2) && std::strcmp(sw_strip_instance_kind(L), "runtime") == 0) {
                L.jit_kernel = sw_jit_strip_kernel(sw_strip_variant(vidx), sc.goe, sc.ge, nullptr, 0);
                jit_used = L.jit_kernel != nullptr;
            }
            // (A "tail split" -- the pairs of the last, partly filled round of equal work items on a
            // side stream with a 2- or 4-lane variant -- was built and measured on 200 k x 1 kb x 10 kb:
            // 262.9 ms against 261.0 ms without it.  The finer items gain what the slower variant loses.)
            for (int c = 0; c < nchunks; ++c) {
                const int a0 = (int)((long long)nq * c / nchunks), a1 = (int)((long long)nq * (c + 1) / nchunks);
                if (a1 <= a0) continue;
                Planned p{L, a0, a1, 0, 0.0};
                p.L.q0 = a0; p.L.nql = a1 - a0; p.L.qidx = nullptr;
                plan.push_back(p);
            }
        } else {
            // lanes needed to keep the GPU busy decide the least lanes per pair; the time budget of a
            // single work item decides when a length group needs more lanes per pair than that
            const double fill = (double)gc.num_sms * 3 * 128;
            int gmin = 1;
            while (gmin < 32 && (double)g.npairs * gmin * (double)strip_q.size() < 0.6 * fill) gmin *= 2;
            const double t_total = (double)g.sum_len * (double)srows / 8.0e12;          // seconds, optimistic
            const double tau = std::max(h->plan_tau * t_total, 1.0e-3);      // the longest items start first
            const int nv = sw_strip_variant_count();
            auto pick = [&](const Seg &sg, const uint32_t *ql, size_t nql, uint32_t maxq, double *item_s) {
                if (const char *e = std::getenv("SW_B200_PLAN_FORCE")) {          // A/B measurements: this variant for every group
                    for (int i = 0; i < nv; ++i) if (std::strcmp(sw_strip_variant(i)->name, e) == 0) { *item_s = 1.0; return i; }
                }
                int best = -1, best_any = -1;
                double best_thr = 0, best_any_cost = 0, best_item = 0, best_any_item = 0;
                const double cols_avg = std::max(1.0, (double)sg.sum_len / (2.0 * std::max<uint32_t>(sg.p1 - sg.p0, 1)));
                for (int i = 0; i < nv; ++i) {
                    const SwStripVariant *v = sw_strip_variant(i);
                    if (v->U != 4) continue;                                     // experimental instances: by name only
                    const int P = v->R * v->G, vpe = v->G * v->S;
                    double rows = 0;
                    for (size_t k = 0; k < nql; ++k) rows += (double)((ql[k] + P - 1) / P) * P;
                    const double speed = variant_speed_at(gc, v, sg.max_len) * 1e9;
                    const double thr = rows * (double)sg.sum_len * (cols_avg + vpe - 1) / cols_avg / speed;
                    const double qrows = (double)((maxq + P - 1) / P) * P;
                    const int ppb = v->block_threads / v->G;
                    const double item = qrows * ((double)sg.max_len + vpe - 1) * 2.0 * ppb * ((double)gc.num_sms * v->min_blocks) / speed;
                    const double any_cost = thr + item + (v->G < gmin ? 10.0 * thr : 0.0);
                    if (best_any < 0 || any_cost < best_any_cost) { best_any = i; best_any_cost = any_cost; best_any_item = item; }
                    if (v->G < gmin || item > tau) continue;
                    if (best < 0 || thr < best_thr) { best = i; best_thr = thr; best_item = item; }
                }
                *item_s = best >= 0 ? best_item : best_any_item;
                return best >= 0 ? best : best_any;
            };
            std::map<int, uint64_t> rows_by_variant;
            for (const Seg &sg : segs) {
                if (sg.p1 <= sg.p0) continue;
                // queries of this length group, grouped by the variant that suits them
                std::map<int, std::vector<int>> by_variant;
                std::map<int, double> item_of;
                if (h->plan_qgroups) {
                    for (int q : strip_q) {
                        const uint32_t ql = h->q_len[q];
                        double it = 0;
                        const int v = pick(sg, &ql, 1, ql, &it);
                        by_variant[v].push_back(q);
                        item_of[v] = std::max(item_of[v], it);
                    }
                } else {
                    double it = 0;
                    const int v = pick(sg, sl.data(), sl.size(), smaxq, &it);
                    by_variant[v] = strip_q;
                    item_of[v] = it;
                }
                // fold small groups into the largest one of this length group (every launch has a tail)
                int big = -1;
                uint64_t big_rows = 0, all_rows = 0;
                std::map<int, uint64_t> vrows;
                for (auto &kv : by_variant) {
                    uint64_t r = 0;
                    for (int q : kv.second) r += h->q_len[q];
                    vrows[kv.first] = r;
                    all_rows += r;
                    if (r >= big_rows) { big_rows = r; big = kv.first; }
                }
                for (auto it = by_variant.begin(); it != by_variant.end();) {
                    const double ms = (double)sg.sum_len * (double)vrows[it->first] / 8.0e9;
                    if (it->first != big && (ms < 2.0 || (double)vrows[it->first] < 0.03 * (double)all_rows)) {
                        std::vector<int> &dst = by_variant[big];
                        dst.insert(dst.end(), it->second.begin(), it->second.end());
                        vrows[big] += vrows[it->first];
                        it = by_variant.erase(it);
                    } else {
                        ++it;
                    }
                }
                for (auto &kv : by_variant) {
                    std::vector<int> &ql = kv.second;
                    // longest queries first inside a super-block: the longest work items start earliest
                    std::sort(ql.begin(), ql.end(), [&](int x, int y) { return h->q_len[x] != h->q_len[y] ? h->q_len[x] > h->q_len[y] : x < y; });
                    uint32_t gmaxq = 0;
                    for (int q : ql) gmaxq = std::max(gmaxq, h->q_len[q]);
                    Planned p{base, 0, 0, 0, item_of[kv.first]};
                    SwStripLaunch &L = p.L;
                    L.vidx = kv.first;
                    // this length group's window of the pair list
                    L.db.pair_subj = db.pair_subj + 2 * (size_t)sg.p0;
                    L.db.pair_len = db.pair_len + 2 * (size_t)sg.p0;
                    L.db.tile_woff = db.tile_woff + sg.p0 / 32;
                    L.db.npairs = sg.p1 - sg.p0;
                    L.db.max_len = sg.max_len;
                    L.bnd_cols = sg.max_len;
                    L.q0 = 0; L.nql = (int)ql.size();
                    L.qidx = (const int *)(uintptr_t)qidx_host.size();          // offset for now, pointer after the upload
                    qidx_host.insert(qidx_host.end(), ql.begin(), ql.end());
                    rows_by_variant[kv.first] += vrows[kv.first] * (sg.sum_len >> 8);
                    plan.push_back(p);
                    ++n_groups_total;
                }
            }
            // longest work items first, round-robin over the streams
            std::stable_sort(plan.begin(), plan.end(), [](const Planned &x, const Planned &y) { return x.item_s > y.item_s; });
            const int ns_used = topk ? 1 : h->plan_streams;   // top-k lists are per block index: one kernel at a time
            for (size_t i = 0; i < plan.size(); ++i) plan[i].stream = (int)(i % ns_used);
            SW_CUDA(h, gc.d_qidx.reserve(std::max<size_t>(1, qidx_host.size()) * sizeof(int)));
            for (Planned &p : plan) {
                SwStripLaunch &L = p.L;
                const size_t off = (size_t)(uintptr_t)L.qidx;
                L.qidx = gc.d_qidx.as<int>() + off;
                uint32_t gmaxq = 0;
                for (int k = 0; k < L.nql; ++k) gmaxq = std::max(gmaxq, h->q_len[qidx_host[off + k]]);
                DevBuf &bb = p.stream == 0 ? gc.d_bnd : gc.d_bnd_aux[p.stream - 1];
                rc = strip_setup(h, gc, bb, L.db.npairs, L.db.max_len, gmaxq, L.nql, L.vidx, &L.grid, &L.chunk_passes, &L.bnd_elems);
                if (rc != SW_OK) return rc;
                // more work items than the 32-bit work counter can address: does not happen per length group
                max_grid = std::max(max_grid, L.grid);
                if (h->jit >= 2 && !sc.limit && std::strcmp(sw_strip_instance_kind(L), "runtime") == 0) {
                    L.jit_kernel = sw_jit_strip_kernel(sw_strip_variant(L.vidx), sc.goe, sc.ge, nullptr, 0);
                    jit_used |= L.jit_kernel != nullptr;
                }
            }
            uint64_t lr = 0;
            for (auto &kv : rows_by_variant) if (kv.second >= lr) { lr = kv.second; label_v = kv.first; }
            SW_CUDA(h, cudaMemcpyAsync(gc.d_qidx.p, qidx_host.data(), qidx_host.size() * sizeof(int), cudaMemcpyHostToDevice, gc.st_compute));
        }
    }
    if (&gc == &h->gpus[0]) {      // one writer: the per-GPU workers run concurrently
        if (label_v >= 0)
            std::snprintf(h->last_kernel, sizeof h->last_kernel, "%s%s%s", sw_strip_variant(label_v)->name, jit_used ? "+jit" : "",
                          n_groups_total > 1 ? "+groups" : "");
        else
            std::snprintf(h->last_kernel, sizeof h->last_kernel, "%s", wave_q.empty() ? "generic32" : sw_wave_kernel_name(0));
        if (!wave_q.empty() && label_v >= 0) {
            uint64_t wrows = 0;
            for (int q : wave_q) wrows += h->q_len[q];
            if (2 * wrows > h->q_sum_len) std::snprintf(h->last_kernel, sizeof h->last_kernel, "%s+groups", sw_wave_kernel_name(0));
        }
    }
    const bool have_strip = !plan.empty();

    const bool use32 = !have_strip && wave_q.empty();        // forced 32-bit scorer
    if (topk) {
        if (!have_strip && wave_q.empty()) return SW_EINVAL;  // the 32-bit scorer has no top-k epilogue
        if (!wave_q.empty()) max_grid = std::max(max_grid, 1);      // list 0 also takes the rows of the band-pipelined queries
        const size_t bytes = (size_t)max_grid * nq * g.topk_k * sizeof(unsigned long long);
        SW_CUDA(h, gc.d_topk_keys.reserve(bytes));
        SW_CUDA(h, cudaMemsetAsync(gc.d_topk_keys.p, 0, bytes, gc.st_compute));
    }

    if (hits && use32) return SW_EINVAL;                      // (rejected at submit: the 32-bit scorer has no hit list)
    if ((topk || hits) && !wave_q.empty()) {
        const size_t rb = wave_q.size() * (size_t)n * sizeof(int32_t);
        SW_CUDA(h, gc.d_wave_rows.reserve(rb));
        SW_CUDA(h, cudaMemsetAsync(gc.d_wave_rows.p, 0xFF, rb, gc.st_compute));    // -1 = not scored here
    }

    // 32-bit scratch (force32, or the overflow fix-up of the few listed pairs)
    const uint32_t max_cols = std::max<uint32_t>(1, std::min<uint32_t>(h->q_max_len, g.max_len));
    int threads32 = 0;
    if (use32 || may_overflow) {
        const size_t budget = (size_t)1 << 30;
        size_t t = budget / ((size_t)2 * max_cols * sizeof(int32_t));
        t = std::min<size_t>(t, use32 ? (size_t)gc.num_sms * 2 * 128 : 4096);
        t = std::max<size_t>(128, t / 128 * 128);
        threads32 = (int)t;
        SW_CUDA(h, gc.d_scratch32.reserve((size_t)2 * max_cols * threads32 * sizeof(int32_t)));
    }
    SwScore32Launch s32;
    s32.db = db; s32.q = dq; s32.sc = sc; s32.out = (topk || hits) ? nullptr : g.d_out.p; s32.out_stride = n; s32.out_mode = g.out_mode;
    s32.scratch = gc.d_scratch32.as<int32_t>(); s32.max_cols = max_cols; s32.threads_total = threads32;

    size_t nev = 0;
    if (!use32) {
        const bool chunk_events = simple && plan.size() > 1 && !may_overflow && !topk && !hits;
        bool forked[kStreams] = {false, false, false, false};
        for (size_t i = 0; i < plan.size(); ++i) {
            Planned &p = plan[i];
            cudaStream_t st = gc.st_compute;
            if (p.stream > 0) {
                st = gc.st_aux[p.stream - 1];
                if (!forked[p.stream]) {
                    // the side streams start after everything queued on the compute stream so far
                    // (output memset, query lists, an earlier batch's kernels)
                    if (!forked[0]) { SW_CUDA(h, cudaEventRecord(gc.ev_fork, gc.st_compute)); forked[0] = true; }
                    SW_CUDA(h, cudaStreamWaitEvent(st, gc.ev_fork, 0));
                    forked[p.stream] = true;
                }
            }
            p.L.bnd = (p.stream == 0 ? gc.d_bnd : gc.d_bnd_aux[p.stream - 1]).as<uint2>();
            SW_CUDA(h, assign_counters(gc, p.L, st, p.L.nparts > 1 ? 0 : h->sticky, simple && sticky_ok, g.tp_words));
            if (p.L.nparts > 1) {
                const SwStripVariant *pv = sw_strip_variant(p.L.vidx);
                const size_t chains = (size_t)((p.L.db.npairs + pv->block_threads / pv->G - 1) / (pv->block_threads / pv->G)) * (size_t)p.L.nql;
                SW_CUDA(h, cudaMemsetAsync(p.L.part_done, 0, chains * sizeof(unsigned), st));
            }
            if (topk) { p.L.topk_keys = gc.d_topk_keys.as<unsigned long long>(); p.L.topk_k = g.topk_k; p.L.topk_nq = nq; }
            SW_CUDA(h, sw_launch_strip(st, p.L));
            h->launches++;
            if (chunk_events) {
                QueryChunk qc{p.q0, p.q1, pool_event(h, g, nev++, &rc)};
                if (rc != SW_OK) return rc;
                SW_CUDA(h, cudaEventRecord(qc.done, gc.st_compute));
                g.chunks.push_back(qc);
            }
        }
        for (int k = 1; k < kStreams; ++k) {
            if (!forked[k]) continue;
            SW_CUDA(h, cudaEventRecord(gc.ev_join[k - 1], gc.st_aux[k - 1]));
            SW_CUDA(h, cudaStreamWaitEvent(gc.st_compute, gc.ev_join[k - 1], 0));
        }
        // ---- band-pipelined launches, one per long query ----------------------------------------
        if (!wave_q.empty()) {
            const uint32_t cols_stride = ((g.max_len + 31u) & ~31u) + 32u;    // + slack for the batched boundary stores (kWaveSlack)
            uint32_t wmaxq = 0;
            for (int q : wave_q) wmaxq = std::max(wmaxq, h->q_len[q]);
            (void)wmaxq;
            {
                // tagged 16-byte boundary elements; zeroed once (tag 0 is never used), later launches
                // are told apart by the epoch in the tag
                const size_t bytes = (size_t)g.npairs * 2 * cols_stride * 16;
                if (gc.d_wave_bnd.cap < bytes || !gc.d_wave_bnd.p) {
                    SW_CUDA(h, cudaStreamSynchronize(gc.st_compute));
                    SW_CUDA(h, gc.d_wave_bnd.reserve(bytes));
                    SW_CUDA(h, cudaMemsetAsync(gc.d_wave_bnd.p, 0, gc.d_wave_bnd.cap, gc.st_compute));
                }
            }
            // state words: best [2 * npairs] | done [npairs]
            const size_t n_state = 3 * (size_t)g.npairs;
            SW_CUDA(h, gc.d_wave_state.reserve(n_state * sizeof(unsigned)));
            int wave_row = -1;
            for (int q : wave_q) {
                ++wave_row;
                SwWaveLaunch W;
                // pair-bands of 256 rows in this launch: many -> throughput-bound (512-row bands,
                // four pairs per block); fewer -> one pair per block, four columns per step; a
                // handful -> two columns per step; many pairs of long subjects -> 512-row bands with two
                // columns per step (measured crossovers, DESIGN.md section 5)
                const size_t warps256 = (size_t)g.npairs * ((h->q_len[q] + 255) / 256);
                const double mean_len = (double)g.sum_len / (2.0 * std::max<uint32_t>(g.npairs, 1));
                W.instance = warps256 < 1200 ? 2 : warps256 < 15000 ? 1 : mean_len >= 1000.0 ? 3 : 0;
                if (const char *e = std::getenv("SW_B200_WAVE_INSTANCE")) {       // A/B measurements
                    const int wi = std::atoi(e);
                    if (wi >= 0 && wi < sw_wave_instance_count() && wi < 16) W.instance = wi;
                }
                if (!gc.wave_bps[W.instance]) SW_CUDA(h, sw_wave_occupancy(W.instance, &gc.wave_bps[W.instance]));
                if (gc.wave_bps[W.instance] < 1) return SW_ECUDA;
                const int rows = sw_wave_rows_per_band(W.instance);
                W.db = db; W.q = dq; W.query = q; W.sc = sc;
                W.npass = (int)((h->q_len[q] + rows - 1) / rows);
                W.out = g.d_out.p; W.out_stride = n; W.out_mode = g.out_mode;
                if (topk || hits) { W.out = gc.d_wave_rows.p; W.out_mode = SW_OUT_I32; W.out_row = wave_row; }
                W.bnd = gc.d_wave_bnd.p; W.cols_stride = cols_stride;
                W.bnd_elems = (size_t)g.npairs * 2 * cols_stride; W.out_elems = (topk || hits) ? wave_q.size() * (size_t)n : (size_t)nq * n;
                gc.wave_epoch = (gc.wave_epoch % 0xFFFFEu) + 1u;            // 1 .. 2^20 - 2
                if (gc.wave_epoch == 1u && gc.counter_next > 0) {
                    // the epoch wrapped (or first use): stale tags must not match again
                    SW_CUDA(h, cudaMemsetAsync(gc.d_wave_bnd.p, 0, gc.d_wave_bnd.cap, gc.st_compute));
                }
                W.epoch = gc.wave_epoch;
                W.best = (int *)gc.d_wave_state.as<unsigned>();
                W.done = gc.d_wave_state.as<unsigned>() + 2 * (size_t)g.npairs;
                W.counter = next_counter(gc);
                const size_t ppb = (size_t)sw_wave_pairs_per_block(W.instance);
                const size_t items = (size_t)W.npass * ((g.npairs + ppb - 1) / ppb);
                W.grid = (int)std::min<size_t>(items, (size_t)gc.num_sms * gc.wave_bps[W.instance]);
                W.ovf_count = base.ovf_count; W.ovf_list = base.ovf_list; W.ovf_cap = base.ovf_cap;
                W.dev_err = gc.d_err.as<unsigned>();
                SW_CUDA(h, cudaMemsetAsync(gc.d_wave_state.p, 0, n_state * sizeof(unsigned), gc.st_compute));
                SW_CUDA(h, cudaMemsetAsync(W.counter, 0, sizeof(unsigned), gc.st_compute));
                SW_CUDA(h, sw_launch_wave(gc.st_compute, W));
                h->launches++;
                if (topk) {
                    // the row's k best scores become list 0 of this query (pairs flagged for the 32-bit
                    // scorer keep the sentinel here and reach the merge through the overflow list)
                    SW_CUDA(h, sw_launch_topk_row(gc.st_compute, (const int32_t *)gc.d_wave_rows.p + (size_t)wave_row * n, (uint32_t)n, q,
                                                  g.topk_k, gc.d_topk_keys.as<unsigned long long>()));
                    h->launches++;
                }
                if (hits) {
                    // the row's entries >= min_score join the list (flagged pairs come from the overflow list)
                    SW_CUDA(h, sw_launch_hits_row(gc.st_compute, (const int32_t *)gc.d_wave_rows.p + (size_t)wave_row * n, (uint32_t)n, q, hl));
                    h->launches++;
                }
                if (&gc == &h->gpus[0] && label_v < 0)
                    std::snprintf(h->last_kernel, sizeof h->last_kernel, "%s", sw_wave_kernel_name(W.instance));
            }
        }
        if (may_overflow) {
            s32.mode = 2; s32.list_count = g.d_ovf_count.as<unsigned>(); s32.list = g.d_ovf_list.as<uint2>();
            s32.list_cap = kOvfCap; s32.list_score = g.d_ovf_score.as<int32_t>();
            if (h->wave32) {
                // long entries (with the default scoring every entry is >= 6 400 x 6 400 nt) are scored
                // by bands on many warps; the launch is list-driven, so nothing is read back here
                SwWave32Launch W;
                W.db = db; W.q = dq; W.sc = sc;
                W.list_count = s32.list_count; W.list = s32.list; W.list_cap = kOvfCap; W.list_score = s32.list_score;
                W.out = s32.out; W.out_stride = n; W.out_elems = (size_t)nq * n; W.out_mode = g.out_mode;
                W.cols_stride = ((g.max_len + 31u) & ~31u) + 32u;
                const size_t per_slot = (size_t)2 * W.cols_stride * 16;
                W.nslots = (uint32_t)std::min<size_t>(64, std::max<size_t>(2, ((size_t)64 << 20) / per_slot));
                W.bnd_elems = (size_t)W.nslots * 2 * W.cols_stride;
                bool fresh = false;
                if (gc.d_wave32_bnd.cap < W.bnd_elems * 16 || !gc.d_wave32_bnd.p) {
                    SW_CUDA(h, cudaStreamSynchronize(gc.st_compute));
                    SW_CUDA(h, gc.d_wave32_bnd.reserve(W.bnd_elems * 16));
                    fresh = true;
                }
                const size_t state_bytes = (size_t)3 * SW_WAVE32_MAX_ENTRIES * sizeof(unsigned);
                SW_CUDA(h, gc.d_wave32_state.reserve(state_bytes));
                W.state = gc.d_wave32_state.as<unsigned>();
                W.maxb = (h->q_max_len + SW_WAVE32_ROWS - 1) / SW_WAVE32_ROWS;
                W.min_cells = h->wave32_min_cells;
                if (!gc.wave32_bps) SW_CUDA(h, sw_wave32_occupancy(&gc.wave32_bps));
                if (gc.wave32_bps < 1) return SW_ECUDA;
                // one warp per scheduler: a larger grid lets the first (few hundred) claiming blocks pile
                // up on a few SMs (measured: 16 blocks per SM = 2.3x slower for one 100 kb entry)
                W.grid = gc.num_sms * std::min(gc.wave32_bps, 4);
                W.dev_err = gc.d_err.as<unsigned>();
                // 4 096 entries per launch (12 tag bits); a launch that finds no entry costs one
                // atomic per block
                W.entry_limit = kWave32Parts * SW_WAVE32_MAX_ENTRIES;
                for (unsigned part = 0; part < kWave32Parts; ++part) {
                    gc.wave32_epoch = gc.wave32_epoch % 255u + 1u;
                    if (fresh || gc.wave32_epoch == 1u)      // stale tags must never match
                        SW_CUDA(h, cudaMemsetAsync(gc.d_wave32_bnd.p, 0, gc.d_wave32_bnd.cap, gc.st_compute));
                    fresh = false;
                    W.bnd = gc.d_wave32_bnd.p; W.epoch = gc.wave32_epoch;
                    W.entry_base = part * SW_WAVE32_MAX_ENTRIES;
                    SW_CUDA(h, cudaMemsetAsync(gc.d_wave32_state.p, 0, state_bytes, gc.st_compute));
                    W.counter = next_counter(gc);
                    SW_CUDA(h, cudaMemsetAsync(W.counter, 0, sizeof(unsigned), gc.st_compute));
                    SW_CUDA(h, sw_launch_wave32(gc.st_compute, W));
                    h->launches++;
                }
                s32.wave32_min_cells = W.min_cells; s32.wave32_limit = W.entry_limit;
            }
            SW_CUDA(h, sw_launch_score32(gc.st_compute, s32));
            h->launches++;
            if (hits) {
                SW_CUDA(h, sw_launch_hits_ovf(gc.st_compute, s32.list_count, s32.list, s32.list_score, kOvfCap, hl));
                h->launches++;
            }
        }
        if (topk) {
            SW_CUDA(h, sw_launch_topk_merge(gc.st_compute, gc.d_topk_keys.as<unsigned long long>(), max_grid, nq, g.topk_k,
                                            may_overflow ? g.d_ovf_count.as<unsigned>() : nullptr, g.d_ovf_list.as<uint2>(),
                                            g.d_ovf_score.as<int32_t>(), kOvfCap, g.d_topk_out.as<unsigned long long>()));
            h->launches++;
        }
    } else {
        s32.mode = 0; s32.q0 = 0; s32.q1 = nq;
        SW_CUDA(h, sw_launch_score32(gc.st_compute, s32));
        h->launches++;
    }
    if (g.chunks.empty()) {
        QueryChunk qc{0, nq, pool_event(h, g, nev++, &rc)};
        if (rc != SW_OK) return rc;
        SW_CUDA(h, cudaEventRecord(qc.done, gc.st_compute));
        g.chunks.push_back(qc);
    }
    SW_CUDA(h, cudaEventRecord(g.ev_stop, gc.st_compute));
    g.ev_stop_deferred = false;
    return SW_OK;
}

// waits for an event with a deadline; forever = no deadline
int wait_event(sw_handle *h, cudaEvent_t ev, const std::chrono::steady_clock::time_point &t_end, bool forever)
{
    const auto t_begin = std::chrono::steady_clock::now();
    for (;;) {
        cudaError_t e = cudaEventQuery(ev);
        if (e == cudaSuccess) return SW_OK;
        if (e != cudaErrorNotReady) { h->last_cuda.store((int)e); return SW_ECUDA; }
        const auto now = std::chrono::steady_clock::now();
        if (!forever && now >= t_end) return SW_ETIMEOUT;
        // short waits (small batches) are polled; long ones block / yield the core
        if (now - t_begin > std::chrono::microseconds(300)) {
            if (forever) { SW_CUDA(h, cudaEventSynchronize(ev)); return SW_OK; }
            std::this_thread::sleep_for(std::chrono::microseconds(50));
        }
    }
}

void finish_timing(sw_handle *h, int si, const std::chrono::steady_clock::time_point &t0,
                   const std::chrono::steady_clock::time_point &t1, double ms_max, double ms_min)
{
    const auto t2 = std::chrono::steady_clock::now();
    h->stats.fetch_wait_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    h->stats.fetch_drain_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
    h->stats.kernel_ms_max = ms_max;
    h->stats.kernel_ms_min = ms_min > 1e299 ? 0.0 : ms_min;
    h->last_ms = ms_max;
    h->last_cells = h->batch[si].cells;
    h->last_slot = si;
}

unsigned device_error_bits(sw_handle *h)
{
    unsigned bits = 0;
    for (auto &g : h->gpus) {
        if (cudaSetDevice(g.dev) != cudaSuccess) continue;
#ifdef SW_BOUNDS_CHECK
        cudaDeviceSynchronize();
        for (DevBuf *d : all_devbufs(g)) if (!d->canaries_ok()) bits |= 0x80000000u;
#endif
        if (g.d_err.p) {
            unsigned v = 0;
            if (cudaMemcpy(&v, g.d_err.p, sizeof v, cudaMemcpyDeviceToHost) == cudaSuccess) bits |= v;
        }
    }
    return bits;
}

// latency path: value of a result word the kernel has not written yet (scores are >= -1)
constexpr int32_t kSmallSentinel = INT32_MIN;

// what a fetch delivers
enum FetchKind { FETCH_I32, FETCH_I16, FETCH_TOPK };

int fetch_slot(sw_handle *h, int si, FetchKind kind, void *scores, uint64_t *index, size_t cap, int timeout_ms)
{
    Batch &bt = h->batch[si];
    const size_t nq = (size_t)bt.nq;
    const bool forever = timeout_ms < 0;
    const auto t_fetch0 = std::chrono::steady_clock::now();
    const auto t_end = t_fetch0 + std::chrono::milliseconds(forever ? 0 : timeout_ms);
    if (bt.hits_min > 0) return SW_ESTATE;                  // a hits batch has no matrix / top-k lists
    if (kind == FETCH_TOPK) {
        if (bt.topk_k <= 0) return SW_ESTATE;
        if (cap < nq * (size_t)bt.topk_k) return SW_ECAPACITY;
    } else {
        if (bt.topk_k > 0) return SW_ESTATE;
        if ((kind == FETCH_I16) != (bt.out_mode == SW_OUT_I16)) return SW_ESTATE;
        if (cap < nq * bt.ns) return SW_ECAPACITY;
    }

    // ---- small (latency) path: scores are already in mapped host memory ----------------------
    if (bt.small) {
        GpuCtx &g = h->gpus[0];
        Slot &b = g.slot[si];
        // Completion is read from mapped host memory.  Default: every result word replaces the
        // sentinel the host wrote before the launch (4-byte stores arrive whole), so the kernel needs
        // no system-scope fence and no flag -- its fence.sys alone was a quarter of the warp time of
        // the config-2 kernel -- and the host sees the last score one PCIe write after it was stored.
        // Otherwise: the flag the kernel's last block writes after its fence.
        volatile unsigned *flag = (volatile unsigned *)b.h_small_flag.p;
        const volatile int32_t *res = (const volatile int32_t *)b.h_small_out.p;
        const size_t nres = nq * bt.ns;
        size_t seen = 0;                                           // results [0, seen) have arrived
        unsigned spins = 0;
        auto complete = [&]() -> bool {
            if (b.small_by_flag) return *flag == b.small_seq;
            while (seen < nres && res[seen] != kSmallSentinel) ++seen;
            return seen == nres;
        };
        while (!complete()) {
            if ((++spins & 0x3FF) == 0) {
                if (!forever && std::chrono::steady_clock::now() >= t_end) return SW_ETIMEOUT;
                cudaError_t qe = cudaStreamQuery(g.st_compute);          // a failed launch would never finish the buffer
                if (qe != cudaSuccess && qe != cudaErrorNotReady) { h->last_cuda.store((int)qe); return SW_ECUDA; }
                if (qe == cudaSuccess && !complete()) { h->last_cuda.store((int)cudaErrorUnknown); return SW_ECUDA; }
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        const auto tr3 = std::chrono::steady_clock::now();
        std::memcpy(scores, b.h_small_out.p, nq * bt.ns * sizeof(int32_t));
        if (h->trace_small) {
            h->tr_wait += std::chrono::duration<double, std::micro>(tr3 - t_fetch0).count();
            h->tr_copy += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tr3).count();
        }
        float ms = 0.f;
        if (b.small_timed) {
            SW_CUDA(h, cudaEventSynchronize(b.ev_stop));
            SW_CUDA(h, cudaEventElapsedTime(&ms, b.ev_start, b.ev_stop));
        }
        finish_timing(h, si, t_fetch0, std::chrono::steady_clock::now(), ms, ms);
#ifdef SW_BOUNDS_CHECK
        if (device_error_bits(h)) return SW_EDEVICE;
#endif
        return SW_OK;
    }

    const size_t esz = kind == FETCH_I16 ? sizeof(int16_t) : sizeof(int32_t);
    bool any_ovf = false;
    for (auto &g : h->gpus) any_ovf |= g.slot[si].ovf_used && g.slot[si].scored && g.slot[si].s1 > g.slot[si].s0;
    bt.ovf_index.clear(); bt.ovf_score.clear();

    if (kind != FETCH_TOPK) {
        size_t maxchunks = 0;
        for (auto &g : h->gpus) maxchunks = std::max(maxchunks, g.slot[si].chunks.size());
        for (size_t c = 0; c < maxchunks; ++c) {
            for (auto &g : h->gpus) {
                Slot &b = g.slot[si];
                if (c >= b.chunks.size()) continue;
                const size_t n = b.s1 - b.s0;
                if (n == 0) continue;
                SW_CUDA(h, cudaSetDevice(g.dev));
                const QueryChunk &qc = b.chunks[c];
                int rc = wait_event(h, qc.done, t_end, forever);
                if (rc != SW_OK) {
                    // copies already enqueued must not outlive this call: the caller owns `scores`
                    for (auto &gg : h->gpus) { cudaSetDevice(gg.dev); cudaStreamSynchronize(gg.st_copy); }
                    return rc;
                }
                SW_CUDA(h, cudaMemcpy2DAsync((char *)scores + ((size_t)qc.q0 * bt.ns + b.s0) * esz, bt.ns * esz,
                                             (char *)b.d_out.p + (size_t)qc.q0 * n * esz, n * esz,
                                             n * esz, (size_t)(qc.q1 - qc.q0), cudaMemcpyDeviceToHost, g.st_copy));
            }
        }
    } else {
        for (auto &g : h->gpus) {
            Slot &b = g.slot[si];
            if (b.s1 == b.s0 || nq == 0 || b.chunks.empty()) continue;
            SW_CUDA(h, cudaSetDevice(g.dev));
            int rc = wait_event(h, b.chunks.back().done, t_end, forever);
            if (rc != SW_OK) return rc;
            const size_t bytes = nq * (size_t)bt.topk_k * sizeof(unsigned long long);
            SW_CUDA(h, b.h_topk.reserve(bytes));
            SW_CUDA(h, cudaMemcpyAsync(b.h_topk.p, b.d_topk_out.p, bytes, cudaMemcpyDeviceToHost, g.st_copy));
        }
    }
    const auto t_fetch1 = std::chrono::steady_clock::now();
    double ms_max = 0.0, ms_min = 1e300;
    for (auto &g : h->gpus) {
        Slot &b = g.slot[si];
        SW_CUDA(h, cudaSetDevice(g.dev));
        SW_CUDA(h, cudaStreamSynchronize(g.st_copy));
        if (b.scored && (b.s1 > b.s0) && nq) {
            SW_CUDA(h, cudaEventSynchronize(b.ev_stop));
            float ms = 0.f;
            SW_CUDA(h, cudaEventElapsedTime(&ms, b.ev_start, b.ev_stop));
            ms_max = std::max(ms_max, (double)ms);
            ms_min = std::min(ms_min, (double)ms);
        }
    }

    // ---- scores that left the 16-bit range (rare): list length check, side list for int16 -----
    if (any_ovf) {
        for (auto &g : h->gpus) {
            Slot &b = g.slot[si];
            if (!b.ovf_used || b.s1 == b.s0) continue;
            SW_CUDA(h, cudaSetDevice(g.dev));
            unsigned cnt = 0;
            SW_CUDA(h, cudaMemcpy(&cnt, b.d_ovf_count.p, sizeof cnt, cudaMemcpyDeviceToHost));
            if (cnt == 0) continue;
            const size_t n = b.s1 - b.s0;
            if (cnt > kOvfCap) {
                if (kind != FETCH_I32) return SW_ERANGE;
                // more flagged pairs than the list holds: rescan the matrix for sentinels (32-bit matrix only)
                SwScore32Launch s32;
                s32.db = dev_db(b); s32.q = dev_queries(h, g); s32.sc = scoring_of(h); s32.out = b.d_out.p; s32.out_stride = n;
                s32.out_mode = SW_OUT_I32; s32.scratch = g.d_scratch32.as<int32_t>();
                s32.max_cols = std::max<uint32_t>(1, std::min<uint32_t>(h->q_max_len, b.max_len));
                s32.threads_total = (int)(g.d_scratch32.cap / ((size_t)2 * s32.max_cols * sizeof(int32_t)) / 128 * 128);
                s32.mode = 1; s32.q0 = 0; s32.q1 = (int)nq;
                SW_CUDA(h, sw_launch_score32(g.st_compute, s32));
                h->launches++;
                SW_CUDA(h, cudaStreamSynchronize(g.st_compute));
                SW_CUDA(h, cudaMemcpy2D((char *)scores + b.s0 * esz, bt.ns * esz, b.d_out.p, n * esz, n * esz, nq, cudaMemcpyDeviceToHost));
                continue;
            }
            if (kind == FETCH_I16) {
                SW_CUDA(h, b.h_ovf.reserve((size_t)cnt * (sizeof(uint2) + sizeof(int32_t))));
                uint2 *hl = (uint2 *)b.h_ovf.p;
                int32_t *hs = (int32_t *)(hl + cnt);
                SW_CUDA(h, cudaMemcpy(hl, b.d_ovf_list.p, (size_t)cnt * sizeof(uint2), cudaMemcpyDeviceToHost));
                SW_CUDA(h, cudaMemcpy(hs, b.d_ovf_score.p, (size_t)cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
                for (unsigned i = 0; i < cnt; ++i) {
                    if (hs[i] <= 32767) continue;
                    bt.ovf_index.push_back((uint64_t)hl[i].x * bt.ns + b.s0 + hl[i].y);
                    bt.ovf_score.push_back(hs[i]);
                }
            }
        }
    }

    // ---- top-k: merge the per-GPU lists on the host -------------------------------------------
    if (kind == FETCH_TOPK) {
        const int K = bt.topk_k;
        int32_t *os = (int32_t *)scores;
        std::vector<std::pair<int64_t, uint64_t>> cand;      // (-score, index): ascending sort = best first
        for (size_t q = 0; q < nq; ++q) {
            cand.clear();
            for (auto &g : h->gpus) {
                Slot &b = g.slot[si];
                if (b.s1 == b.s0) continue;
                if (!b.chunks.empty() && b.h_topk.p && b.npairs) {
                    const unsigned long long *keys = (const unsigned long long *)b.h_topk.p + q * K;
                    for (int j = 0; j < K; ++j) {
                        if (keys[j] == 0) continue;
                        cand.emplace_back(-(int64_t)(keys[j] >> 32), b.s0 + (uint64_t)(uint32_t)~(uint32_t)(keys[j] & 0xFFFFFFFFu));
                    }
                }
                for (uint32_t e : b.empties) cand.emplace_back(0, b.s0 + e);     // zero-length subjects score 0
            }
            std::sort(cand.begin(), cand.end());
            for (int j = 0; j < K; ++j) {
                if ((size_t)j < cand.size()) { os[q * K + j] = (int32_t)(-cand[j].first); index[q * K + j] = cand[j].second; }
                else { os[q * K + j] = -1; index[q * K + j] = ~0ull; }
            }
        }
    }
    finish_timing(h, si, t_fetch0, t_fetch1, ms_max, ms_min);
    if (device_error_bits(h)) return SW_EDEVICE;
    return SW_OK;
}

// Hit list of a batch: per GPU wait for the kernels, read the count, radix-sort the list by (row, subject) and copy
// it to pinned staging -- on the copy stream, so that the next batch's kernels keep running -- then stitch the
// shards on the host.  Shards are contiguous input ranges in GPU order, so row-major order = for every row, the
// run of GPU 0, then of GPU 1, ...  The stitched list stays in the Batch until a fetch has room for it.
int fetch_hits_slot(sw_handle *h, int si, uint32_t *row, uint64_t *index, int32_t *score, size_t cap, size_t *count, int timeout_ms)
{
    Batch &bt = h->batch[si];
    if (bt.hits_min <= 0) return SW_ESTATE;
    const bool forever = timeout_ms < 0;
    const auto t_fetch0 = std::chrono::steady_clock::now();
    const auto t_end = t_fetch0 + std::chrono::milliseconds(forever ? 0 : timeout_ms);
    if (!bt.hits_staged) {
        const size_t ng = h->gpus.size();
        std::vector<unsigned long long> cnt(ng, 0);
        bool too_many = false;
        for (size_t gi = 0; gi < ng; ++gi) {
            GpuCtx &g = h->gpus[gi];
            Slot &b = g.slot[si];
            if (b.s1 == b.s0 || bt.nq == 0 || b.chunks.empty()) continue;
            SW_CUDA(h, cudaSetDevice(g.dev));
            int rc = wait_event(h, b.chunks.back().done, t_end, forever);
            if (rc != SW_OK) return rc;
            SW_CUDA(h, cudaMemcpy(&cnt[gi], b.d_hits_count.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            too_many |= cnt[gi] > bt.hits_max;
            if (b.ovf_used) {
                unsigned novf = 0;
                SW_CUDA(h, cudaMemcpy(&novf, b.d_ovf_count.p, sizeof novf, cudaMemcpyDeviceToHost));
                too_many |= novf > kOvfCap;
            }
        }
        const auto t_fetch1 = std::chrono::steady_clock::now();
        *count = 0;
        for (unsigned long long c : cnt) *count += (size_t)c;
        if (too_many) return SW_ERANGE;
        int row_bits = 0;
        while ((1ull << row_bits) < (uint64_t)bt.nq) ++row_bits;
        for (size_t gi = 0; gi < ng; ++gi) {
            GpuCtx &g = h->gpus[gi];
            Slot &b = g.slot[si];
            const size_t c = (size_t)cnt[gi];
            if (c == 0) continue;
            SW_CUDA(h, cudaSetDevice(g.dev));
            const int end_bit = std::max(1, b.hits_shift + row_bits);          // only the key bits in use
            // sized for max_hits (a count never exceeds it here): a buffer that grows would be freed, and cudaFree
            // waits for the whole device -- the next batch's kernels included
            if (g.d_hits_key2.cap < bt.hits_max * sizeof(unsigned long long) || g.d_hits_score2.cap < bt.hits_max * sizeof(int32_t)) {
                SW_CUDA(h, g.d_hits_key2.reserve(bt.hits_max * sizeof(unsigned long long)));
                SW_CUDA(h, g.d_hits_score2.reserve(bt.hits_max * sizeof(int32_t)));
            }
            size_t tmp = 0;
            SW_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp, b.d_hits_key.as<unsigned long long>(), g.d_hits_key2.as<unsigned long long>(),
                                                      b.d_hits_score.as<int32_t>(), g.d_hits_score2.as<int32_t>(), (int)bt.hits_max, 0, 64, g.st_copy));
            SW_CUDA(h, g.d_sort_tmp.reserve(tmp));
            tmp = g.d_sort_tmp.cap;
            SW_CUDA(h, cub::DeviceRadixSort::SortPairs(g.d_sort_tmp.p, tmp, b.d_hits_key.as<unsigned long long>(), g.d_hits_key2.as<unsigned long long>(),
                                                      b.d_hits_score.as<int32_t>(), g.d_hits_score2.as<int32_t>(), (int)c, 0, end_bit, g.st_copy));
            h->launches++;
            SW_CUDA(h, b.h_hits.reserve((size_t)c * (sizeof(unsigned long long) + sizeof(int32_t))));
            SW_CUDA(h, cudaMemcpyAsync(b.h_hits.p, g.d_hits_key2.p, (size_t)c * sizeof(unsigned long long), cudaMemcpyDeviceToHost, g.st_copy));
            SW_CUDA(h, cudaMemcpyAsync((unsigned long long *)b.h_hits.p + c, g.d_hits_score2.p, (size_t)c * sizeof(int32_t),
                                       cudaMemcpyDeviceToHost, g.st_copy));
        }
        double ms_max = 0.0, ms_min = 1e300;
        size_t total = 0;
        for (size_t gi = 0; gi < ng; ++gi) {
            GpuCtx &g = h->gpus[gi];
            Slot &b = g.slot[si];
            SW_CUDA(h, cudaSetDevice(g.dev));
            SW_CUDA(h, cudaStreamSynchronize(g.st_copy));
            total += cnt[gi];
            if (b.scored && b.s1 > b.s0 && bt.nq) {
                SW_CUDA(h, cudaEventSynchronize(b.ev_stop));
                float ms = 0.f;
                SW_CUDA(h, cudaEventElapsedTime(&ms, b.ev_start, b.ev_stop));
                ms_max = std::max(ms_max, (double)ms);
                ms_min = std::min(ms_min, (double)ms);
            }
        }
        bt.hits_row.resize(total); bt.hits_index.resize(total); bt.hits_score.resize(total);
        std::vector<size_t> cur(ng, 0);
        size_t o = 0;
        for (int r = 0; r < bt.nq && o < total; ++r) {
            for (size_t gi = 0; gi < ng; ++gi) {
                const Slot &b = h->gpus[gi].slot[si];
                if (cnt[gi] == 0) continue;
                const unsigned long long *keys = (const unsigned long long *)b.h_hits.p;
                const int32_t *sc = (const int32_t *)(keys + cnt[gi]);
                const unsigned long long mask = (1ull << b.hits_shift) - 1ull;
                for (size_t &k = cur[gi]; k < cnt[gi] && (keys[k] >> b.hits_shift) == (unsigned long long)r; ++k, ++o) {
                    bt.hits_row[o] = (uint32_t)r; bt.hits_index[o] = b.s0 + (keys[k] & mask); bt.hits_score[o] = sc[k];
                }
            }
        }
        bt.hits_staged = true;
        bt.ovf_index.clear(); bt.ovf_score.clear();          // sw_fetch_overflow: nothing for a hits batch
        finish_timing(h, si, t_fetch0, t_fetch1, ms_max, ms_min);
        if (device_error_bits(h)) { bt.hits_staged = false; return SW_EDEVICE; }
    }
    *count = bt.hits_row.size();
    if (cap < *count) return SW_ECAPACITY;
    if (*count) {
        std::memcpy(row, bt.hits_row.data(), *count * sizeof(uint32_t));
        std::memcpy(index, bt.hits_index.data(), *count * sizeof(uint64_t));
        std::memcpy(score, bt.hits_score.data(), *count * sizeof(int32_t));
    }
    bt.hits_staged = false;
    h->last_slot = si;
    return SW_OK;
}

int load_batch(sw_handle *h, int si, const uint8_t *packed, const uint32_t *len, const uint64_t *off,
               const uint64_t *ids, size_t ns)
{
    const auto t_load0 = std::chrono::steady_clock::now();
    Batch &bt = h->batch[si];
    bt.ns = ns; bt.loaded = false; bt.scored = false; bt.cells = 0; bt.small = false;
    bt.have_ids = ids != nullptr;
    if (ids) bt.ids.assign(ids, ids + ns); else bt.ids.clear();
    const size_t ng = h->gpus.size();
    std::vector<uint64_t> starts(ng + 1);
    sw_plan_shards(len, ns, (int)ng, starts.data());
    for (size_t gi = 0; gi < ng; ++gi) { h->gpus[gi].slot[si].s0 = starts[gi]; h->gpus[gi].slot[si].s1 = starts[gi + 1]; }
    // one host worker per GPU: the shards' length sort / pairing / uploads run concurrently
    int rc_load = SW_OK;
    if (ng == 1) {
        rc_load = load_shard(h, h->gpus[0], h->gpus[0].slot[si], packed, len, off);
    } else {
        std::vector<int> rcs(ng, SW_OK);
        std::vector<std::thread> workers;
        for (size_t gi = 0; gi < ng; ++gi)
            workers.emplace_back([&, gi]() { rcs[gi] = load_shard(h, h->gpus[gi], h->gpus[gi].slot[si], packed, len, off); });
        for (auto &w : workers) w.join();
        for (int rc : rcs) if (rc != SW_OK && rc_load == SW_OK) rc_load = rc;
    }
    // the caller's buffers must be reusable on return -- on success AND on failure (copies of
    // the GPUs that did not fail may still be reading them)
    for (auto &g : h->gpus) {
        cudaError_t e = cudaSetDevice(g.dev);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.st_copy);
        if (e != cudaSuccess && rc_load == SW_OK) { h->last_cuda.store((int)e); rc_load = SW_ECUDA; }
    }
    if (rc_load != SW_OK) return rc_load;
    h->stats.load_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_load0).count();
    bt.loaded = true;
    h->last_slot = si;
    return SW_OK;
}

int score_batch_slot(sw_handle *h, int si)
{
    const auto t_enq0 = std::chrono::steady_clock::now();
    Batch &bt = h->batch[si];
    uint64_t db_len = 0;
    for (auto &g : h->gpus) db_len += g.slot[si].sum_len;
    bt.cells = db_len * h->q_sum_len;
    bt.nq = (int)h->q_len.size();
    bt.out_mode = h->out_mode;
    bt.topk_k = h->topk_k;
    bt.hits_min = h->hits_min; bt.hits_max = h->hits_max; bt.hits_staged = false;
    h->last_cells = bt.cells;
    const size_t ng = h->gpus.size();
    std::vector<int> rcs(ng, SW_OK);
    if (ng == 1) {
        rcs[0] = score_gpu(h, h->gpus[0], h->gpus[0].slot[si]);
    } else {
        // one host worker per GPU: launch plans, allocations and (first call) autotune run concurrently
        std::vector<std::thread> workers;
        for (size_t gi = 0; gi < ng; ++gi)
            workers.emplace_back([&, gi]() { rcs[gi] = score_gpu(h, h->gpus[gi], h->gpus[gi].slot[si]); });
        for (auto &w : workers) w.join();
    }
    for (int rc : rcs) {
        if (rc != SW_OK) {
            // GPUs that already launched keep reading this slot: drain them before the slot can be
            // reused (the failed batch is not recorded in the fifo)
            for (auto &gg : h->gpus) { cudaSetDevice(gg.dev); cudaStreamSynchronize(gg.st_compute); gg.slot[si].scored = false; }
            return rc;
        }
    }
    bt.scored = true;
    h->stats.enqueue_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enq0).count();
    return SW_OK;
}

// ---- small (latency) path ------------------------------------------------------------------------
// One staging buffer [pair_subj | pair_len | off | raw], one H2D copy, one DIRECT strip launch with a
// static schedule, scores written into mapped pinned host memory.  *taken = false when the batch
// does not qualify (the regular path then handles it).
int small_variant(const sw_handle *h, uint32_t qmax, size_t npairs)
{
    if (h->force_variant >= 0) return sw_strip_variant(h->force_variant)->has_direct ? h->force_variant : -1;
    if (h->force_R || h->force_G || h->force32) return -1;
    const char *want;
    if (const char *e = std::getenv("SW_B200_SMALL_VARIANT")) {          // A/B measurements
        for (int i = 0; i < sw_strip_variant_count(); ++i)
            if (std::strcmp(sw_strip_variant(i)->name, e) == 0 && sw_strip_variant(i)->has_direct &&
                (uint32_t)(sw_strip_variant(i)->R * sw_strip_variant(i)->G) >= qmax) return i;
    }
    if (qmax <= 32) want = "strip_s16x2_R1x1_G32";
    else if (qmax <= 64) want = "strip_s16x2_R2x1_G32";
    else if (qmax <= 128) want = npairs <= 1500 ? "strip_s16x2_R4x1_G32" : npairs <= 3000 ? "strip_s16x2_R8x1_G16" : "strip_s16x2_R16x1_G8";
    else if (qmax <= 256) want = "strip_s16x2_R8x1_G32";
    else want = "strip_s16x2_R16x1_G32";
    for (int i = 0; i < sw_strip_variant_count(); ++i)
        if (std::strcmp(sw_strip_variant(i)->name, want) == 0) return i;
    return -1;
}

int small_submit(sw_handle *h, int si, const uint8_t *packed, const uint32_t *len, const uint64_t *off,
                 const uint64_t *ids, size_t ns, bool *taken)
{
    *taken = false;
    const int nq = (int)h->q_len.size();
    if (!h->small_path || ns == 0 || nq == 0 || ns > 8192 || (size_t)nq * ns > (1u << 20)) return SW_OK;
    // (hits mode: the completion protocol below reads a fixed number of result words, a list has no such end)
    if (h->topk_k > 0 || h->hits_min > 0 || h->out_mode != SW_OUT_I32 || h->params.score_width != 0) return SW_OK;
    uint64_t bmin = ~0ull, bmax = 0, sum = 0;
    uint32_t maxlen = 0;
    size_t n_empty = 0;
    for (size_t i = 0; i < ns; ++i) {
        if (len[i] == 0) { ++n_empty; continue; }
        bmin = std::min(bmin, off[i]);
        bmax = std::max<uint64_t>(bmax, off[i] + ((len[i] + 3ull) >> 2));
        maxlen = std::max(maxlen, len[i]);
        sum += len[i];
    }
    // the DIRECT instances stage a pair's code words in shared memory: subjects of up to 1024 bases
    if (maxlen == 0 || bmax - bmin > (1u << 20) || maxlen > 1024) return SW_OK;
    const SwScoring sc = scoring_of(h);
    if ((uint64_t)sc.match * std::min<uint64_t>(h->q_max_len, maxlen) + (uint64_t)sc.match >= 32000ull) return SW_OK;
    GpuCtx &gc = h->gpus[0];
    Slot &g = gc.slot[si];
    const size_t np_max = (ns + 1) / 2;
    const int vidx = small_variant(h, h->q_max_len, np_max);
    if (vidx < 0) return SW_OK;
    {
        // DIRECT instances with a pass of fewer than 512 rows have no multi-pass code
        const SwStripVariant *sv = sw_strip_variant(vidx);
        const uint32_t P = (uint32_t)(sv->R * sv->G);
        if (P < 512 && h->q_max_len > P) return SW_OK;
    }
    *taken = true;
    const auto tr0 = std::chrono::steady_clock::now();

    SW_CUDA(h, cudaSetDevice(gc.dev));
    Batch &bt = h->batch[si];
    bt.ns = ns; bt.loaded = true; bt.scored = true; bt.small = true;
    bt.have_ids = ids != nullptr;
    if (ids) bt.ids.assign(ids, ids + ns); else bt.ids.clear();
    bt.nq = nq; bt.out_mode = SW_OUT_I32; bt.topk_k = 0; bt.hits_min = 0; bt.hits_staged = false;
    bt.cells = sum * h->q_sum_len;
    h->last_cells = bt.cells;
    for (auto &gg : h->gpus) { gg.slot[si].s0 = 0; gg.slot[si].s1 = 0; gg.slot[si].chunks.clear(); gg.slot[si].ovf_used = false; }
    g.s0 = 0; g.s1 = ns; g.is_small = true; g.max_len = maxlen; g.sum_len = sum; g.out_mode = SW_OUT_I32; g.topk_k = 0;

    // ---- staging layout: [pair descriptors (32 bytes each) | raw bases]
    const size_t ntiles = (np_max + 31) / 32;
    const size_t o_desc = 0;
    const size_t o_raw = o_desc + ntiles * 32 * 32;
    const size_t raw_bytes = (size_t)(bmax - bmin);
    const size_t total = o_raw + raw_bytes + 16;
    SW_CUDA(h, g.h_small_in.reserve(total, true));
    SW_CUDA(h, g.d_small_in.reserve(total));
    SW_CUDA(h, g.h_small_out.reserve((size_t)nq * ns * sizeof(int32_t), true));
    if (!g.h_small_flag.p) {
        SW_CUDA(h, g.h_small_flag.reserve(64, true));
        std::memset(g.h_small_flag.p, 0, 64);
        SW_CUDA(h, g.d_small_done.reserve(sizeof(unsigned)));
        SW_CUDA(h, cudaMemset(g.d_small_done.p, 0, sizeof(unsigned)));
    }
    // the staging buffer is reused: the previous copy out of it finished before its batch was fetched
    char *st = (char *)g.h_small_in.p;
    sort_by_length(g, len, ns, maxlen);
    g.pair_tmp.resize(ntiles * 32 * 4);
    uint32_t *t_subj = g.pair_tmp.data(), *t_len = t_subj + ntiles * 32 * 2;
    const size_t np = make_pairs(g, len, ns, t_subj, t_len);
    g.npairs = (uint32_t)np;
    uint32_t *desc = (uint32_t *)(st + o_desc);
    for (size_t p = 0; p < np; ++p) {
        const uint32_t slo = t_subj[2 * p], shi = t_subj[2 * p + 1];
        uint32_t *d = desc + 8 * p;
        d[0] = t_len[2 * p]; d[1] = t_len[2 * p + 1]; d[2] = slo; d[3] = shi;
        d[4] = (uint32_t)(off[slo] - bmin);
        d[5] = shi != SW_NO_SUBJECT ? (uint32_t)(off[shi] - bmin) : 0u;
        d[6] = 0; d[7] = 0;
    }
    std::memcpy(st + o_raw, packed + bmin, raw_bytes);
    std::memset(st + o_raw + raw_bytes, 0, 16);
    // scores of empty subjects (never touched by the kernel)
    int32_t *hout = (int32_t *)g.h_small_out.p;
    g.small_by_flag = !h->small_sentinel;
    for (uint32_t l : h->q_len) if (l == 0) g.small_by_flag = true;       // be safe: rows the kernel may not write
    if (!g.small_by_flag) std::fill(hout, hout + (size_t)nq * ns, kSmallSentinel);
    if (n_empty)        // (np * 2 == ns says nothing: one empty subject and an odd number of others pair up to ns / 2 as well)
        for (size_t k = 0; k < ns; ++k) if (len[k] == 0) for (int q = 0; q < nq; ++q) hout[(size_t)q * ns + k] = 0;

    // ---- one copy, one kernel
    const auto tr1 = std::chrono::steady_clock::now();
    cudaStream_t cs = gc.st_compute;
    const bool zero_copy = h->small_zero_copy && total <= (64u << 10);
    if (!zero_copy) SW_CUDA(h, cudaMemcpyAsync(g.d_small_in.p, st, total, cudaMemcpyHostToDevice, cs));
    const SwStripVariant *v = sw_strip_variant(vidx);
    SwStripLaunch L;
    char *d = zero_copy ? (char *)g.h_small_in.dptr : (char *)g.d_small_in.p;
    L.vidx = vidx; L.direct = true;
    L.db.raw = (const uint8_t *)(d + o_raw); L.db.off = nullptr; L.db.len = nullptr;
    L.db.ns = (uint32_t)ns; L.db.pair_subj = nullptr; L.db.pair_len = nullptr; L.db.pair_desc = (const uint4 *)(d + o_desc);
    L.db.tile_woff = nullptr; L.db.tp = nullptr; L.db.tp_words = 0; L.db.npairs = (uint32_t)np; L.db.max_len = maxlen;
    L.q = dev_queries(h, gc); L.q0 = 0; L.nql = nq; L.qidx = nullptr; L.sc = sc;
    L.out = g.h_small_out.dptr; L.out_stride = ns; L.out_elems = (size_t)nq * ns; L.out_mode = SW_OUT_I32;
    L.bnd_cols = maxlen; L.counter = nullptr;
    L.dev_err = gc.d_err.as<unsigned>();
    const int P = v->R * v->G;
    const int need_passes = (int)((h->q_max_len + P - 1) / P);
    const size_t pass_bytes = sw_strip_smem_bytes(vidx, 1);
    L.chunk_passes = std::max(1, std::min(need_passes, std::max<int>(1, (int)((48 * 1024) / pass_bytes))));
    const int ppb = v->block_threads / v->G;
    const size_t items = ((np + ppb - 1) / ppb) * (size_t)nq;
    L.grid = (int)std::min<size_t>(std::max<size_t>(items, 1), (size_t)gc.num_sms * 4);
    if (need_passes > 1) {
        const size_t per_block = (size_t)maxlen * ppb * sizeof(uint2);
        SW_CUDA(h, gc.d_bnd.reserve((size_t)L.grid * per_block));
        L.bnd_elems = (size_t)L.grid * per_block / sizeof(uint2);
    }
    L.bnd = gc.d_bnd.as<uint2>();
    // completion: the kernel's last block writes small_seq into a mapped host word the host polls
    g.small_seq++;
    if (g.small_seq == 0) g.small_seq = 1;
    if (g.small_by_flag) { L.done_count = g.d_small_done.as<unsigned>(); L.done_flag = (unsigned *)g.h_small_flag.dptr; L.done_seq = g.small_seq; }
    g.small_timed = h->small_timing;
    if (g.small_timed) SW_CUDA(h, cudaEventRecord(g.ev_start, cs));
    SW_CUDA(h, sw_launch_strip(cs, L));
    h->launches++;
    // load_shard orders a later reuse of the slot after ev_stop; without the timing events it is
    // recorded there, when needed (one driver call less on the latency path)
    g.ev_stop_deferred = !g.small_timed;
    if (g.small_timed) SW_CUDA(h, cudaEventRecord(g.ev_stop, cs));
    g.scored = true;
    std::snprintf(h->last_kernel, sizeof h->last_kernel, "%s+direct", v->name);
    h->last_slot = si;
    if (h->trace_small) {
        const auto tr2 = std::chrono::steady_clock::now();
        h->tr_prep += std::chrono::duration<double, std::micro>(tr1 - tr0).count();
        h->tr_launch += std::chrono::duration<double, std::micro>(tr2 - tr1).count();
        h->tr_n++;
    }
    return SW_OK;
}

int pop_fifo(sw_handle *h, int rc)
{
    if (rc == SW_ETIMEOUT || rc == SW_ECAPACITY || rc == SW_ESTATE) return rc;   // batch stays in flight; fetch again
    h->fifo[0] = h->fifo[1];
    h->n_inflight--;
    return rc;
}

int fetch_db_common(sw_handle_t *h, FetchKind kind, void *scores, uint64_t *index, size_t cap)
{
    if (!h || !scores) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    if (!h->batch[0].loaded || !h->batch[0].scored) return SW_ESTATE;
    return fetch_slot(h, 0, kind, scores, index, cap, -1);
}

// hits mode with the forced 32-bit scorer: refused before anything is enqueued (that scorer has no hit list)
bool hits_need_strip(const sw_handle *h) { return h->hits_min > 0 && h->force32; }

int fetch_common(sw_handle_t *h, FetchKind kind, void *scores, uint64_t *index, size_t cap, int timeout_ms)
{
    if (!h || (!scores && cap)) return SW_EINVAL;
    if (h->n_inflight == 0) return SW_ESTATE;
    return pop_fifo(h, fetch_slot(h, h->fifo[0], kind, scores, index, cap, timeout_ms));
}

}  // namespace

// ================================================================================================
extern "C" {

int sw_params_in_exact_domain(const sw_params_t *p)
{
    sw_params_t d;
    if (!p) { sw_default_params(&d); p = &d; }
    if (validate_params(p) != SW_OK) return SW_EINVAL;
    return ((int)p->match + (int)p->gap_open <= 0) ? 1 : 0;
}

void sw_default_params(sw_params_t *p)
{
    if (!p) return;
    p->match = 5; p->mismatch = -4; p->gap_open = -12; p->gap_extend = -4; p->score_width = 0;
}

const char *sw_version(void)
{
#ifdef SW_BOUNDS_CHECK
    return "sw_b200 0.2 (sm_100a, bounds-check build)";
#else
    return "sw_b200 0.2 (sm_100a)";
#endif
}

int sw_is_check_build(void)
{
#ifdef SW_BOUNDS_CHECK
    return 1;
#else
    return 0;
#endif
}

int sw_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *sw_strerror(int code)
{
    switch (code) {
        case SW_OK: return "ok";
        case SW_EINVAL: return "invalid argument or unsupported parameter set";
        case SW_ENOMEM: return "out of memory";
        case SW_ECUDA: return "CUDA error (see sw_last_cuda_error)";
        case SW_ENODEV: return "no usable CUDA device";
        case SW_ESTATE: return "call out of order";
        case SW_ETIMEOUT: return "timed out";
        case SW_ECAPACITY: return "output buffer too small";
        case SW_EIO: return "I/O error";
        case SW_EAGAIN: return "busy: both batch buffers are in flight (fetch one first)";
        case SW_ERANGE: return "too many scores beyond the 16-bit range for this output mode (use int32 output)";
        case SW_EDEVICE: return "device-side check failed (see sw_device_error_bits)";
        default: return "unknown error";
    }
}

int sw_init(sw_handle_t **out, const sw_params_t *p, const int *gpu_ids, int n_gpus)
{
    if (!out) return SW_EINVAL;
    *out = nullptr;
    sw_params_t prm;
    if (p) prm = *p; else sw_default_params(&prm);
    int rc = validate_params(&prm);
    if (rc != SW_OK) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return SW_ENODEV; }
    std::vector<int> ids;
    if (!gpu_ids || n_gpus <= 0) ids.push_back(0);
    else ids.assign(gpu_ids, gpu_ids + n_gpus);
    for (int id : ids) if (id < 0 || id >= ndev) return SW_ENODEV;

    sw_handle *h = new (std::nothrow) sw_handle();
    if (!h) return SW_ENOMEM;
    h->params = prm;
    if (const char *e = std::getenv("SW_B200_AUTOTUNE")) h->autotune = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_JIT")) h->jit = std::atoi(e);
    if (const char *e = std::getenv("SW_B200_SMALL_PATH")) h->small_path = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_WAVE")) h->wave = std::atoi(e);
    if (const char *e = std::getenv("SW_B200_WAVE32")) h->wave32 = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_TRACE_SMALL")) h->trace_small = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_SMALL_SENTINEL")) h->small_sentinel = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_SMALL_ZEROCOPY")) h->small_zero_copy = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_PLAN_SEGS")) h->plan_segs = std::atoi(e);
    if (const char *e = std::getenv("SW_B200_PLAN_QGROUPS")) h->plan_qgroups = (e[0] != '0');
    if (const char *e = std::getenv("SW_B200_STREAMS")) h->plan_streams = std::max(1, std::min(kStreams, std::atoi(e)));
    if (const char *e = std::getenv("SW_B200_TAU")) h->plan_tau = std::atof(e);
    if (const char *e = std::getenv("SW_B200_STICKY")) h->sticky = std::atoi(e);
    if (const char *e = std::getenv("SW_B200_PASS_SPLIT")) h->pass_split = std::atoi(e);
    if (const char *e = std::getenv("SW_B200_SUPERBLOCK_MB")) h->superblock_mb = std::max(0.01, std::atof(e));
    h->gpus.resize(ids.size());
    for (size_t i = 0; i < ids.size(); ++i) {
        GpuCtx &g = h->gpus[i];
        g.dev = ids[i];
        cudaError_t e = cudaSetDevice(g.dev);
        cudaDeviceProp prop;
        if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, g.dev);
        if (e == cudaSuccess) {
            g.num_sms = prop.multiProcessorCount;
            if (prop.major < 10) e = cudaErrorInvalidDevice;      // sm_100a cubin only
        }
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g.st_compute, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g.st_copy, cudaStreamNonBlocking);
        for (int k = 0; k < kStreams - 1; ++k) {
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g.st_aux[k], cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g.ev_join[k], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g.ev_fork, cudaEventDisableTiming);
        for (Slot &b : g.slot) {
            if (e == cudaSuccess) e = cudaEventCreate(&b.ev_start);
            if (e == cudaSuccess) e = cudaEventCreate(&b.ev_stop);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b.ev_upload, cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = g.d_err.reserve(sizeof(unsigned));
        if (e == cudaSuccess) e = cudaMemset(g.d_err.p, 0, sizeof(unsigned));
        if (e != cudaSuccess) {
            for (auto &gg : h->gpus) free_gpu(gg);
            delete h;
            cudaGetLastError();
            return e == cudaErrorInvalidDevice ? SW_ENODEV : SW_ECUDA;
        }
    }
    *out = h;
    return SW_OK;
}

void sw_destroy(sw_handle_t *h)
{
    if (!h) return;
    if (h->trace_small && h->tr_n)
        std::fprintf(stderr, "[sw_b200] latency path, %ld batches: host prep %.2f us, driver calls %.2f us, wait in fetch %.2f us, copy out %.2f us\n",
                     h->tr_n, h->tr_prep / h->tr_n, h->tr_launch / h->tr_n, h->tr_wait / h->tr_n, h->tr_copy / h->tr_n);
    for (auto &g : h->gpus) {
        cudaSetDevice(g.dev);
        cudaDeviceSynchronize();
        free_gpu(g);
    }
    delete h;
}

int sw_set_strands(sw_handle_t *h, int both)
{
    if (!h) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    h->both_strands = both != 0;
    return SW_OK;
}

int sw_set_output(sw_handle_t *h, int mode)
{
    if (!h || (mode != SW_OUTPUT_I32 && mode != SW_OUTPUT_I16)) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    h->out_mode = mode == SW_OUTPUT_I16 ? SW_OUT_I16 : SW_OUT_I32;
    for (Batch &bt : h->batch) bt.scored = false;
    return SW_OK;
}

int sw_set_topk(sw_handle_t *h, int k)
{
    if (!h || k < 0 || k > SW_MAX_TOPK || (k > 0 && h->hits_min > 0)) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    h->topk_k = k;
    for (Batch &bt : h->batch) bt.scored = false;
    return SW_OK;
}

int sw_set_hits(sw_handle_t *h, int32_t min_score, size_t max_hits)
{
    // (the device counter is 32-bit and counts past the list's end; the radix sort takes an int count)
    if (!h || min_score < 0 || (min_score > 0 && (max_hits == 0 || max_hits > 0x7FFFFFFFu))) return SW_EINVAL;
    if (min_score > 0 && h->topk_k > 0) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    h->hits_min = min_score;
    h->hits_max = min_score > 0 ? max_hits : 0;
    for (Batch &bt : h->batch) bt.scored = false;
    return SW_OK;
}

int sw_fetch_hits(sw_handle_t *h, uint32_t *row, uint64_t *index, int32_t *score, size_t cap, size_t *count, int timeout_ms)
{
    if (!h || !count || (cap && (!row || !index || !score))) return SW_EINVAL;
    *count = 0;
    if (h->n_inflight == 0) return SW_ESTATE;
    return pop_fifo(h, fetch_hits_slot(h, h->fifo[0], row, index, score, cap, count, timeout_ms));
}

int sw_fetch_db_hits(sw_handle_t *h, uint32_t *row, uint64_t *index, int32_t *score, size_t cap, size_t *count)
{
    if (!h || !count || (cap && (!row || !index || !score))) return SW_EINVAL;
    *count = 0;
    if (h->n_inflight) return SW_EAGAIN;
    if (!h->batch[0].loaded || !h->batch[0].scored) return SW_ESTATE;
    return fetch_hits_slot(h, 0, row, index, score, cap, count, -1);
}

int sw_set_queries(sw_handle_t *h, const uint8_t *packed, const uint32_t *len, const uint64_t *off, int nq)
{
    if (!h || nq < 0 || (nq > 0 && (!packed || !len || !off))) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    // kernels of a previous sw_score_db may still read the query buffers
    for (auto &g : h->gpus) { cudaSetDevice(g.dev); cudaStreamSynchronize(g.st_compute); }
    h->q_packed.clear(); h->q_off.clear(); h->q_len.clear();
    h->q_max_len = 0; h->q_sum_len = 0;
    h->nq_user = nq;
    const int strands = h->both_strands ? 2 : 1;
    for (int st = 0; st < strands; ++st) {
        for (int i = 0; i < nq; ++i) {
            const size_t bytes = ((size_t)len[i] + 3) / 4;
            if (h->q_packed.size() + bytes > 0xFFFFFFF0ull) return SW_EINVAL;
            h->q_off.push_back((uint32_t)h->q_packed.size());
            h->q_len.push_back(len[i]);
            const uint8_t *src = packed + off[i];
            if (st == 0) {
                h->q_packed.insert(h->q_packed.end(), src, src + bytes);
                if (len[i] & 3) h->q_packed.back() &= (uint8_t)((1u << (2 * (len[i] & 3))) - 1u);
            } else {
                // reverse complement: A(10) <-> T(00), C(01) <-> G(11)  =  code ^ 2, order reversed
                const size_t base = h->q_packed.size();
                h->q_packed.resize(base + bytes, 0);
                for (uint32_t k = 0; k < len[i]; ++k) {
                    const uint32_t j = len[i] - 1 - k;
                    const uint8_t c = (uint8_t)(((src[j >> 2] >> ((j & 3) * 2)) & 3) ^ 2);
                    h->q_packed[base + (k >> 2)] |= (uint8_t)(c << ((k & 3) * 2));
                }
            }
            h->q_max_len = std::max(h->q_max_len, len[i]);
            h->q_sum_len += len[i];
        }
    }
    h->q_packed.resize(h->q_packed.size() + 16, 0);
    for (auto &g : h->gpus) {
        int rc = upload_queries(h, g);
        if (rc != SW_OK) return rc;
    }
    for (Batch &bt : h->batch) bt.scored = false;
    return SW_OK;
}

int sw_plan_shards(const uint32_t *len, size_t ns, int n_shards, uint64_t *starts)
{
    if (n_shards <= 0 || !starts || (ns > 0 && !len)) return SW_EINVAL;
    uint64_t total = 0;
    for (size_t s = 0; s < ns; ++s) total += len[s];
    size_t s = 0;
    uint64_t acc = 0;
    for (int gi = 0; gi < n_shards; ++gi) {
        starts[gi] = s;
        const uint64_t target = (total * (uint64_t)(gi + 1)) / (uint64_t)n_shards;
        if (gi + 1 == n_shards) s = ns;
        else while (s < ns && acc + len[s] / 2 < target) { acc += len[s]; ++s; }
    }
    starts[n_shards] = ns;
    return SW_OK;
}

int sw_load_db(sw_handle_t *h, const uint8_t *packed, const uint32_t *len, const uint64_t *off,
               const uint64_t *ids, size_t ns)
{
    if (!h || (ns > 0 && (!packed || !len || !off))) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    return load_batch(h, 0, packed, len, off, ids, ns);
}

int sw_score_db(sw_handle_t *h)
{
    if (!h) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    if (!h->batch[0].loaded || h->batch[0].small) return SW_ESTATE;
    if (hits_need_strip(h)) return SW_EINVAL;
    return score_batch_slot(h, 0);
}

int sw_wait(sw_handle_t *h, int timeout_ms)
{
    if (!h) return SW_EINVAL;
    const bool forever = timeout_ms < 0;
    const auto t_end = std::chrono::steady_clock::now() + std::chrono::milliseconds(forever ? 0 : timeout_ms);
    double ms_max = 0.0;
    for (auto &g : h->gpus) {
        Slot &b = g.slot[0];
        if (!b.scored || b.chunks.empty()) continue;
        SW_CUDA(h, cudaSetDevice(g.dev));
        int rc = wait_event(h, b.chunks.back().done, t_end, forever);
        if (rc != SW_OK) return rc;
        SW_CUDA(h, cudaEventSynchronize(b.ev_stop));
        float ms = 0.f;
        SW_CUDA(h, cudaEventElapsedTime(&ms, b.ev_start, b.ev_stop));
        ms_max = std::max(ms_max, (double)ms);
    }
    h->last_ms = ms_max;
    h->last_cells = h->batch[0].cells;
    return SW_OK;
}

int sw_fetch_db(sw_handle_t *h, int32_t *scores, size_t cap) { return fetch_db_common(h, FETCH_I32, scores, nullptr, cap); }
int sw_fetch_db_i16(sw_handle_t *h, int16_t *scores, size_t cap) { return fetch_db_common(h, FETCH_I16, scores, nullptr, cap); }
int sw_fetch_db_topk(sw_handle_t *h, int32_t *scores, uint64_t *index, size_t cap)
{
    if (!index) return SW_EINVAL;
    return fetch_db_common(h, FETCH_TOPK, scores, index, cap);
}

int sw_score_batch(sw_handle_t *h, const uint8_t *packed, const uint32_t *len, const uint64_t *off,
                   const uint64_t *ids, size_t ns)
{
    if (!h || (ns > 0 && (!packed || !len || !off))) return SW_EINVAL;
    if (h->n_inflight >= 2) return SW_EAGAIN;          // both buffers busy: the bank's `full`
    if (hits_need_strip(h)) return SW_EINVAL;
    // take the slot that is not in flight; this replaces whatever sw_load_db left there
    const int si = (h->n_inflight == 1) ? (1 - h->fifo[0]) : 0;
    bool taken = false;
    int rc = small_submit(h, si, packed, len, off, ids, ns, &taken);
    if (rc != SW_OK) return rc;
    if (!taken) {
        rc = load_batch(h, si, packed, len, off, ids, ns);
        if (rc != SW_OK) return rc;
        rc = score_batch_slot(h, si);
        if (rc != SW_OK) return rc;
    }
    h->fifo[h->n_inflight++] = si;
    return SW_OK;
}

int sw_fetch(sw_handle_t *h, int32_t *scores, size_t cap, int timeout_ms)
{
    return fetch_common(h, FETCH_I32, scores, nullptr, cap, timeout_ms);
}
int sw_fetch_i16(sw_handle_t *h, int16_t *scores, size_t cap, int timeout_ms)
{
    return fetch_common(h, FETCH_I16, scores, nullptr, cap, timeout_ms);
}
int sw_fetch_topk(sw_handle_t *h, int32_t *scores, uint64_t *index, size_t cap, int timeout_ms)
{
    if (!index && cap) return SW_EINVAL;
    return fetch_common(h, FETCH_TOPK, scores, index, cap, timeout_ms);
}

int sw_fetch_overflow(sw_handle_t *h, uint64_t *flat_index, int32_t *score, size_t cap, size_t *count)
{
    if (!h || !count) return SW_EINVAL;
    const Batch &bt = h->batch[h->last_slot];
    *count = bt.ovf_index.size();
    const size_t n = std::min(cap, bt.ovf_index.size());
    if (n && (!flat_index || !score)) return SW_EINVAL;
    for (size_t i = 0; i < n; ++i) { flat_index[i] = bt.ovf_index[i]; score[i] = bt.ovf_score[i]; }
    return SW_OK;
}

int sw_batches_in_flight(const sw_handle_t *h) { return h ? h->n_inflight : 0; }

int sw_fetch_ids(sw_handle_t *h, uint64_t *ids, size_t cap)
{
    if (!h || !ids) return SW_EINVAL;
    const Batch &bt = h->batch[h->last_slot];
    if (cap < bt.ns) return SW_ECAPACITY;
    for (size_t s = 0; s < bt.ns; ++s) ids[s] = bt.have_ids ? bt.ids[s] : (uint64_t)s;
    return SW_OK;
}

int sw_fetch_best(sw_handle_t *h, int32_t *best_score, uint64_t *best_index, int nq_cap)
{
    if (!h || !best_score || !best_index) return SW_EINVAL;
    if (h->n_inflight) return SW_EAGAIN;
    const Batch &bt = h->batch[0];
    const int nq = bt.nq;
    if (!bt.loaded || !bt.scored || bt.small || bt.topk_k > 0 || bt.hits_min > 0 || bt.out_mode != SW_OUT_I32) return SW_ESTATE;
    if (nq_cap < nq) return SW_ECAPACITY;
    for (int q = 0; q < nq; ++q) { best_score[q] = 0; best_index[q] = 0; }
    std::vector<int32_t> hs(nq);
    std::vector<uint32_t> hi(nq);
    bool first = true;
    for (auto &g : h->gpus) {
        Slot &b = g.slot[0];
        const size_t n = b.s1 - b.s0;
        if (n == 0 || nq == 0) continue;
        SW_CUDA(h, cudaSetDevice(g.dev));
        SW_CUDA(h, g.d_best_score.reserve(nq * sizeof(int32_t)));
        SW_CUDA(h, g.d_best_index.reserve(nq * sizeof(uint32_t)));
        SW_CUDA(h, sw_launch_best(g.st_compute, b.d_out.as<int32_t>(), n, (uint32_t)n, nq,
                                  g.d_best_score.as<int32_t>(), g.d_best_index.as<uint32_t>()));
        h->launches++;
        SW_CUDA(h, cudaMemcpyAsync(hs.data(), g.d_best_score.p, nq * sizeof(int32_t), cudaMemcpyDeviceToHost, g.st_compute));
        SW_CUDA(h, cudaMemcpyAsync(hi.data(), g.d_best_index.p, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, g.st_compute));
        SW_CUDA(h, cudaStreamSynchronize(g.st_compute));
        for (int q = 0; q < nq; ++q) {
            if (first || hs[q] > best_score[q]) { best_score[q] = hs[q]; best_index[q] = b.s0 + hi[q]; }
        }
        first = false;
    }
    return SW_OK;
}

int sw_query_rows(const sw_handle_t *h) { return h ? (int)h->q_len.size() : 0; }

int sw_get_stats(const sw_handle_t *h, sw_stats_t *out)
{
    if (!h || !out) return SW_EINVAL;
    *out = h->stats;
    return SW_OK;
}

unsigned sw_device_error_bits(sw_handle_t *h) { return h ? device_error_bits(h) : 0u; }

int sw_last_cuda_error(const sw_handle_t *h) { return h ? h->last_cuda.load() : 0; }
const char *sw_last_cuda_error_string(const sw_handle_t *h)
{
    return cudaGetErrorString((cudaError_t)(h ? h->last_cuda.load() : 0));
}
double sw_last_kernel_ms(const sw_handle_t *h) { return h ? h->last_ms : 0.0; }
uint64_t sw_kernel_launches(const sw_handle_t *h) { return h ? h->launches.load() : 0; }
uint64_t sw_last_cells(const sw_handle_t *h) { return h ? h->last_cells : 0; }
const char *sw_last_kernel_name(const sw_handle_t *h) { return h ? h->last_kernel : "none"; }

int sw_set_kernel_choice(sw_handle_t *h, int rows_per_lane, int lanes_per_pair, int force32)
{
    if (!h) return SW_EINVAL;
    h->force_R = rows_per_lane; h->force_G = lanes_per_pair; h->force32 = force32;
    return SW_OK;
}

int sw_kernel_variant_count(void) { return sw_strip_variant_count(); }

const char *sw_kernel_variant_name(int idx)
{
    const SwStripVariant *v = sw_strip_variant(idx);
    return v ? v->name : nullptr;
}

int sw_set_kernel_name(sw_handle_t *h, const char *name)
{
    if (!h) return SW_EINVAL;
    if (!name || !*name) { h->force_variant = -1; return SW_OK; }
    for (int i = 0; i < sw_strip_variant_count(); ++i)
        if (std::strcmp(sw_strip_variant(i)->name, name) == 0) { h->force_variant = i; return SW_OK; }
    return SW_EINVAL;
}

int sw_set_fixed_penalty_kernels(int enable)
{
    sw_strip_disable_fixed(enable == 0);
    return SW_OK;
}

int sw_set_autotune(sw_handle_t *h, int enable)
{
    if (!h) return SW_EINVAL;
    h->autotune = enable != 0;
    for (auto &g : h->gpus) g.tune_choice = -1;
    return SW_OK;
}

int sw_set_jit(sw_handle_t *h, int mode)
{
    if (!h || mode < 0 || mode > 2) return SW_EINVAL;
    h->jit = mode;
    return SW_OK;
}

int sw_set_launch_plan(sw_handle_t *h, int length_groups, int query_groups)
{
    if (!h || length_groups < 0 || length_groups > 2) return SW_EINVAL;
    h->plan_segs = length_groups;
    h->plan_qgroups = query_groups != 0;
    return SW_OK;
}

int sw_set_pass_split(sw_handle_t *h, int mode)
{
    if (!h || mode < -1 || mode == 1) return SW_EINVAL;
    h->pass_split = mode;
    return SW_OK;
}

int sw_plan_pass_parts(int npass, int chunk_passes, unsigned long long chains, int grid, int mode, int *nparts, int *part_passes)
{
    return plan_pass_parts(npass, chunk_passes, chains, grid, mode, nparts, part_passes);
}

int sw_last_pass_parts(const sw_handle_t *h)
{
    return h ? std::max(1, h->last_parts) : SW_EINVAL;
}

int sw_set_wave_mode(sw_handle_t *h, int mode)
{
    if (!h || mode < 0 || mode > 2) return SW_EINVAL;
    h->wave = mode;
    return SW_OK;
}

int sw_set_overflow_wave(sw_handle_t *h, int enable, unsigned long long min_cells)
{
    if (!h) return SW_EINVAL;
    h->wave32 = enable != 0;
    h->wave32_min_cells = min_cells ? min_cells : 1ull;
    return SW_OK;
}

int sw_jit_is_available(void) { return sw_jit_available(); }

int sw_jit_compile_check(const char *variant_name, int gap_open, int gap_extend, char *msg, size_t msg_cap)
{
    if (!variant_name) return SW_EINVAL;
    for (int i = 0; i < sw_strip_variant_count(); ++i) {
        if (std::strcmp(sw_strip_variant(i)->name, variant_name) != 0) continue;
        return sw_jit_strip_kernel(sw_strip_variant(i), gap_open + gap_extend, gap_extend, msg, msg_cap) ? 1 : 0;
    }
    return SW_EINVAL;
}

int sw_set_small_batch_path(sw_handle_t *h, int enable)
{
    if (!h) return SW_EINVAL;
    h->small_path = enable != 0;
    return SW_OK;
}

int sw_set_small_batch_timing(sw_handle_t *h, int enable)
{
    if (!h) return SW_EINVAL;
    h->small_timing = enable != 0;
    return SW_OK;
}

int sw_set_arith(sw_handle_t *h, int arith)
{
    if (!h || arith < -1 || arith > 0) return SW_EINVAL;     /* only packed s16 is compiled in */
    h->force_arith = arith;
    return SW_OK;
}

}  // extern "C"
