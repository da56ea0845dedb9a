/*
 * sw_kernels.h -- host-side launch interface of the CUDA kernels (internal to
 * libsw_b200.so; the public boundary is include/sw_b200.h).
 */
#ifndef SW_KERNELS_H_
#define SW_KERNELS_H_

#include <cuda_runtime.h>
#include <stdint.h>

#define SW_NO_SUBJECT 0xFFFFFFFFu
#define SW_OVERFLOW_SENTINEL (-1)   /* strip kernel: 16-bit range possibly exceeded, recomputed in 32 bit */
#define SW_OUT_I32  0
#define SW_OUT_I16  1
#define SW_OUT_TOPK 2
#define SW_OUT_HITS 3
#define SW_OUT_SBEST 4
#define SW_MAX_TOPK 32

/* Database shard resident in HBM.  Layout (DESIGN.md "data layout"):
 *   raw/off/len   : the caller's 2-bit packed records, as uploaded
 *   pair_subj     : [2*npairs] shard-local subject index of the low / high 16-bit
 *                   lane of pair p (SW_NO_SUBJECT = lane unused)
 *   pair_len      : [2*npairs] columns of the two members (low lane = the longer one)
 *   tp            : column codes, one byte per column (0..15 = t_lo | t_hi << 2; 16..19 = the
 *                   shorter member has ended; 20 = no column), four columns per 32-bit
 *                   word, tiles of 32 pairs, word k of the 32 pairs of a tile contiguous:
 *                   tp[tile_woff[tile] + k*32 + slot]   (null for DIRECT launches)
 */
struct SwDevDb {
    const uint8_t  *raw;
    const uint64_t *off;
    const uint32_t *len;
    uint32_t        ns;
    const uint32_t *pair_subj;
    const uint32_t *pair_len;
    const uint4    *pair_desc;   /* DIRECT launches: {n_lo, n_hi, subj_lo, subj_hi | off_lo, off_hi, 0, 0} per pair */
    const uint64_t *tile_woff;
    uint32_t       *tp;
    uint64_t        tp_words;
    uint32_t        npairs;
    uint32_t        max_len;
};

struct SwDevQueries {
    const uint8_t  *packed;   /* 2-bit packed, each query byte aligned */
    const uint32_t *off;      /* byte offset of each query             */
    const uint32_t *len;
    int             nq;
    uint32_t        max_len;
};

struct SwScoring {
    int match, mismatch, goe /* gap_open + gap_extend */, ge;
    int limit;                /* 0 = exact; else 2^(W-1)-1: M above it restarts at 0 */
};

/* One strip-kernel variant = (rows per lane R = RS*S, lanes per pair G). */
struct SwStripVariant {
    int R, G;
    int block_threads;
    int S;            /* independent sub-strips per lane (R = RS * S) */
    int min_blocks;   /* resident blocks per SM the kernel was compiled for */
    const char *name;
    int has_direct;   /* a DIRECT instance exists (codes formed on the fly: small-batch path) */
    int U;            /* columns per trip of the step loop */
    int FL;           /* interior-trip flags of the instance (sw_strip.cuh, SW_FAST_LOOP) */
};

int sw_strip_variant_count(void);
/* testing hook: true = never use the instances with compile-time gap penalties */
void sw_strip_disable_fixed(bool off);
const SwStripVariant *sw_strip_variant(int idx);

/* Dynamic shared memory of variant idx when the query profile of chunk_passes passes is resident. */
size_t sw_strip_smem_bytes(int idx, int chunk_passes);

/* Resident blocks per SM of variant idx with smem_bytes of dynamic shared memory. */
cudaError_t sw_strip_occupancy(int idx, size_t smem_bytes, int *blocks_per_sm);

/* Hit list (SW_OUT_HITS): keys[i] = row << shift | shard-local subject, score[i] = its score, for every pair
 * scoring >= min_score; *count counts past cap, stores stop there.  keys == null: append nothing. */
struct SwHitList {
    unsigned long long *keys = nullptr;
    int32_t *score = nullptr;
    unsigned long long *count = nullptr;   /* 64-bit: it counts past cap, and a shard can have >= 2^32 pairs */
    unsigned cap = 0;
    int min_score = 1, shift = 0;
};

/* Per-subject best (SW_OUT_SBEST): key[s] = score << 32 | (0xFFFFFFFF - row) of subject s's best row, second[s] = the
 * best score of its other rows (sbest_update in sw_strip.cuh); both over the shard's subjects.  key == null: update
 * nothing; second == null: one row only. */
struct SwSubjectBest {
    unsigned long long *key = nullptr;
    int32_t *second = nullptr;
};

/* One strip-kernel launch: queries qidx[0..nql) (or q0 .. q0+nql-1 when qidx is null) against all
 * pairs of db.  bnd: scratch for pass boundaries, grid * bnd_cols * (block_threads/G) uint2.
 * counter: zeroed device word (work queue) or null for a static schedule.  chunk_passes: passes (of
 * R*G rows) whose query profile is held in shared memory at once. */
struct SwStripLaunch {
    int vidx = -1;
    bool direct = false;
    SwDevDb db{};
    SwDevQueries q{};
    int q0 = 0, nql = 0;
    const int *qidx = nullptr;
    SwScoring sc{};
    void *out = nullptr;
    size_t out_stride = 0, out_elems = 0;
    int out_mode = SW_OUT_I32;
    uint2 *bnd = nullptr;
    uint32_t bnd_cols = 0;
    size_t bnd_elems = 0;
    unsigned *counter = nullptr;
    int sticky = 0;               /* > 0: counter points to nql zeroed words, one work queue per query (sw_strip.cuh);
                                     the value bounds the drift between the queues (pair blocks) */
    int grid = 0, chunk_passes = 1;
    /* pass split (sw_strip.cuh): nparts > 1 = an item covers part_passes passes (a multiple of chunk_passes)
       of its (pair block, query) chain; bnd then holds one boundary row per CHAIN (nql * pair blocks),
       part_done = zeroed progress words [chains], part_best = parked running maxima [chains * block threads] */
    int nparts = 0, part_passes = 0;
    unsigned *part_done = nullptr;
    uint32_t *part_best = nullptr;
    uint32_t superblock = 0;      /* pair blocks per super-block of the work order (0 = a tenth... npb / 8) */
    unsigned *ovf_count = nullptr;
    uint2 *ovf_list = nullptr;
    unsigned ovf_cap = 0;
    unsigned long long *topk_keys = nullptr;
    int topk_k = 0, topk_nq = 0;
    SwHitList hits{};             /* SW_OUT_HITS; out_elems is then the list's allocated length (bounds-check build) */
    SwSubjectBest sbest{};        /* SW_OUT_SBEST; out_elems is then the shard's subject count (bounds-check build) */
    unsigned *dev_err = nullptr;
    unsigned *done_count = nullptr, *done_flag = nullptr;   /* latency path: completion flag in mapped host memory */
    unsigned done_seq = 0;
    void *jit_kernel = nullptr;   /* cudaKernel_t of a run-time specialised instance (sw_jit.cu), or null */
};
cudaError_t sw_launch_strip(cudaStream_t st, const SwStripLaunch &L);
/* name of the instance sw_launch_strip would run ("fixed" / "runtime" / "w12" / "direct" / "jit") */
const char *sw_strip_instance_kind(const SwStripLaunch &L);

/* Band-pipelined kernel for few, long pairs (sw_wave.cuh): ONE query per launch, its bands are
 * separate work items that run concurrently on different warps.  bnd: npairs * 2 * cols_stride
 * 16-byte tagged elements (zeroed once when allocated; epoch makes the tags of earlier launches
 * stale); best: 2 * npairs ints, done: npairs words -- zeroed before the launch; counter: zeroed
 * work-queue word. */
#define SW_WAVE_ROWS_PER_BAND 512     /* instance 0; instances 1 and 2 have bands of 256 rows */
struct SwWaveLaunch {
    int instance = 0;
    SwDevDb db{};
    SwDevQueries q{};
    int query = 0;
    int out_row = -1;        /* row of out the scores go to; -1 = query */
    int npass = 0;
    SwScoring sc{};
    void *out = nullptr;
    size_t out_stride = 0;
    int out_mode = SW_OUT_I32;
    void *bnd = nullptr;
    uint32_t cols_stride = 0;
    size_t bnd_elems = 0, out_elems = 0;      /* sizes of bnd (16-byte elements) and out, for the check build */
    uint32_t epoch = 1;
    int *best = nullptr;
    unsigned *done = nullptr;
    unsigned *counter = nullptr;
    int grid = 0;
    unsigned *ovf_count = nullptr;
    uint2 *ovf_list = nullptr;
    unsigned ovf_cap = 0;
    unsigned *dev_err = nullptr;
};
cudaError_t sw_wave_occupancy(int instance, int *blocks_per_sm);
cudaError_t sw_launch_wave(cudaStream_t st, const SwWaveLaunch &L);
const char *sw_wave_kernel_name(int instance);
int sw_wave_rows_per_band(int instance);
int sw_wave_instance_count(void);
int sw_wave_pairs_per_block(int instance);

/* 32-bit band-pipelined scorer of the overflow list (sw_wave.cuh, sw_wave32_kernel): the first
 * SW_WAVE32_MAX_ENTRIES entries per launch (entry_base), of those below entry_limit with at least
 * min_cells cells; score32 (mode 2) with the same wave32_min_cells / wave32_limit skips exactly those.  bnd: nslots * 2 * cols_stride 16-byte elements (zeroed once
 * and whenever epoch restarts at 1); state: 3 * SW_WAVE32_MAX_ENTRIES zeroed words per launch. */
#define SW_WAVE32_MAX_ENTRIES 4096
#define SW_WAVE32_ROWS 256
struct SwWave32Launch {
    SwDevDb db{};
    SwDevQueries q{};
    SwScoring sc{};
    const unsigned *list_count = nullptr;
    const uint2 *list = nullptr;
    unsigned list_cap = 0;
    unsigned entry_base = 0, entry_limit = SW_WAVE32_MAX_ENTRIES;   /* this launch's first list entry; entries all launches take */
    int32_t *list_score = nullptr;
    void *out = nullptr;
    size_t out_stride = 0, out_elems = 0;
    int out_mode = SW_OUT_I32;
    void *bnd = nullptr;
    uint32_t cols_stride = 0, nslots = 0, epoch = 1;
    size_t bnd_elems = 0;
    unsigned *state = nullptr;
    unsigned *counter = nullptr;
    uint32_t maxb = 1;
    unsigned long long min_cells = 0;
    int grid = 0;
    unsigned *dev_err = nullptr;
};
cudaError_t sw_wave32_occupancy(int *blocks_per_sm);
cudaError_t sw_launch_wave32(cudaStream_t st, const SwWave32Launch &L);

/* 32-bit kernel: any length, any score range.  scratch: 2 * max_cols * threads_total int32 where
 * max_cols = min(longest query, longest subject) (the recurrence is symmetric: the shorter sequence
 * is walked as columns).  mode 0: every (query, subject) job of q0..q1; mode 1: only matrix entries
 * equal to SW_OVERFLOW_SENTINEL; mode 2: the (query, subject) entries of the overflow list, results
 * to the matrix (if out != null) and to list_score[i]. */
struct SwScore32Launch {
    SwDevDb db{};
    SwDevQueries q{};
    int q0 = 0, q1 = 0;
    SwScoring sc{};
    void *out = nullptr;
    size_t out_stride = 0;
    int out_mode = SW_OUT_I32;
    int32_t *scratch = nullptr;
    uint32_t max_cols = 0;
    int threads_total = 0;
    int mode = 0;
    const unsigned *list_count = nullptr;
    const uint2 *list = nullptr;
    unsigned list_cap = 0;
    int32_t *list_score = nullptr;
    unsigned long long wave32_min_cells = 0;   /* mode 2: entries sw_wave32_kernel takes are skipped (0 = none) */
    unsigned wave32_limit = 0;                 /* ... among the first wave32_limit list entries */
};
cudaError_t sw_launch_score32(cudaStream_t st, const SwScore32Launch &L);

/* Begin / end of the best local alignment of selected pairs (sw_locate.cu, sw_locate_db): one thread per entry of
 * pairs[0 .. npairs) = {query row, shard-local subject}; score[i] = its score, coord[i] = {q_begin, q_end, s_begin,
 * s_end}.  scratch: 2 * max_cols * threads_total int32, max_cols >= the longest subject of the pairs.  raw_bytes /
 * q_bytes / out_elems: sizes of db.raw, q.packed and the two result arrays (bounds-check build).  Exact scores only (sc.limit is ignored). */
struct SwLocateLaunch {
    SwDevDb db{};
    size_t raw_bytes = 0;
    SwDevQueries q{};
    size_t q_bytes = 0;
    SwScoring sc{};
    const uint2 *pairs = nullptr;
    uint32_t npairs = 0;
    int32_t *score = nullptr;
    uint4 *coord = nullptr;
    size_t out_elems = 0;
    int32_t *scratch = nullptr;
    uint32_t max_cols = 0;
    int threads_total = 0;
    unsigned *dev_err = nullptr;
};
cudaError_t sw_launch_locate(cudaStream_t st, const SwLocateLaunch &L);

/* CIGAR of the located best alignment of selected pairs (sw_locate.cu, sw_align_db): one thread per pair of
 * loc.pairs[job0 .. job1).  loc.score / loc.coord hold sw_launch_locate's results for those pairs (read here).  Each
 * pair with score > 0 stores 4 direction bits per cell of its rectangle in trace[trace_off[i] ..], ceil(m / 16) * n
 * words for an m x n rectangle, and writes its run-length BAM ops to ops[ops_off[i] ..], at most m + n - 1 of them,
 * and their count to nops[i] (0 for score 0).  loc.scratch as for sw_launch_locate. */
struct SwAlignLaunch {
    SwLocateLaunch loc{};
    uint32_t job0 = 0, job1 = 0;
    const uint64_t *trace_off = nullptr;
    uint64_t *trace = nullptr;
    uint64_t trace_words = 0;
    const uint64_t *ops_off = nullptr;
    uint32_t *ops = nullptr;
    uint64_t ops_elems = 0;
    uint32_t *nops = nullptr;
};
cudaError_t sw_launch_align(cudaStream_t st, const SwAlignLaunch &L);

cudaError_t sw_launch_build_tp(cudaStream_t st, const SwDevDb &db);

/* Per-query arg-max over subjects of a materialised int32 matrix (first index reaching the max). */
cudaError_t sw_launch_best(cudaStream_t st, const int32_t *scores, size_t stride, uint32_t ns,
                           int nq, int32_t *best_score, uint32_t *best_index);

/* Folds the per-block top-k lists (nlists x nq x k keys) and the recomputed overflow entries into
 * out_keys[nq][k] (descending; key = score << 32 | ~subject, 0 = no entry). */
/* Top-k of one materialised score row (entries < 0 are skipped) written as list 0 of query q in the
 * per-block key lists that sw_launch_topk_merge folds: the band-pipelined kernel has no top-k epilogue. */
cudaError_t sw_launch_topk_row(cudaStream_t st, const int32_t *row, uint32_t n, int q, int k, unsigned long long *keys);
cudaError_t sw_launch_topk_merge(cudaStream_t st, const unsigned long long *keys, int nlists, int nq, int k,
                                 const unsigned *ovf_count, const uint2 *ovf_list, const int32_t *ovf_score,
                                 unsigned ovf_cap, unsigned long long *out_keys);

/* Hit-list entries that do not come from the strip epilogue, appended with one atomicAdd per warp like
 * there: hits_row = the entries >= min_score of one materialised score row of query row q
 * (entries < 0 are skipped: not scored here, or the overflow sentinel) -- the band-pipelined kernel's rows;
 * hits_ovf = the overflow-list entries whose exact 32-bit score (ovf_score) is >= min_score. */
cudaError_t sw_launch_hits_row(cudaStream_t st, const int32_t *row, uint32_t n, int q, const SwHitList &hl);
cudaError_t sw_launch_hits_ovf(cudaStream_t st, const unsigned *ovf_count, const uint2 *ovf_list, const int32_t *ovf_score,
                               unsigned ovf_cap, const SwHitList &hl);

/* Per-subject best updates that do not come from the strip epilogue: sbest_row = every entry >= 0 of one
 * materialised score row of query row q (entries < 0 are skipped: not scored here, or the overflow sentinel) -- the
 * band-pipelined kernel's rows; sbest_ovf = the overflow-list entries with their exact 32-bit score (ovf_score). */
cudaError_t sw_launch_sbest_row(cudaStream_t st, const int32_t *row, uint32_t n, int q, const SwSubjectBest &sb);
cudaError_t sw_launch_sbest_ovf(cudaStream_t st, const unsigned *ovf_count, const uint2 *ovf_list, const int32_t *ovf_score,
                                unsigned ovf_cap, const SwSubjectBest &sb);

#endif
