/*
 * sw_b200.h -- C ABI of the B200-native score-only Smith-Waterman engine
 *              (libsw_b200.so, built from smith-waterman-fpga-module_b200/csrc/).
 *
 * This is the drop-in boundary for the reference's hot path: the systolic
 * scoring datapath (SW_ProcessingElement_v1 -> ScoringModule_v1_1 ->
 * ScoreBank_v2) and the CAPI job/MMIO/DMA shell that reaches it.  Each entry
 * point cites the reference interface it replaces; paths are relative to the
 * reference checkout.  Plain C types only (no torch / CUDA types).
 *
 * Operator surface that is kept (ScoreBank_v2.v:31-44):
 *   load penalties once -> load a query -> stream targets -> collect one
 *   max local-alignment score per (query, target).
 * Sequences are 2-bit packed exactly as the reference host packs them
 * (aligner_Header.c:14-47): A=10 C=01 G=11 T=00, base k in byte k/4 at bit
 * 2*(k%4), anything else packs as 00.
 *
 * Threading: a handle is not re-entrant (the reference host is strictly
 * single-threaded, main_test.c:214-537); distinct handles are independent.
 * Every call returns 0 (SW_OK) or a negative SW_E* code.  There is no CPU
 * fallback: without a usable CUDA device sw_init fails with SW_ENODEV.
 */
#ifndef SW_B200_H_
#define SW_B200_H_

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (replace the WED error bitfield, main_test.c:64-100) ---- */
#define SW_OK          0
#define SW_EINVAL     -1   /* bad argument / unsupported parameter set          */
#define SW_ENOMEM     -2   /* host or device allocation failed                  */
#define SW_ECUDA      -3   /* CUDA runtime error, see sw_last_cuda_error()      */
#define SW_ENODEV     -4   /* no CUDA device / requested GPU id not present     */
#define SW_ESTATE     -5   /* call out of order (e.g. fetch before score_batch) */
#define SW_ETIMEOUT   -6   /* sw_fetch timed out (the host's -t option)         */
#define SW_ECAPACITY  -7   /* caller's score buffer too small                   */
#define SW_EIO        -8   /* file could not be read / written                  */
#define SW_EAGAIN     -9   /* both batch buffers in flight (the bank's `full`)   */
#define SW_ERANGE     -10  /* more scores beyond 16 bits than the side list holds: use int32 output */
#define SW_EDEVICE    -11  /* a device-side check failed (bounds-check build / wavefront watchdog)   */

/* The `penalties` bus + SCORE_WIDTH parameter.
 * Replaces: ScoreBank_v2.v:34,161 (ld_penalties, penalties[4*W]),
 *           SW_ProcessingElement_v1.0.v:15 (SCORE_WIDTH),
 *           defaults ScoreBank_v1_tb.sv:16-19. */
typedef struct sw_params {
    int16_t match;        /* default   5 */
    int16_t mismatch;     /* default  -4 */
    int16_t gap_open;     /* default -12 */
    int16_t gap_extend;   /* default  -4  (first gap residue costs open+extend) */
    int32_t score_width;  /* 0 = exact integers (default); 12 = RTL-faithful
                             12-bit biased machine: M wraps to 0 above 2047   */
} sw_params_t;

typedef struct sw_handle sw_handle_t;

/* Fills *p with the reference defaults (5/-4/-12/-4, exact width). */
void sw_default_params(sw_params_t *p);

/* Exactness domain.  sw_init accepts every parameter set with match > 0, gap_extend <= 0 and
 * gap_open + gap_extend <= 0 and scores it with the general recurrence (I(i,1) takes M(i-1,1)
 * into account).  The RTL itself is only schedule-INdependent when match + gap_open <= 0: for the
 * first target base of a stream the PE may ignore the upper neighbour's M -- always in PE v0.3
 * (SW_ProcessingElement_v0.3.v:145-158), and in v1.0 whenever neither time-share slot is
 * mid-sequence (SW_ProcessingElement_v1.0.v:120 vs :131-141).  Both forms coincide iff
 * match + gap_open <= 0 (default: 5 - 12 < 0).
 * Returns 1 = bit-exact against the RTL for every input, 0 = accepted, but the RTL's own result
 * depends on its feeder schedule there (this engine returns the general-form score),
 * SW_EINVAL = the set is rejected by sw_init.  p == NULL asks about the defaults. */
int sw_params_in_exact_domain(const sw_params_t *p);

/* Replaces: cxl_afu_open_dev + cxl_afu_attach (main_test.c:342,370) and the
 * ld_penalties cycle (ScoreBank_v1_tb.sv:175-181).  gpu_ids == NULL with
 * n_gpus == 0 means "device 0".  One stream set + pinned staging per GPU. */
int sw_init(sw_handle_t **h, const sw_params_t *p, const int *gpu_ids, int n_gpus);

/* Replaces: cxl_afu_free (main_test.c:533). */
void sw_destroy(sw_handle_t *h);

/* Replaces: the type-01 record / ld_q (ScoreBank_v2.v:162,181-182;
 * ScoringModule_v1.1.v:121-126).  Queries are copied and replicated to every
 * GPU.  packed + off[i] is the first byte of query i, len[i] its base count. */
int sw_set_queries(sw_handle_t *h, const uint8_t *packed, const uint32_t *len,
                   const uint64_t *off, int nq);

/* Both strands: when enabled (before sw_set_queries), every query is also scored as its reverse
 * complement; the score matrix then has 2*nq rows, row nq + i = reverse complement of query i.
 * The reference ran ssearch36 with -3 to switch this off (data/ssearch36_command:2) while
 * data/res shows [r] hits; default is forward only.  sw_query_rows = rows per subject. */
int sw_set_strands(sw_handle_t *h, int both);
int sw_query_rows(const sw_handle_t *h);

/* Replaces: the stream of type-10 records with feeder / PrioEncoder arbitration
 * (ScoreBank_v2.v:142-169, SM_Feeder2.v:104-205, PrioEncoder.v:18-21) and the
 * DMA read of the sequence array (afu.v:383-398).  Subjects are length-bucketed,
 * sharded over the handle's GPUs, copied H2D and scored against every query.
 * Asynchronous with respect to the GPUs: returns once the work is enqueued; the
 * caller's buffers may be reused as soon as it returns.  ids may be NULL
 * (then id = input index); they are returned by sw_fetch_ids.
 * Streaming: TWO batches may be in flight (double buffering like the feeder's two target
 * slots): submit batch k+1 before fetching batch k and its sort / H2D / kernels overlap the
 * D2H of batch k.  SW_EAGAIN when both buffers are busy (the bank's `full` wire);
 * sw_fetch returns batches in submission order. */
int sw_score_batch(sw_handle_t *h, const uint8_t *packed, const uint32_t *len,
                   const uint64_t *off, const uint64_t *ids, size_t ns);

/* Replaces: the (IDs, results, vld) outputs (ScoreBank_v2.v:39-41), the WED
 * status poll with timeout (main_test.c:422-477) and `*result-2048`
 * (main_test.c:528).  Blocks until the batch is complete or timeout_ms elapses
 * (timeout_ms < 0 = wait forever).  scores[iq * ns + is] = unbiased score of
 * query iq against subject is, in INPUT order (deterministic, unlike the RTL's
 * completion order).  cap = number of int32 the buffer holds. */
int sw_fetch(sw_handle_t *h, int32_t *scores, size_t cap, int timeout_ms);
int sw_batches_in_flight(const sw_handle_t *h);      /* 0, 1 or 2 */

/* Replaces: the 48-bit ID that travels with every target record and comes back next to
 * its score (ScoreBank_v2.v:26-28,40; fifo.v:36-64).  ids[is] = the id given to
 * sw_score_batch / sw_load_db for subject is (or is itself when ids was NULL). */
int sw_fetch_ids(sw_handle_t *h, uint64_t *ids, size_t cap);

/* ---- resident-database path (database stays in HBM between calls) ---------
 * sw_load_db     = the H2D half of sw_score_batch (bucket, shard, upload).
 * sw_score_db    = enqueue scoring of all current queries against the resident db.
 * sw_wait        = block until enqueued work is done.
 * sw_fetch_db    = D2H of the score matrix of the last sw_score_db.
 * These replace nothing in the reference (its feeder holds two targets); they
 * exist so that a database larger than one batch is not re-uploaded per query set. */
int sw_load_db(sw_handle_t *h, const uint8_t *packed, const uint32_t *len,
               const uint64_t *off, const uint64_t *ids, size_t ns);
int sw_score_db(sw_handle_t *h);
int sw_wait(sw_handle_t *h, int timeout_ms);
int sw_fetch_db(sw_handle_t *h, int32_t *scores, size_t cap);

/* The shard plan sw_load_db uses: contiguous input ranges [starts[g], starts[g+1]) balanced by
 * residue count (the work of a subject is proportional to its length).  Pure host code;
 * starts must hold n_shards + 1 entries.  Replaces the bank's broadcast-query /
 * distribute-targets structure (ScoreBank_v2.v:78-139) at the GPU level. */
int sw_plan_shards(const uint32_t *len, size_t ns, int n_shards, uint64_t *starts);

/* Per-query best hit over the resident db, reduced on the GPU: the `max` /
 * `vld_max` outputs ScoreBank_v2 declares but never drives (ScoreBank_v2.v:42-43).
 * best_score[iq], best_index[iq] (input index of the first subject reaching it).
 * Matrix output modes only; in top-k mode use sw_fetch_db_topk. */
int sw_fetch_best(sw_handle_t *h, int32_t *best_score, uint64_t *best_index, int nq_cap);

/* ---- output path ------------------------------------------------------------
 * The bank returns a 12-bit score per (ID) slot (ScoreBank_v2.v:39-41); the result buffer the
 * reference planned (CAPI_template/ResBuffer.v:11-22) has ports only.  Four shapes here (the fourth, the hit
 * list of sw_set_hits, is described below):
 *   SW_OUTPUT_I32   int32 matrix [rows][ns]                     (default; sw_fetch / sw_fetch_db)
 *   SW_OUTPUT_I16   int16 matrix [rows][ns]: half the HBM and half the D2H bytes.  A score above
 *                   32767 is stored as -1 in the matrix and returned exactly by sw_fetch_overflow
 *                   (flat index iq * ns + is, int32 score); SW_ERANGE if there are more than 2^20.
 *   top-k           sw_set_topk(h, k), 1 <= k <= 32 (0 = back to matrices): NO score matrix is
 *                   allocated or shipped; the strip kernel's epilogue keeps the k best
 *                   (score, subject) per query -- the `max` / `vld_max` outputs of
 *                   ScoreBank_v2.v:42-43, generalised to k -- merged across blocks, launches and
 *                   the handle's GPUs.  Order: score descending, ties by ascending input index.
 *                   With fewer than k subjects the tail has index UINT64_MAX and score -1.
 * Modes are set while no batch is in flight and apply to the following sw_score_batch /
 * sw_score_db calls.  Streaming (two batches in flight) works in every mode; each batch has its
 * own top-k (merge across batches with a k-way merge on (score, index) if needed). */
#define SW_OUTPUT_I32 0
#define SW_OUTPUT_I16 1
int sw_set_output(sw_handle_t *h, int mode);
int sw_set_topk(sw_handle_t *h, int k);
int sw_fetch_i16(sw_handle_t *h, int16_t *scores, size_t cap, int timeout_ms);
int sw_fetch_db_i16(sw_handle_t *h, int16_t *scores, size_t cap);
/* Scores above 32767 of the batch / database fetched last in SW_OUTPUT_I16 mode.  *count = how many
 * there are; at most cap are written. */
int sw_fetch_overflow(sw_handle_t *h, uint64_t *flat_index, int32_t *score, size_t cap, size_t *count);
/* scores[iq * k + j], index[iq * k + j] (input index within the batch), j-th best hit of query iq;
 * cap = entries both arrays hold (>= rows * k). */
int sw_fetch_topk(sw_handle_t *h, int32_t *scores, uint64_t *index, size_t cap, int timeout_ms);
int sw_fetch_db_topk(sw_handle_t *h, int32_t *scores, uint64_t *index, size_t cap);

/* Hit list: every (row, subject) pair with score >= min_score, in place of a matrix.  Replaces the bank's
 * (IDs, results, vld) stream (ScoreBank_v2.v:39-41), filtered on `results`.  min_score >= 1 turns it on,
 * 0 turns it off (back to matrices).  Each GPU's list holds max_hits entries per batch slot.
 *   Entries: exactly the entries of the int32 matrix that are >= min_score -- row = query row (row nq + i =
 *   reverse complement of query i with sw_set_strands(h, 1)), index = input index within the batch (ids via
 *   sw_fetch_ids), score = the exact int32 score, above 32767 too -- in row-major order (row ascending, then
 *   index ascending), the same for every kernel, work order and GPU count.  The int16 / int32 output setting is
 *   ignored while hits are on.
 *   Setting: like the other modes, only while no batch is in flight (SW_EAGAIN), and scored batches become
 *   stale.  Hits and top-k exclude each other (SW_EINVAL either way round); min_score < 0, min_score > 0 with
 *   max_hits == 0 or max_hits > 2^31 - 1 is SW_EINVAL.  Submitting with the forced 32-bit scorer
 *   (sw_set_kernel_choice force32) is SW_EINVAL; nothing is enqueued then.
 *   Fetching: *count = the exact number of hits.  cap < *count: SW_ECAPACITY, nothing written, the batch stays
 *   fetchable and a retry with larger arrays returns the same list without rescoring (cap = 0 with null arrays
 *   is the size query).  A GPU that found more than max_hits hits, or more scores beyond 16 bits than the side
 *   list holds: SW_ERANGE, nothing written, the batch is consumed (raise max_hits or min_score and score
 *   again).  Fetching a hits batch with a matrix / top-k / best-hit call, or a batch of another mode with these
 *   two, is SW_ESTATE. */
int sw_set_hits(sw_handle_t *h, int32_t min_score, size_t max_hits);
int sw_fetch_hits(sw_handle_t *h, uint32_t *row, uint64_t *index, int32_t *score, size_t cap, size_t *count, int timeout_ms);
int sw_fetch_db_hits(sw_handle_t *h, uint32_t *row, uint64_t *index, int32_t *score, size_t cap, size_t *count);

/* ---- introspection --------------------------------------------------------- */
const char *sw_strerror(int code);
int sw_last_cuda_error(const sw_handle_t *h);          /* cudaError_t as int */
const char *sw_last_cuda_error_string(const sw_handle_t *h);
/* Device time (CUDA events on the launching stream) of the scoring kernels of the
 * last sw_score_db / sw_score_batch, max over the handle's GPUs, milliseconds. */
double sw_last_kernel_ms(const sw_handle_t *h);
/* Host-visible phase times of the last sw_score_batch / sw_load_db (load_ms: length sort, pairing,
 * H2D issue and completion; enqueue_ms: kernel launches) and of the last sw_fetch / sw_fetch_db
 * (fetch_wait_ms: waiting for kernels while issuing the D2H copies of finished query chunks;
 * fetch_drain_ms: waiting for the last copies).  kernel_ms_max / _min: device time (CUDA events) of
 * the slowest / fastest GPU of the handle -- their ratio is the shard imbalance.  The reference's
 * counterpart is the `_DEBUGGING_` cycle counter of afu.v:497-532. */
typedef struct sw_stats {
    double load_ms, enqueue_ms, fetch_wait_ms, fetch_drain_ms, kernel_ms_max, kernel_ms_min;
} sw_stats_t;
int sw_get_stats(const sw_handle_t *h, sw_stats_t *out);
/* Device-side error word, OR-ed over the handle's GPUs (0 = clean): set by the index checks of the
 * bounds-check build (libsw_b200_check.so, make CHECK=1 -- this pool has no compute-sanitizer) and
 * by the wavefront kernel's spin-wait watchdog.  Also reports canary damage around device buffers
 * (bit 31).  Fetch calls return SW_EDEVICE when it is non-zero. */
unsigned sw_device_error_bits(sw_handle_t *h);
/* 1 if this library was built with -DSW_BOUNDS_CHECK */
int sw_is_check_build(void);
/* Number of kernels this library launched since sw_init (all GPUs). */
uint64_t sw_kernel_launches(const sw_handle_t *h);
/* Cell updates (sum of qlen*tlen over all pairs) of the last scoring call. */
uint64_t sw_last_cells(const sw_handle_t *h);
/* Name of the kernel variant chosen for the last scoring call, e.g.
 * "strip_s16x2_R50_G1"; static storage. */
const char *sw_last_kernel_name(const sw_handle_t *h);
/* Overrides the automatic kernel choice (testing / benchmarking):
 * rows_per_lane in {0=auto, ...}, lanes_per_pair in {0=auto,1,2,4,8,16,32},
 * force32 != 0 forces the 32-bit fallback kernel. */
int sw_set_kernel_choice(sw_handle_t *h, int rows_per_lane, int lanes_per_pair, int force32);
/* arith: -1 = automatic, 0 = packed signed 16-bit (DPX).  Other arithmetic policies were
 * measured and dropped (DESIGN.md section 5.1); anything else is SW_EINVAL. */
int sw_set_arith(sw_handle_t *h, int arith);
/* The strip-kernel variants compiled into the library, and forcing one by name
 * (NULL or "" = back to automatic).  Names look like "strip_s16x2_R25x2_G1":
 * 25 rows x 2 sub-strips per lane, 1 lane per subject pair. */
/* The main variants also exist with the reference's gap penalty sets (-12 / -4, and -8 / -4 of its
 * swalign vectors) compiled in as immediates (about 6 % faster: fewer register operands); they are
 * used automatically when the handle's penalties match.  enable = 0 forces the run-time-penalty kernels (process-wide;
 * for A/B measurements and tests). */
int sw_set_fixed_penalty_kernels(int enable);
/* Large jobs (>= ~0.4 s of estimated work): the three variants the cost model ranks best are timed
 * on a ~20 ms sample of the actual workload and the fastest one runs; the decision is cached per
 * workload shape.  enable = 0 uses the model's first choice only.  Default: on
 * (environment SW_B200_AUTOTUNE=0 turns it off at sw_init). */
int sw_set_autotune(sw_handle_t *h, int enable);
/* Run-time specialisation of the gap penalties (the reference loads them at run time: ld_penalties,
 * ScoreBank_v2.v:34,161).  For a penalty set that is not compiled in, the one kernel variant a job
 * uses is compiled with the penalties as immediates (NVRTC, loaded lazily with dlopen; cubins are
 * cached in $SW_B200_JIT_CACHE, default ~/.cache/sw_b200) -- same speed as the default set instead
 * of ~7 % less.  mode 0 = never, 1 = jobs of >= ~2 s of estimated work (default), 2 = always
 * (environment SW_B200_JIT).  Without NVRTC the run-time-operand kernels are used; nothing fails. */
int sw_set_jit(sw_handle_t *h, int mode);
int sw_jit_is_available(void);
/* Compiles (or takes from the cache) the specialised instance of one variant: 1 = ready, 0 = not
 * available, msg says why (NVRTC missing, compile error, or no GPU to load the cubin on). */
int sw_jit_compile_check(const char *variant_name, int gap_open, int gap_extend, char *msg, size_t msg_cap);
/* Small batches (<= 8192 subjects, <= 1 MB of packed bases) submitted with sw_score_batch take a
 * latency path: one staging copy, one kernel, scores written to mapped host memory (the regime of
 * the reference's own data sets: data/data500.fa is 499 x 128 nt).  enable = 0 forces the regular
 * path (environment SW_B200_SMALL_PATH=0). */
int sw_set_small_batch_path(sw_handle_t *h, int enable);
/* The latency path records two CUDA events around its kernel so that sw_last_kernel_ms works
 * (about 2 us of host time per batch); enable = 0 drops them (sw_last_kernel_ms then reports 0). */
int sw_set_small_batch_timing(sw_handle_t *h, int enable);
/* Few, long pairs (a long query against a handful of subjects, down to ONE pair): the 512-row bands
 * of the query become separate work items that run concurrently on different warps / SMs, each
 * band consuming the bottom row of the band above as it is produced -- the module chaining the
 * reference left "for future use" (ScoringModule_v1.1.v:36-39, 49-54).  mode 0 = never,
 * 1 = automatic (default: <= 1536 subject pairs and a query of >= 1024 rows, or <= 64 pairs and a
 * query of > 512 rows, or every query >= 1024 rows and too few pairs to fill whole rounds of the
 * strip kernel's work items), 2 = whenever the query has more than one band (environment SW_B200_WAVE). */
int sw_set_wave_mode(sw_handle_t *h, int mode);
/* Scores that leave the 16-bit range of the packed kernels (the reference's SCORE_WIDTH is a
 * synthesis parameter, SW_ProcessingElement_v1.0.v:26; here 32 bits are used where needed) are
 * recomputed from the overflow list.  With the default scoring such a pair is at least 6 400 x
 * 6 400 nt, so entries of at least min_cells cells (default 10^6; the first 16 384 of a call) are
 * scored by 256-row bands on many warps in 32-bit arithmetic, the rest by one thread each.
 * enable = 0 leaves every entry to the one-thread scorer (environment SW_B200_WAVE32=0). */
int sw_set_overflow_wave(sw_handle_t *h, int enable, unsigned long long min_cells);
/* Launch plan of a scoring call.  The bank hands every target to the first free module
 * (PrioEncoder.v:18-21, SM_Feeder2.v:104-205); here the sorted pair list can be cut into length
 * groups (a group ends where the length has halved), each with its own launch, kernel variant and
 * pass-boundary scratch, running on concurrent streams.  length_groups: 0 = one launch over all
 * lengths, 1 = always one launch per length group, 2 = automatic (default): length groups only when
 * one launch would need more than 4 GB of pass-boundary scratch (a few very long subjects next to
 * many short ones).  query_groups != 0: additionally choose the variant per query length (default
 * off: on the mixed-length config the extra launches cost more than the better fit gains --
 * measured 7.3 vs 8.2 TCUPS). */
int sw_set_launch_plan(sw_handle_t *h, int length_groups, int query_groups);
/* Pass split.  A free module of the bank is handed the next target at once, whatever it is
 * (ScoreBank_v2.v:78-139), so the bank idles only at the very end of a database.  A strip-kernel work item
 * is (block of pairs, query) for ALL passes of the query: with a long query and a database of a few
 * rounds of such items (200 k x 1 kb subjects against one 10 kb query = 2.64 rounds) the last, partly
 * filled round leaves much of the GPU idle for the length of a whole item.  The split cuts the passes
 * of an item into parts that are handed out as separate items, part-major; the chain's boundary row and
 * running maximum wait in device scratch between parts.  mode: 0 = never, -1 = automatic (default: one
 * launch of 1 .. 16 rounds of multi-chunk items), n >= 2 = about n parts whenever the query spans at
 * least two profile chunks (environment SW_B200_PASS_SPLIT).  sw_last_pass_parts: parts per item of
 * the last scoring call's plan on the handle's first GPU (1 = not split). */
int sw_set_pass_split(sw_handle_t *h, int mode);
int sw_last_pass_parts(const sw_handle_t *h);
/* The split's arithmetic, without a device (what the automatic rule would do for npass passes in profile
 * chunks of chunk_passes, `chains` = pair blocks x queries of the launch, on `grid` resident blocks).
 * Returns 1 and the number of parts / passes per part, or 0 = not split (nparts = 1). */
int sw_plan_pass_parts(int npass, int chunk_passes, unsigned long long chains, int grid, int mode, int *nparts, int *part_passes);
int sw_kernel_variant_count(void);
const char *sw_kernel_variant_name(int idx);
int sw_set_kernel_name(sw_handle_t *h, const char *name);
int sw_device_count(void);
const char *sw_version(void);

/* ---- pure-host helpers (file-level drop-in) -------------------------------- */
/* Replaces: charTo2bit (aligner_Header.c:14-47).  out must hold (len+3)/4 bytes. */
void sw_pack_2bit(const char *seq, size_t len, uint8_t *out);
void sw_unpack_2bit(const uint8_t *packed, size_t len, char *out /* len+1 */);

/* A set of sequences, packed.  Owned by the library; free with sw_seqset_free. */
typedef struct sw_seqset {
    size_t    n;
    uint8_t  *packed;     /* concatenated 2-bit data, each record byte-aligned   */
    uint32_t *len;        /* bases per record                                     */
    uint64_t *off;        /* byte offset of each record in packed                 */
    char    **name;       /* record names without the leading '>'                 */
    size_t    packed_bytes;
} sw_seqset_t;

/* Replaces: the testbench FASTA parser (ScoreBank_v1_tb.sv:184-216): `>name`
 * then sequence; wrapped sequence lines are concatenated.  A file with no '>'
 * line is read like main_test.c:304,310 does: first whitespace token = the
 * sequence, name "seq0". */
int sw_read_fasta(const char *path, sw_seqset_t **out);
void sw_seqset_free(sw_seqset_t *s);

/* Replaces: Display_results (ScoreBank_v1_tb.sv:271-285), one line per subject,
 * "@%6dns: %10s score: \t%11d" with the name prefixed by '>'.  The engine has no
 * simulation clock: time_ns[i] is printed if given, else 0. */
int sw_write_out_txt(FILE *f, const sw_seqset_t *db, const int32_t *scores,
                     const uint64_t *time_ns);
/* ssearch36 -R style rows (data/score500.txt:1-3): score is the 6th field. */
int sw_write_ssearch_R(FILE *f, const char *query_file, const char *db_file,
                       const sw_seqset_t *query, const sw_seqset_t *db,
                       const int32_t *scores);

#ifdef __cplusplus
}
#endif
#endif /* SW_B200_H_ */
