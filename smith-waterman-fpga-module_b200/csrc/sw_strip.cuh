/*
 * sw_strip.cuh -- the strip kernel of the score-only Smith-Waterman engine (hand-written sm_100a).
 * Included by the sw_variants_*.cu translation units (ahead-of-time instances) and embedded as
 * source text for run-time specialisation of the gap penalties (sw_jit.cu).
 *
 * What is computed (reference: ScoreBank/SW_ProcessingElement_v1.0.v:119-129, 287-291,
 * 411-420; SURVEY Appendix A.1), per (query, subject) pair, i = query row, j = subject column:
 *     M(i,j) = max(0, s(i,j) + H(i-1,j-1))          H = max(M, I)
 *     I(i,j) = max(G(i-1,j), G(i,j-1))              G = max(M + go + ge, I + ge)
 *     score  = max over all cells of H
 * with H = 0 and G = max(go+ge, ge) on both boundaries.  G is "the gap value leaving a
 * cell"; substituting it back gives exactly the RTL's M_open / I_extend form.
 *
 * How it is mapped to the GPU (replaces the systolic array of ScoringModule_v1.1.v and the
 * two-way time sharing of each PE, SW_ProcessingElement_v1.0.v:25-27):
 *   - two subjects of similar length share every 32-bit register (low / high 16-bit lane) --
 *     the PE's toggle-0 / toggle-1 sequences; the shorter one sees PAD scores once it has ended;
 *   - a lane keeps R consecutive query rows of H and G in registers and walks the subject
 *     columns; per cell pair the arithmetic is 3.5 ALU-pipe + 1 FMA-pipe instructions
 *     (VIMNMX.S16x2, VIADDMNMX.S16x2.RELU, VIADDMNMX.S16x2, 1/2 VIMNMX3.S16x2; VIADD.16x2);
 *   - G lanes of a warp form a systolic group over R*G rows: lane l is one column behind
 *     lane l-1 and receives (H, G, column code) with __shfl_up_sync, exactly like
 *     M_in / I_in / data_in travel from PE to PE;
 *   - queries longer than R*G rows are processed in passes; the bottom row of a pass is kept
 *     in an L2-resident scratch line per column and read back by lane 0 in the next pass;
 *   - substitution scores come from a shared-memory query profile
 *     prof[sub-strip][row pair][column code][lane of the group] (one uint2 = two rows), laid out
 *     so that the lanes of a warp hit distinct banks: one LDS.64 per two rows.
 * The recurrence is evaluated in an algebraically equivalent "clamped, goe-shifted" form (see
 * column_step_multi) that needs 3.5 ALU-pipe + 1 FMA-pipe instructions per two cells; the
 * RTL-faithful 12-bit mode keeps the explicit M form.
 */
#ifndef SW_STRIP_CUH_
#define SW_STRIP_CUH_

#ifndef SW_JIT_BUILD
#include <stdint.h>
#endif

#ifndef SW_STEP_UNROLL
#define SW_STEP_UNROLL 4      /* columns per trip of the step loop; nsteps is rounded up to a multiple */
#endif

#ifndef SW_FAST_LOOP
#define SW_FAST_LOOP 0        /* bit 0: G = 1 instances run predicate-free trips over the interior columns of a
                                 warp; bits 1 / 2 (A/B): no L1 prefetch of the code stream / boundary row there */
#endif

#define SW_NO_SUBJECT 0xFFFFFFFFu
#define SW_OVERFLOW_SENTINEL (-1)   /* 16-bit range possibly exceeded: the pair is on the overflow list */

/* output modes of the strip epilogue */
#define SW_OUT_I32  0               /* int32 out[q][subject]                                     */
#define SW_OUT_I16  1               /* int16 out[q][subject]                                     */
#define SW_OUT_TOPK 2               /* no matrix: per-block private top-k lists, merged later    */
#define SW_OUT_HITS 3               /* no matrix: (row << hits_shift | subject, score) of every score >= min_score */
#define SW_OUT_SBEST 4              /* no matrix: per subject the best (score, lowest row) and the runner-up score */

/* device-side error word (bit set = which check failed); only written by SW_BOUNDS_CHECK builds
 * and by the wave kernel's spin-wait guard */
#define SW_DEVERR_TP     1u
#define SW_DEVERR_BND    2u
#define SW_DEVERR_PROF   4u
#define SW_DEVERR_OUT    8u
#define SW_DEVERR_SPIN  16u
#define SW_DEVERR_TOPK  32u

namespace swk {

template <bool B> struct BoolTag { static constexpr bool value = B; };

constexpr int kPadScoreS16 = -8192;   // profile value of padding rows: M becomes 0, nothing can grow

// ------------------------------------------------------------------------------------------
// Packed signed 16-bit arithmetic: two independent subjects per 32-bit register, one DPX
// instruction per operation.
// ------------------------------------------------------------------------------------------
struct ArithS16 {
    static constexpr int kPad = kPadScoreS16;
    static __device__ __forceinline__ uint32_t addmax_relu(uint32_t a, uint32_t b, uint32_t c) {
        return __viaddmax_s16x2_relu(a, b, c);   // max(a + b, c, 0)
    }
    static __device__ __forceinline__ uint32_t pack(int lo, int hi) {
        return (uint32_t)(lo & 0xFFFF) | ((uint32_t)(hi & 0xFFFF) << 16);
    }
    static __device__ __forceinline__ uint32_t pack_score(int lo, int hi) { return pack(lo, hi); }
    static __device__ __forceinline__ int extract(uint32_t v, int h) {
        return (int)(int16_t)(h ? (v >> 16) : (v & 0xFFFF));
    }
    // max(a + b, 0): `zero` is an opaque register holding 0 (a literal makes ptxas emit a PRMT per use)
    static __device__ __forceinline__ uint32_t add_relu(uint32_t a, uint32_t b, uint32_t zero) {
        return __viaddmax_s16x2_relu(a, b, zero);
    }
    static __device__ __forceinline__ uint32_t add(uint32_t a, uint32_t b) { return __vadd2(a, b); }
    static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return __vmaxs2(a, b); }
    static __device__ __forceinline__ uint32_t addmax(uint32_t a, uint32_t b, uint32_t c) {
        return __viaddmax_s16x2(a, b, c);   // max(a + b, c)
    }
    // values above `lim` restart at 0 (W-bit wrap-then-clamp, SW_ProcessingElement_v1.0.v:287-288)
    static __device__ __forceinline__ uint32_t wrap_clamp(uint32_t m, uint32_t lim) {
        return m & ~__vcmpgts2(m, lim);
    }
};

// Plain signed 32-bit arithmetic, one subject per register: the band-pipelined 32-bit scorer of
// the overflow list (sw_wave.cuh, sw_wave32_kernel).  Same DPX instruction per operation.
struct ArithS32 {
    static constexpr int kPad = -(1 << 28);
    static __device__ __forceinline__ uint32_t addmax_relu(uint32_t a, uint32_t b, uint32_t c) {
        return (uint32_t)__viaddmax_s32_relu((int)a, (int)b, (int)c);
    }
    static __device__ __forceinline__ uint32_t pack_score(int lo, int) { return (uint32_t)lo; }
    static __device__ __forceinline__ int extract(uint32_t v, int) { return (int)v; }
    static __device__ __forceinline__ uint32_t add_relu(uint32_t a, uint32_t b, uint32_t) { return (uint32_t)max((int)(a + b), 0); }
    static __device__ __forceinline__ uint32_t wrap_clamp(uint32_t m, uint32_t) { return m; }   // exact mode only
    static __device__ __forceinline__ uint32_t add(uint32_t a, uint32_t b) { return a + b; }
    static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return (uint32_t)max((int)a, (int)b); }
    static __device__ __forceinline__ uint32_t addmax(uint32_t a, uint32_t b, uint32_t c) {
        return (uint32_t)__viaddmax_s32((int)a, (int)b, (int)c);
    }
};

// Pass-boundary scratch accesses, tagged evict_last so that the scratch lines, which are rewritten
// every pass, stay resident in L2 instead of being written back to HBM between passes.  A slot is
// written and read by the same warp only (lane G-1 / lane 0), so L1 is coherent for it: loads are
// cached in L1 and an explicit L1 prefetch runs a few steps ahead -- the load itself then costs an
// L1 hit wherever ptxas schedules it inside the step (placed late, an L2-latency load showed up
// as long-scoreboard stalls: ALU pipe 89 % -> 84 %).
__device__ __forceinline__ uint64_t l2_evict_last_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint2 bnd_load(const uint2 *p, uint64_t pol)
{
    uint2 v;
    asm volatile("ld.global.ca.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
}
// Progress word of a pass-split chain (gpu scope): the acquire load also drops the SM's L1 lines, so the
// L1-cached boundary loads that follow it see the rows another SM released.
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned *p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void prefetch_l1(const void *p)
{
    asm volatile("prefetch.global.L1 [%0];" :: "l"(p));
}
__device__ __forceinline__ void bnd_store(uint2 *p, uint2 v, uint64_t pol)
{
    asm volatile("st.global.cg.L2::cache_hint.v2.u32 [%0], {%1, %2}, %3;" :: "l"(p), "r"(v.x), "r"(v.y), "l"(pol) : "memory");
}

struct StripArgs {
    const uint32_t *tp;
    const uint64_t *tile_woff;
    const uint32_t *pair_len;
    const uint32_t *pair_subj;
    uint32_t npairs;
    uint32_t npb;              // pair blocks = ceil(npairs / pairs-per-block)
    uint32_t superblock;       // pair blocks per super-block of the work order (0 = npb / 8)
    const uint8_t *qpacked;
    const uint32_t *qoff;
    const uint32_t *qlen;
    const int *qidx;           // queries of this launch: qidx[0 .. nql), or null = q0 .. q0 + nql - 1
    int q0, nql;
    void *out;                 // int32 / int16 [q][out_stride] (null in top-k mode)
    size_t out_stride;
    int out_mode;              // SW_OUT_*
    uint2 *bnd;
    uint32_t bnd_cols;
    unsigned *counter;         // work queue; null = static schedule (item = blockIdx.x + k * gridDim.x)
    int sticky;                // > 0: counter[0 .. nql) = one work queue per query of the launch (see "work order");
                               // the value = how many pair blocks the queues may drift apart
    int chunk_passes;          // passes whose query profile is resident in shared memory at once
    // Pass split (nparts > 1, multi-pass queries with few work items, see "pass split"): an item covers
    // part_passes passes of its (pair block, query) chain; the boundary row and the running maximum of a
    // chain live in per-CHAIN scratch between parts, part_done[chain] counts the finished parts.
    int nparts, part_passes;
    unsigned *part_done;       // [nql * npb], zeroed before the launch
    uint32_t *part_best;       // [nql * npb * block threads]
    int match, mismatch, goe, ge, limit;
    uint32_t goe2, ge2;        // goe / ge packed in both 16-bit lanes (host side: uniform operands)
    int ovf_limit;             // 32767 - match - 1: a larger final maximum means a possible wrap
    uint32_t zero;             // always 0, but opaque to the compiler
    // DIRECT instances: column codes are formed on the fly from the uploaded 2-bit records
    const uint8_t *raw;
    const uint64_t *off;
    // DIRECT: one 32-byte descriptor per pair {n_lo, n_hi, subj_lo, subj_hi | off_lo, off_hi, 0, 0}: one
    // load gives a pair's lengths, subjects and record offsets (the latency path pays a memory round
    // trip per DEPENDENT load, so the chain pair table -> offsets -> bases is cut to two links)
    const uint4 *pair_desc;
    // pairs whose score may have left the 16-bit range: (query, subject) appended here
    unsigned *ovf_count;
    uint2 *ovf_list;
    unsigned ovf_cap;
    // fused per-query top-k (SW_OUT_TOPK): keys[(blockIdx.x * topk_nq + q) * topk_k + i], descending
    unsigned long long *topk_keys;
    int topk_k, topk_nq;
    unsigned *dev_err;         // device-side error word (bounds-check builds)
    // completion flag of the latency path: the last block to finish writes done_seq to *done_flag
    // (mapped host memory), which the host polls -- no event, no stream query on the critical path
    unsigned *done_count;
    unsigned *done_flag;
    unsigned done_seq;
    // hit list (SW_OUT_HITS): hits[i] = row << hits_shift | subject, hits_score[i] = score, for every pair with
    // score >= min_score that is not on the overflow list; hits_count counts past hits_cap, stores stop there
    unsigned long long *hits;  // null = append nothing (autotune's sample launches)
    int32_t *hits_score;
    unsigned long long *hits_count;   // 64-bit: a shard of 10 M subjects x 1 000 rows has 10^10 pairs
    unsigned hits_cap;
    int min_score, hits_shift;
    // per-subject best (SW_OUT_SBEST, sbest_update): sbest_key[subject] = score << 32 | (0xFFFFFFFF - row) of the
    // best row so far, sbest_second[subject] = the best score of the other rows, for every pair not on the overflow list
    unsigned long long *sbest_key;   // null = update nothing (autotune's sample launches)
    int *sbest_second;               // null = one row only (no runner-up)
#ifdef SW_BOUNDS_CHECK
    unsigned long long tp_words, bnd_elems, out_elems;
#endif
};

#ifdef SW_BOUNDS_CHECK
#define SW_CHECK(cond, bit, args) do { if (!(cond)) { if ((args).dev_err) atomicOr((args).dev_err, (bit)); } } while (0)
#define SW_CHECKED(cond, bit, args) ((cond) ? true : (((args).dev_err ? (void)atomicOr((args).dev_err, (bit)) : (void)0), false))
#else
#define SW_CHECK(cond, bit, args) do { } while (0)
#define SW_CHECKED(cond, bit, args) (true)
#endif

// Hit-list slots of up to two entries per lane (take0, take1): one atomicAdd per warp on *count.  Every
// lane of the warp calls it.  Returns false when the warp has nothing to append.
__device__ __forceinline__ bool hits_slots(unsigned long long *count, bool take0, bool take1, unsigned long long &p0,
                                           unsigned long long &p1)
{
    const unsigned b0 = __ballot_sync(0xFFFFFFFFu, take0), b1 = __ballot_sync(0xFFFFFFFFu, take1);
    if ((b0 | b1) == 0u) return false;
    const unsigned lane = threadIdx.x & 31u, below = (1u << lane) - 1u, n0 = __popc(b0);
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(count, (unsigned long long)(n0 + __popc(b1)));
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    p0 = base + __popc(b0 & below);
    p1 = base + n0 + __popc(b1 & below);
    return true;
}

// Per-subject best: the update of one (subject, row) pair.  Keys are score << 32 | (0xFFFFFFFF - row), so the
// largest key is the best score at its lowest row (key 0 = a phantom row scoring 0).  A key that held the maximum
// and is displaced reaches `second` through the update that displaced it; any other key reaches it directly.  So
// `second` ends as the best score of every row but the final best one -- provided each pair arrives exactly once
// (a pair that arrives twice would set second = best).  second == null: one row, no runner-up.
__device__ __forceinline__ void sbest_update(unsigned long long *key, int *second, uint32_t s, int row, int score)
{
    const unsigned long long k = ((unsigned long long)(uint32_t)score << 32) | (0xFFFFFFFFu - (uint32_t)row);
    const unsigned long long old = atomicMax(key + s, k);
    if (second) atomicMax(second + s, k > old ? (int)(old >> 32) : score);
}

// Column codes: 0..15 = t_lo | t_hi << 2 (both members have a base in this column);
// 16..19 = 16 + t_lo (the shorter member, always the high lane, has ended: its lane sees PAD);
// 20 = no column at all (pipeline fill / drain, past the end of the pair).
constexpr int kHiEndedCode = 16;
constexpr int kPadCode = 20;
constexpr int kCodesPerRow = 32;    // profile entries per row pair (codes 0..20 used): 256 bytes
constexpr int kMaxTopK = 32;
constexpr int kQueryBytes = 512;    // packed query bytes staged per profile chunk (2048 rows; host-checked)

// The four column codes of columns 4k .. 4k+3 of a pair: a / b = the packed byte k of the longer /
// shorter member (0 past its end), nlo >= nhi their lengths.  Used by build_tp_kernel (code stream
// in HBM) and by the DIRECT instances (codes formed on the fly).
__device__ __forceinline__ uint32_t make_code_word(uint32_t a, uint32_t b, uint32_t k, uint32_t nlo, uint32_t nhi)
{
    uint32_t w = 0;
#pragma unroll
    for (uint32_t c = 0; c < 4; ++c) {
        const uint32_t col = 4 * k + c;
        const uint32_t tlo = (a >> (2 * c)) & 3u, thi = (b >> (2 * c)) & 3u;
        const uint32_t code = col < nhi ? (tlo | (thi << 2)) : col < nlo ? (kHiEndedCode + tlo) : (uint32_t)kPadCode;
        w |= code << (8 * c);
    }
    return w;
}

// One column step of the S sub-strips of a lane, each sub-strip on its own column (sub-strip s
// is one column behind s-1): S independent dependency chains in one basic block, so a warp
// always has an instruction whose operands are ready (the PE array's pipelining, inside one
// thread).  H[s][r] / Gl[s][r] hold H and G of the previous column on entry and of this column
// on exit; hd_top = H(row0-1, c-1), g_top = G(row0-1, c); sv[s][k] = the substitution scores of
// rows 2k, 2k+1 of sub-strip s against this column's code (load_scores: one LDS.64 per row pair).
template <int RS, int S, int G, int CODES = kCodesPerRow>
__device__ __forceinline__ void load_scores(uint2 (&sv)[S][(RS + 1) / 2], const uint2 *prof_lane, const uint32_t (&code)[S])
{
    constexpr int RP = (RS + 1) / 2;
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const uint2 *prow = prof_lane + (s * RP * CODES + code[s]) * G;
#pragma unroll
        for (int k = 0; k < RP; ++k) sv[s][k] = prow[k * CODES * G];
    }
}

template <int RS, int S, int G, class AR, bool W12>
__device__ __forceinline__ void column_step_multi(uint32_t (&H)[S][RS], uint32_t (&Gl)[S][RS], uint32_t &best,
                                                  const uint32_t (&hd_top)[S], const uint32_t (&g_top)[S],
                                                  const uint2 (&sv)[S][(RS + 1) / 2], uint32_t goe2,
                                                  uint32_t ge2, uint32_t zero, uint32_t lim2)
{
    if constexpr (!W12) {
        // Clamped, goe-shifted form (exact, DESIGN.md section 2).  Every gap value is clamped at 0
        // (non-positive gap values can never reach H because M >= 0) and the register strip holds
        // K = H + goe instead of H.  With tg = K(r-1,c-1) + s  (= H_diag + s + goe):
        //     I = max(G_left, G_up)            >= 0                 VIMNMX
        //     G = max(I + ge, tg, 0)                                VIADDMNMX.RELU
        //     K = max(I + goe, tg)    (= max(I, H_diag + s) + goe)  VIADDMNMX
        // M = max(H_diag + s, 0) is never materialised (I >= 0 does the clamping) and both adds
        // of the gap path are fused: 3.5 ALU-pipe + 1 FMA-pipe instruction per cell pair.
        // tg of row r+1 is formed one row ahead from the still-old H[r], so H[r] is overwritten
        // in place.  The reported score is max K - goe.
        uint32_t gu[S], t_cur[S];
#pragma unroll
        for (int s = 0; s < S; ++s) {
            gu[s] = g_top[s];
            t_cur[s] = AR::add(hd_top[s], sv[s][0].x);
        }
#pragma unroll
        for (int r = 0; r < RS; ++r) {
#pragma unroll
            for (int s = 0; s < S; ++s) {
                uint32_t t_next = zero;
                if (r + 1 < RS) {
                    const uint32_t sc = ((r + 1) & 1) ? sv[s][(r + 1) >> 1].y : sv[s][(r + 1) >> 1].x;
                    t_next = AR::add(H[s][r], sc);
                }
                const uint32_t i_ = AR::max2(Gl[s][r], gu[s]);
                gu[s] = AR::addmax_relu(i_, ge2, t_cur[s]);
                Gl[s][r] = gu[s];
                H[s][r] = AR::addmax(i_, goe2, t_cur[s]);
                best = AR::max2(best, H[s][r]);
                t_cur[s] = t_next;
            }
        }
        return;
    }
    // W-bit faithful mode (score_width != 0): the explicit form of SW_ProcessingElement_v1.0.v with
    // the M overflow ("MSB clear => ZERO", :287-288) applied to every M.  M of row r+1 is formed one
    // row ahead, from the still-old H[r] (its diagonal), so that H[r] is overwritten in place.
    uint32_t gu[S], m_cur[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
        gu[s] = g_top[s];
        uint32_t m = AR::add_relu(hd_top[s], sv[s][0].x, zero);     // M(r,c) = relu(H(r-1,c-1) + s)
        if (W12) m = AR::wrap_clamp(m, lim2);
        m_cur[s] = m;
    }
#pragma unroll
    for (int r = 0; r < RS; ++r) {
#pragma unroll
        for (int s = 0; s < S; ++s) {
            uint32_t m_next = zero;
            if (r + 1 < RS) {
                const uint32_t sc = ((r + 1) & 1) ? sv[s][(r + 1) >> 1].y : sv[s][(r + 1) >> 1].x;
                m_next = AR::add_relu(H[s][r], sc, zero);
                if (W12) m_next = AR::wrap_clamp(m_next, lim2);
            }
            // the serial chain of a column is I -> I+ge -> G; the S chains interleave
            const uint32_t i_ = AR::max2(Gl[s][r], gu[s]);      // I = max(G_left, G_up)
            const uint32_t j_ = AR::add(i_, ge2);               // I + ge          (FMA-side pipe)
            gu[s] = AR::addmax(m_cur[s], goe2, j_);             // G = max(M + goe, I + ge)
            Gl[s][r] = gu[s];
            H[s][r] = AR::max2(m_cur[s], i_);                   // H = max(M, I)
            best = AR::max2(best, H[s][r]);                     // ptxas pairs these into 3-input max
            m_cur[s] = m_next;
        }
    }
}

// Fused per-query top-k (the bank's never-driven max / vld_max, ScoreBank_v2.v:42-43): every
// resident block keeps a private, sorted list of its K best keys per query in global memory
// (L2-resident: grid x queries x K x 8 bytes), so the epilogue needs no lock and no atomics on
// shared lists.  key = score << 32 | ~subject: the K largest keys are the K best scores, ties
// broken towards the lower subject index -- independent of the order in which items are processed.
// A merge kernel folds the per-block lists into one list per query afterwards.
// cand[0..ncand) in shared memory; executed by warp 0 of the block.
__device__ __forceinline__ void topk_insert_warp(unsigned long long *list, int K, const unsigned long long *cand, int ncand)
{
    const int lane = threadIdx.x & 31;
    unsigned long long key = (lane < K) ? __ldcg(list + lane) : 0ull;
    for (int j = 0; j < ncand; ++j) {
        const unsigned long long c = cand[j];
        const unsigned pos = __popc(__ballot_sync(0xFFFFFFFFu, lane < K && key > c));   // keys ahead of c
        const unsigned long long up = __shfl_up_sync(0xFFFFFFFFu, key, 1);
        if ((int)pos < K) {
            if (lane > (int)pos) key = up;
            else if (lane == (int)pos) key = c;
        }
    }
    if (lane < K) __stcg(list + lane, key);
}

// RS rows per sub-strip, S sub-strips per lane, G lanes per pair: R = RS*S rows per lane,
// P = R*G rows per pass.  Virtual PE v = lane_in_group*S + s works on column t - v at step t.
// A virtual PE that has no column at step t (pipeline fill / drain, shorter pair in the warp)
// works on the PAD column code whose profile entries are very negative: H keeps decaying values
// <= the best already recorded and G stays clamped / non-positive, which never reaches H
// (DESIGN.md section 2).  That keeps the loop body free of per-lane branches.
// CGOE / CGE != 0: gap penalties fixed at compile time.  ptxas then encodes them as immediates
// (VIADDMNMX.S16x2 R, R, 0xfffcfffc, R): two register operands instead of three per fused
// add-max, which removes register-bank conflicts on the ALU pipe (+6..13 % measured).  Compiled in
// for the reference's own penalty sets (ScoreBank_v1_tb.sv:16-19); any other set is specialised at
// run time (sw_jit.cu) or takes the run-time-operand instance.
// DIRECT: the column codes are formed on the fly from the uploaded 2-bit records instead of being
// read from the code stream -- no build_tp launch: the small-batch (latency) path.
template <int RS, int S, int G, class AR, bool W12, int BT, int MINB, int CGOE = 0, int CGE = 0, bool DIRECT = false,
          int U = SW_STEP_UNROLL, int FL = SW_FAST_LOOP>
__global__ void __launch_bounds__(BT, MINB) sw_strip_kernel(const StripArgs a)
{
    extern __shared__ uint2 s_prof[];
    __shared__ unsigned s_work, s_iter;
    __shared__ uint8_t s_qb[kQueryBytes];             // packed query bytes of the resident profile chunk
    __shared__ uint32_t s_codes[DIRECT ? BT / G : 1][DIRECT ? 256 : 1];   // DIRECT: staged code words per pair slot
    constexpr int R = RS * S;
    constexpr int P = R * G;
    constexpr int RP = (RS + 1) / 2;
    constexpr int VPE = G * S;                       // virtual PEs per pair
    constexpr int PASS_ENTRIES = VPE * RP * kCodesPerRow;
    constexpr int PPB = BT / G;
    constexpr unsigned FULL = 0xFFFFFFFFu;
    static_assert(U % 4 == 0, "the step loop consumes 4-column code words");
    // EARLY (wide systolic groups): the column codes travel from lane to lane ONE STEP AHEAD of the
    // (H, G) values, so the profile load of step t+1 is issued during step t and the per-step
    // dependency chain is shuffle -> add -> max chain instead of shuffle -> LDS -> add -> max chain.
    // These variants are latency-bound (one warp = one pair), so that is what sets their speed.
    constexpr bool EARLY = (G >= 8);
    constexpr int kDirectWords = 256;                // DIRECT: code words staged per pair slot (1024 columns)
    // DIRECT instances with a short pass (P < 512 rows) are only used for queries of at most P rows
    // (the host checks): no pass-boundary code at all in their step loop
    constexpr bool MULTIPASS = !(DIRECT && P < 512);
    // (A column-blocked schedule for these instances -- four columns per trip and one shuffle round
    // trip per block -- was measured and dropped: 25.0 vs 23.0 us for config 2, 19.8 vs 16.4 us for
    // one pair: the extra fill / drain costs more than the shuffles it saves.)
    static_assert(sizeof(s_codes[0]) == (DIRECT ? kDirectWords : 1) * sizeof(uint32_t), "s_codes row = kDirectWords");

    const int lane = threadIdx.x & 31;
    const int gl = (G == 1) ? 0 : (lane & (G - 1));
    const int pslot = threadIdx.x / G;
    const uint32_t zero = a.zero;
    const uint32_t goe2 = CGOE ? ((uint32_t)(CGOE & 0xFFFF) * 0x10001u) : a.goe2;
    const uint32_t ge2 = CGOE ? ((uint32_t)(CGE & 0xFFFF) * 0x10001u) : a.ge2;
    // boundary gap value G(0,j) = G(i,0): max(goe, ge) <= 0, or its clamp 0 in the clamped form
    const int gbv = !W12 ? 0 : (a.goe > a.ge ? a.goe : a.ge);
    const uint32_t gb2 = AR::pack(gbv, gbv);
    const uint32_t lim2 = AR::pack(a.limit, a.limit);
    // value of "H = 0" in the strip's representation (K = H + goe in the clamped form)
    const uint32_t h0 = !W12 ? goe2 : zero;
    uint2 *bnd = a.bnd + (size_t)blockIdx.x * a.bnd_cols * PPB + pslot;     // (pass split: per chain, set per item)
    const uint64_t bnd_pol = l2_evict_last_policy();

    // work item -> (pair block, query).  Pairs are sorted by ascending length: the longest blocks go
    // first so that the tail is made of short items.  Order: super-blocks of B pair blocks, longest
    // first; inside a super-block query-major.  With B >> grid (large databases) consecutive items
    // of a thread block share the query and the profile in shared memory is reused, and the host
    // sizes B so that a super-block's code stream stays in L2 while its queries pass over it; with B
    // small the order degenerates to longest-first over everything, which is what short launches
    // need for their tail.  (Decoded twice per item -- before the column loops and again in the epilogue --
    // so that nothing but s_work has to stay live across the hot loop.)
    // Sticky order (a.sticky, launches with several queries): one queue of pair blocks PER QUERY, every
    // thread block stays with "its" query (blockIdx.x mod queries) until that queue is empty and then
    // moves on to the next one.  The profile in shared memory is rebuilt about once per launch instead
    // of every few items, and the queries sweep the pair blocks side by side, so a code-stream line is
    // read from HBM once and from L2 by the other queries (DRAM traffic of a config-3 launch: 19.2 GB in
    // super-block order, 3.7 GB in this one -- profiles/r02_traffic.json; algorithmic 1.3 GB; and
    // 9 000 vs 8 970 GCUPS).  work = query slot * npb + block.
    // Pass split (a.nparts > 1): the passes of a long query are cut into parts of a.part_passes passes and
    // an item is (part, pair block, query), handed out PART-MAJOR: work = part * items_per_part + the index
    // above.  Items get shorter in time without losing lanes, so a launch of few long items (200 k x 1 kb
    // subjects against one 10 kb query: 781 items on 296 resident blocks = 2.64 rounds, a third of the GPU
    // idle in the last one) ends on a short tail.  Part p of a chain starts from the boundary row and the
    // running maximum that part p - 1 left in the chain's scratch; it waits for part_done[chain] >= p
    // (acquire; the producer releases after a block barrier).  The item it waits for has a smaller work
    // index, so it was claimed earlier by a block that is resident and running: no deadlock (and a
    // watchdog raises SW_DEVERR_SPIN instead of hanging).  ScoreBank_v2.v:78-139 keeps its modules busy
    // the same way: a module is handed the next target as soon as it is free, whatever that target is.
    const unsigned items_per_part = a.npb * (unsigned)a.nql;
    auto decode = [&](unsigned work, unsigned &pair, int &q, unsigned &chain, int &part) {
        part = 0;
        if (a.nparts > 1) { part = (int)(work / items_per_part); work -= (unsigned)part * items_per_part; }
        if (a.sticky) {
            const unsigned qk = work / a.npb;
            const unsigned pb = a.npb - 1u - (work - qk * a.npb);      // longest pair blocks first
            q = a.qidx ? a.qidx[qk] : a.q0 + (int)qk;
            pair = pb * PPB + pslot;
            chain = qk * a.npb + pb;
            return;
        }
        const unsigned nql = (unsigned)a.nql;
        const unsigned B = a.superblock ? a.superblock : max(1u, a.npb >> 3);
        const unsigned sb = work / (nql * B);
        const unsigned rem = work - sb * nql * B;
        const unsigned bcur = min(B, a.npb - sb * B);
        const unsigned pb = a.npb - 1u - (sb * B + rem % bcur);
        const int qk = (int)(rem / bcur);
        q = a.qidx ? a.qidx[qk] : a.q0 + qk;
        pair = pb * PPB + pslot;
        chain = (unsigned)qk * a.npb + pb;
    };

    int prof_q = -1, prof_pass = -1;     // which (query, first pass) the shared-memory profile holds
    if (threadIdx.x == 0) s_iter = a.sticky ? blockIdx.x % (unsigned)a.nql : 0u;     // sticky: the block's query slot
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) {
            // work queue (atomic counter) or, for small launches, a static schedule
            if (a.sticky) {
                unsigned qk = s_iter, w = 0xFFFFFFFFu;
                // bounded drift: the queries' sweeps over the code stream stay within a.sticky pair blocks
                // of each other (the window the L2 keeps) -- a block whose queue is further ahead than
                // that of the slowest queue joins that one (one profile rebuild)
                if (a.nql <= 32) {
                    const unsigned mine = *(volatile const unsigned *)(a.counter + qk);
                    unsigned lo = mine, lo_k = qk;
                    for (int k = 0; k < a.nql; ++k) {
                        const unsigned c = *(volatile const unsigned *)(a.counter + k);
                        if (c < lo) { lo = c; lo_k = (unsigned)k; }
                    }
                    if (mine > lo + (unsigned)a.sticky) qk = lo_k;
                }
                for (int tries = 0; tries < a.nql; ++tries) {
                    const unsigned pb = atomicAdd(a.counter + qk, 1u);
                    if (pb < a.npb) { w = qk * a.npb + pb; break; }
                    qk = (qk + 1u == (unsigned)a.nql) ? 0u : qk + 1u;
                }
                s_iter = qk;
                s_work = w;
            }
            else if (a.counter) s_work = atomicAdd(a.counter, 1u);
            else { s_work = blockIdx.x + s_iter * gridDim.x; s_iter++; }
        }
        __syncthreads();
        if (s_work >= items_per_part * (unsigned)max(a.nparts, 1)) break;
        unsigned pair, chain;
        int q, part;
        decode(s_work, pair, q, chain, part);
        if (MULTIPASS && a.nparts > 1) {
            bnd = a.bnd + (size_t)chain * a.bnd_cols * PPB + pslot;
            if (part > 0) {
                if (threadIdx.x == 0) {
                    unsigned spins = 0;
                    while (ld_acquire_gpu(a.part_done + chain) < (unsigned)part) {
                        __nanosleep(128);
                        if (++spins > (1u << 26)) {                    // watchdog: never hang the GPU
                            if (a.dev_err) atomicOr(a.dev_err, SW_DEVERR_SPIN);
                            break;
                        }
                    }
                }
                __syncthreads();      // the acquire above orders the whole block behind the producer's release
            }
        }

        const bool valid = pair < a.npairs;
        int ncols_v = 0;                                                   // longer member (low lane)
        const uint32_t *tpp = a.tp;
        const uint8_t *rlo = nullptr, *rhi = nullptr;
        uint32_t nhi = 0;
        // the query's length / offset are requested now, so that their round trip overlaps the pair's
        const int m = (int)a.qlen[q];
        const uint8_t *qp = a.qpacked + a.qoff[q];
        if (valid) {
            if constexpr (DIRECT) {
                const uint4 d0 = __ldg(a.pair_desc + 2 * pair), d1 = __ldg(a.pair_desc + 2 * pair + 1);
                ncols_v = (int)d0.x;
                nhi = d0.y;
                rlo = a.raw + d1.x;
                if (d0.w != SW_NO_SUBJECT) rhi = a.raw + d1.y;
            } else {
                ncols_v = (int)a.pair_len[2 * pair];
                tpp += a.tile_woff[pair >> 5] + (pair & 31);
            }
        }
        const int ncols = ncols_v;
        // single-pass DIRECT instances: this thread's byte of the packed query, requested before the
        // code staging below waits for the subject bytes (the profile build stores it to shared memory)
        uint32_t my_qbyte = 0;
        if constexpr (!MULTIPASS) {
            if ((int)threadIdx.x < ((m + 3) >> 2)) my_qbyte = qp[threadIdx.x];
        }
        // DIRECT: the lanes of the group form the pair's code words in parallel, once, into shared
        // memory (the host sends only subjects of up to 4 * kDirectWords bases down this path)
        if constexpr (DIRECT) {
            for (int k = gl; 4 * k < ncols && k < kDirectWords; k += G) {
                const uint32_t ba = (uint32_t)__ldg(rlo + k);
                const uint32_t bb = (rhi != nullptr && 4 * (uint32_t)k < nhi) ? (uint32_t)__ldg(rhi + k) : 0u;
                s_codes[pslot][k] = make_code_word(ba, bb, (uint32_t)k, (uint32_t)ncols, nhi);
            }
            __syncwarp();
        }
        // word k of the pair's column code stream (columns 4k .. 4k+3)
        auto code_word = [&](int k) -> uint32_t {
            if constexpr (DIRECT) {
                return s_codes[pslot][k & (kDirectWords - 1)];
            } else {
                SW_CHECK((unsigned long long)(tpp - a.tp) + (unsigned long long)k * 32 < a.tp_words, SW_DEVERR_TP, a);
                return __ldg(tpp + k * 32);
            }
        };
        // rounded up: the step loop is unrolled (extra steps are PAD columns)
        const int nsteps = (__reduce_max_sync(FULL, ncols) + (VPE - 1) + U - 1) / U * U;
        const int ncols_min = __reduce_min_sync(FULL, ncols);     // shortest pair of the warp (interior trips)

        uint32_t best = h0;
        {
            const int npass = (m + P - 1) / P;
            int pass_lo = 0, pass_hi = npass;
            if (MULTIPASS && a.nparts > 1) {
                pass_lo = min(npass, part * a.part_passes);
                pass_hi = (part + 1 == a.nparts) ? npass : min(npass, pass_lo + a.part_passes);
                if (part > 0) best = __ldcg(a.part_best + (size_t)chain * BT + threadIdx.x);
            }

            for (int pass = pass_lo; pass < pass_hi; ++pass) {
                const int pass_in_chunk = pass % a.chunk_passes;
                if (pass_in_chunk == 0 && (prof_q != q || prof_pass != pass)) {
                    prof_q = q;
                    prof_pass = pass;
                    // (re)build the profile chunk: entry (vpe, row pair, code) = packed scores of
                    // rows 2k, 2k+1 of that virtual PE against column code = t_lo | t_hi << 2
                    __syncthreads();
                    const int npc = min(a.chunk_passes, npass - pass);
                    // the chunk's query bytes first (one coalesced load): the entry loop below would
                    // otherwise pay a global-memory round trip per entry, which is what a small
                    // (latency-bound) launch consists of
                    const int qb0 = (pass * P) >> 2;
                    const int qnb = ((min((pass + npc) * P, m) + 3) >> 2) - qb0;
                    if constexpr (!MULTIPASS) {
                        if ((int)threadIdx.x < qnb) s_qb[threadIdx.x] = (uint8_t)my_qbyte;     // P < 512: qnb <= BT
                    } else {
                        for (int i = threadIdx.x; i < qnb && i < kQueryBytes; i += BT) s_qb[i] = qp[qb0 + i];
                    }
                    __syncthreads();
                    for (int idx = threadIdx.x; idx < npc * PASS_ENTRIES; idx += BT) {
                        // layout: (((pass * S + s) * RP + rp) * 32 + code) * G + gl -- the G lanes of a
                        // group sit in consecutive 8-byte slots, so a warp-wide group reads 32 banks
                        const int lg = idx % G;
                        const int code = (idx / G) & (kCodesPerRow - 1);
                        if (code > kPadCode) continue;
                        const int rp = (idx / (G * kCodesPerRow)) % RP;
                        const int ss = (idx / (G * kCodesPerRow * RP)) % S;
                        const int pc = idx / PASS_ENTRIES;
                        const int vpe = lg * S + ss;
                        uint32_t e[2];
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const int rr = 2 * rp + k;
                            const int i = (pass + pc) * P + vpe * RS + rr;
                            int lo = AR::kPad, hi = AR::kPad;
                            if (rr < RS && i < m && code < kPadCode) {
                                const int qi = (s_qb[(i >> 2) - qb0] >> ((i & 3) * 2)) & 3;
                                lo = (qi == (code & 3)) ? a.match : a.mismatch;   // v1.0.v:119
                                if (code < kHiEndedCode) hi = (qi == (code >> 2)) ? a.match : a.mismatch;
                            }
                            e[k] = AR::pack_score(lo, hi);
                        }
                        s_prof[idx] = make_uint2(e[0], e[1]);
                    }
                    __syncthreads();
                }
                const uint2 *prof_lane = s_prof + (size_t)pass_in_chunk * PASS_ENTRIES + gl;
                const bool has_top = pass > 0;
                const bool has_bottom = pass + 1 < npass;

                uint32_t H[S][RS], Gl[S][RS];
#pragma unroll
                for (int s = 0; s < S; ++s)
#pragma unroll
                    for (int r = 0; r < RS; ++r) { H[s][r] = h0; Gl[s][r] = gb2; }

                uint32_t wcur = 0, wnext = 0;
                uint2 bcur = make_uint2(h0, gb2);            // (H, G) of the row above, column c
                if (gl == 0 && ncols > 0) {
                    wcur = code_word(0);
                    if (ncols > 4) wnext = code_word(1);
                    if (MULTIPASS && has_top) {
                        SW_CHECK((unsigned long long)(bnd - a.bnd) < a.bnd_elems, SW_DEVERR_BND, a);
                        bcur = bnd_load(bnd, bnd_pol);
                        for (int c = 1; c < 4 && c < ncols; ++c) prefetch_l1(bnd + (size_t)c * PPB);
                    }
                }
                // what each sub-strip hands to the next virtual PE (the next sub-strip, or for
                // s = S-1 the next lane): bottom H, bottom G and a column code -- the code it just
                // used, or in EARLY mode the code it uses in the CURRENT step (one step ahead of H, G)
                uint32_t pub_h[S], pub_g[S], pub_t[S], hd_top[S];
#pragma unroll
                for (int s = 0; s < S; ++s) { pub_h[s] = h0; pub_g[s] = gb2; pub_t[s] = kPadCode; hd_top[s] = h0; }
                uint2 sv[S][RP];                              // substitution scores of the current step
                if constexpr (EARLY) {
                    // step 0: the head PE is on column 0, every other virtual PE on PAD
                    if (gl == 0 && ncols > 0) pub_t[0] = wcur & 255u;
                    load_scores<RS, S, G>(sv, prof_lane, pub_t);
                }

                // One column step of every virtual PE of the lane.  INTERIOR trips (G = 1 only): every
                // lane of the warp has a column at each step of the trip, a code word two words ahead and
                // (t + 4 < ncols), so the head's predicates, selects and the divergent region around the
                // boundary loads disappear from the loop body (about 7 of 10 ALU-pipe bookkeeping
                // instructions per column; the general body handles the first trip and the last few).
                auto step = [&](auto interior_tag, const int t, const int uu) {
                    constexpr bool INTERIOR = decltype(interior_tag)::value;
                    const int u = uu & 3;                 // column inside the current 4-column code word
                    // in_t: the code of THIS step (of the NEXT step in EARLY mode) of each virtual PE
                    uint32_t in_h[S], in_g[S], in_t[S];
                    if (G > 1) {
                        in_h[0] = __shfl_up_sync(FULL, pub_h[S - 1], 1, G);
                        in_g[0] = __shfl_up_sync(FULL, pub_g[S - 1], 1, G);
                        in_t[0] = __shfl_up_sync(FULL, pub_t[S - 1], 1, G);
                    }
                    if constexpr (EARLY) {
                        // head of the systolic group, written without divergent branches (these
                        // variants are latency-bound): every lane evaluates the head's expressions
                        // on its own (empty) word registers, the head lane keeps them
                        const bool head = gl == 0;
                        const uint32_t wsel = (u < 3) ? wcur : wnext;
                        const uint32_t lead_t = (t + 1 < ncols) ? ((wsel >> (8 * ((u + 1) & 3))) & 255u) : (uint32_t)kPadCode;
                        in_h[0] = head ? bcur.x : in_h[0];
                        in_g[0] = head ? bcur.y : in_g[0];
                        in_t[0] = head ? lead_t : in_t[0];
                        if (u == 3) {
                            wcur = wnext;
                            const int k = (t >> 2) + 2;
                            if (head && k * 4 < ncols) wnext = code_word(k);
                            if (!DIRECT && head && (k + 1) * 4 < ncols) prefetch_l1(tpp + (k + 1) * 32);
                        }
                        if constexpr (MULTIPASS) {
                            if (has_top && head) {
                                if (t + 1 < ncols) {
                                    SW_CHECK((unsigned long long)(bnd - a.bnd) + (unsigned long long)(t + 1) * PPB < a.bnd_elems, SW_DEVERR_BND, a);
                                    bcur = bnd_load(bnd + (size_t)(t + 1) * PPB, bnd_pol);
                                }
                                if (t + 4 < ncols) prefetch_l1(bnd + (size_t)(t + 4) * PPB);
                            }
                        }
                    } else if constexpr (INTERIOR) {
                        in_h[0] = bcur.x;
                        in_g[0] = bcur.y;
                        in_t[0] = (wcur >> (8 * u)) & 255u;
                        if (u == 3) {
                            wcur = wnext;
                            const int k = (t >> 2) + 2;
                            wnext = code_word(k);
                            if (!DIRECT && !(FL & 2)) prefetch_l1(tpp + (k + 1) * 32);
                        }
                        if (has_top) {
                            SW_CHECK((unsigned long long)(bnd - a.bnd) + (unsigned long long)(t + 1) * PPB < a.bnd_elems, SW_DEVERR_BND, a);
                            bcur = bnd_load(bnd + (size_t)(t + 1) * PPB, bnd_pol);
                            if (!(FL & 4)) prefetch_l1(bnd + (size_t)(t + 4) * PPB);
                        }
                    } else if (G == 1 || gl == 0) {
                        // head of the systolic group: column t comes from the code stream, the row
                        // above from the previous pass (or the zero boundary)
                        const bool on = t < ncols;
                        in_h[0] = bcur.x;
                        in_g[0] = bcur.y;
                        // t2 % 4 == 0: columns t2 + 4j .. t2 + 4j + 3 are the four bytes of one code word
                        in_t[0] = on ? ((wcur >> (8 * u)) & 255u) : (uint32_t)kPadCode;
                        if (on) {
                            if (u == 3) {
                                wcur = wnext;
                                const int k = (t >> 2) + 2;
                                if (k * 4 < ncols) wnext = code_word(k);
                                // the word after that goes to L1 now, so the load above stays
                                // short even if ptxas sinks it towards its use to save a register
                                if (!DIRECT && (k + 1) * 4 < ncols) prefetch_l1(tpp + (k + 1) * 32);
                            }
                            if (has_top) {
                                if (t + 1 < ncols) {
                                    SW_CHECK((unsigned long long)(bnd - a.bnd) + (unsigned long long)(t + 1) * PPB < a.bnd_elems, SW_DEVERR_BND, a);
                                    bcur = bnd_load(bnd + (size_t)(t + 1) * PPB, bnd_pol);
                                }
                                if (t + 4 < ncols) prefetch_l1(bnd + (size_t)(t + 4) * PPB);
                            }
                        }
                    }
#pragma unroll
                    for (int s = 1; s < S; ++s) { in_h[s] = pub_h[s - 1]; in_g[s] = pub_g[s - 1]; in_t[s] = pub_t[s - 1]; }
#pragma unroll
                    for (int s = 0; s < S; ++s) SW_CHECK(in_t[s] <= (uint32_t)kPadCode, SW_DEVERR_PROF, a);

                    if constexpr (EARLY) {
                        // scores of step t + 1 are requested now and consumed one step later
                        uint2 sv_next[S][RP];
                        load_scores<RS, S, G>(sv_next, prof_lane, in_t);
                        column_step_multi<RS, S, G, AR, W12>(H, Gl, best, hd_top, in_g, sv, goe2, ge2, zero, lim2);
#pragma unroll
                        for (int s = 0; s < S; ++s)
#pragma unroll
                            for (int k = 0; k < RP; ++k) sv[s][k] = sv_next[s][k];
                    } else {
                        load_scores<RS, S, G>(sv, prof_lane, in_t);
                        column_step_multi<RS, S, G, AR, W12>(H, Gl, best, hd_top, in_g, sv, goe2, ge2, zero, lim2);
                    }
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        hd_top[s] = in_h[s];
                        pub_h[s] = H[s][RS - 1]; pub_g[s] = Gl[s][RS - 1]; pub_t[s] = in_t[s];
                    }
                    if (MULTIPASS && has_bottom && gl == G - 1) {
                        const int cl = t - (VPE - 1);          // column the last virtual PE just finished
                        // (an interior trip that starts at column 0 -- FL bit 3 -- skips the stores of the fill steps)
                        if (INTERIOR ? (!(FL & 8) || uu >= VPE - 1 || t > uu) : (cl >= 0 && cl < ncols)) {
                            SW_CHECK((unsigned long long)(bnd - a.bnd) + (unsigned long long)cl * PPB < a.bnd_elems, SW_DEVERR_BND, a);
                            bnd_store(bnd + (size_t)cl * PPB, make_uint2(pub_h[S - 1], pub_g[S - 1]), bnd_pol);
                        }
                    }
                };
                // interior trips: t2 in [t_int0, t_int).  The last column touched ahead of a trip is
                // t2 + U + 8 (L1 prefetch of the code stream), t2 + U + 4 without that prefetch (next
                // code word); the first trip holds the pipeline fill (no boundary store before column 0)
                // and is interior only with FL bit 3.  FL bit 4: the general trips run one column per
                // loop trip (small code: both loop bodies stay in the instruction cache).
                constexpr bool kInt = (FL & 1) && G == 1 && !EARLY && MULTIPASS;
                constexpr int kAhead = (FL & 8) ? ((FL & 2) ? 5 : 9) : 9;
                const int t_int0 = (FL & 8) ? 0 : U;
                const int t_int = kInt ? ((ncols_min - kAhead) / U * U) : 0;
                static_assert(!kInt || U >= S - 1, "interior trips start behind the pipeline fill");
#pragma unroll 1
                for (int t2 = 0; t2 < nsteps;) {
                    if (kInt && t2 >= t_int0 && t2 < t_int) {
#pragma unroll 1
                        do {
#pragma unroll
                            for (int uu = 0; uu < U; ++uu) step(BoolTag<true>{}, t2 + uu, uu);
                            t2 += U;
                        } while (t2 < t_int);
                    } else if constexpr (kInt && (FL & 16)) {
#pragma unroll 1
                        for (int uu = 0; uu < U; ++uu) step(BoolTag<false>{}, t2 + uu, uu);
                        t2 += U;
                    } else {
#pragma unroll
                        for (int uu = 0; uu < U; ++uu) step(BoolTag<false>{}, t2 + uu, uu);
                        t2 += U;
                    }
                }
                if (has_bottom) __syncwarp();   // bottom row written by lane G-1, read by lane 0
            }
        }

        unsigned epair, echain;          // (decoded again: nothing but s_work stays live across the hot loop)
        int eq, epart;
        decode(s_work, epair, eq, echain, epart);
        if (MULTIPASS && a.nparts > 1 && epart + 1 < a.nparts) {
            // pass split, not the last part: park the running maximum, publish the part (the boundary row
            // went to the chain's scratch in the step loop) and take the next item
            __stcg(a.part_best + (size_t)echain * BT + threadIdx.x, best);
            __syncthreads();
            if (threadIdx.x == 0) st_release_gpu(a.part_done + echain, (unsigned)epart + 1u);
            continue;
        }
#pragma unroll
        for (int o = G / 2; o >= 1; o >>= 1) best = AR::max2(best, __shfl_xor_sync(FULL, best, o));
        // While every value so far is <= 32767 - match the next cell cannot wrap, and the running
        // maximum is monotone: a final best above that threshold is the only way a 16-bit overflow
        // can have happened.  Such pairs get a sentinel, are appended to the overflow list and are
        // recomputed in 32 bit (fix32_list_kernel).
        const int shift = !W12 ? a.goe : 0;
        const bool owner = gl == 0 && epair < a.npairs;
        uint32_t subj_lo = SW_NO_SUBJECT, subj_hi = SW_NO_SUBJECT;
        if (owner) {
            if constexpr (DIRECT) { const uint4 d0 = __ldg(a.pair_desc + 2 * epair); subj_lo = d0.z; subj_hi = d0.w; }
            else { subj_lo = a.pair_subj[2 * epair]; subj_hi = a.pair_subj[2 * epair + 1]; }
        }
        int sc0 = AR::extract(best, 0) , sc1 = AR::extract(best, 1);
        const bool ov0 = !W12 && sc0 > a.ovf_limit, ov1 = !W12 && sc1 > a.ovf_limit;
        sc0 -= shift; sc1 -= shift;
        const bool has1 = owner && subj_hi != SW_NO_SUBJECT;
        if (owner && (ov0 || (has1 && ov1)) && a.ovf_list) {
            if (ov0) { const unsigned p = atomicAdd(a.ovf_count, 1u); if (p < a.ovf_cap) a.ovf_list[p] = make_uint2((unsigned)eq, subj_lo); }
            if (has1 && ov1) { const unsigned p = atomicAdd(a.ovf_count, 1u); if (p < a.ovf_cap) a.ovf_list[p] = make_uint2((unsigned)eq, subj_hi); }
        }
        if (DIRECT || a.out_mode == SW_OUT_I32) {            // (the latency path delivers int32 matrices only)
            if (owner) {
                int32_t *orow = (int32_t *)a.out + (size_t)eq * a.out_stride;
                SW_CHECK((unsigned long long)eq * a.out_stride + subj_lo < a.out_elems, SW_DEVERR_OUT, a);
                orow[subj_lo] = ov0 ? SW_OVERFLOW_SENTINEL : sc0;
                if (has1) orow[subj_hi] = ov1 ? SW_OVERFLOW_SENTINEL : sc1;
            }
        } else if (a.out_mode == SW_OUT_I16) {
            if (owner) {
                int16_t *orow = (int16_t *)a.out + (size_t)eq * a.out_stride;
                SW_CHECK((unsigned long long)eq * a.out_stride + subj_lo < a.out_elems, SW_DEVERR_OUT, a);
                orow[subj_lo] = (int16_t)(ov0 ? SW_OVERFLOW_SENTINEL : sc0);
                if (has1) orow[subj_hi] = (int16_t)(ov1 ? SW_OVERFLOW_SENTINEL : sc1);
            }
        } else if (a.out_mode == SW_OUT_HITS) {
            // every thread of the block is here (the item loop is block-uniform); flagged pairs reach the
            // list from their exact score (hits_ovf_kernel), never from here
            unsigned long long p0 = 0, p1 = 0;
            const bool t0 = owner && !ov0 && sc0 >= a.min_score, t1 = has1 && !ov1 && sc1 >= a.min_score;
            if (a.hits && hits_slots(a.hits_count, t0, t1, p0, p1)) {
                const unsigned long long row = (unsigned long long)(unsigned)eq << a.hits_shift;
                if (t0 && p0 < a.hits_cap) {
                    SW_CHECK(p0 < a.out_elems, SW_DEVERR_OUT, a);
                    a.hits[p0] = row | subj_lo; a.hits_score[p0] = sc0;
                }
                if (t1 && p1 < a.hits_cap) {
                    SW_CHECK(p1 < a.out_elems, SW_DEVERR_OUT, a);
                    a.hits[p1] = row | subj_hi; a.hits_score[p1] = sc1;
                }
            }
        } else if (a.out_mode == SW_OUT_SBEST) {
            // flagged pairs are updated from their exact score (sbest_ovf_kernel), never from here; pass-split
            // parts other than the last left the item above, so each (subject, row) arrives once
            if (owner && a.sbest_key) {
                if (!ov0) {
                    SW_CHECK(subj_lo < a.out_elems, SW_DEVERR_OUT, a);
                    sbest_update(a.sbest_key, a.sbest_second, subj_lo, eq, sc0);
                }
                if (has1 && !ov1) {
                    SW_CHECK(subj_hi < a.out_elems, SW_DEVERR_OUT, a);
                    sbest_update(a.sbest_key, a.sbest_second, subj_hi, eq, sc1);
                }
            }
        } else {
            // fused top-k: candidates = keys above the block's current K-th key for this query
            __shared__ unsigned long long s_cand[2 * BT];
            __shared__ int s_ncand;
            const int K = a.topk_k;
            unsigned long long *list = a.topk_keys + ((size_t)blockIdx.x * a.topk_nq + eq) * K;
            const unsigned long long thr = __ldcg(list + K - 1);
            const unsigned long long k0 = (owner && !ov0) ? (((unsigned long long)(uint32_t)sc0 << 32) | (uint32_t)(~subj_lo)) : 0ull;
            const unsigned long long k1 = (has1 && !ov1) ? (((unsigned long long)(uint32_t)sc1 << 32) | (uint32_t)(~subj_hi)) : 0ull;
            if (threadIdx.x == 0) s_ncand = 0;
            const int any = __syncthreads_or((k0 > thr) | (k1 > thr));
            if (any) {
                if (k0 > thr) s_cand[atomicAdd(&s_ncand, 1)] = k0;
                if (k1 > thr) s_cand[atomicAdd(&s_ncand, 1)] = k1;
                __syncthreads();
                if (threadIdx.x < 32) topk_insert_warp(list, K, s_cand, s_ncand);
            }
        }
    }
    if (a.done_flag) {
        // every thread's result stores (mapped host memory) are ordered before the flag: block
        // barrier, then a system-scope fence by the thread that counts the block as finished
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();
            if (gridDim.x == 1) {
                *(volatile unsigned *)a.done_flag = a.done_seq;      // one block: its own fence is enough
            } else if (atomicAdd(a.done_count, 1u) == gridDim.x - 1) {
                *a.done_count = 0;
                __threadfence_system();
                *(volatile unsigned *)a.done_flag = a.done_seq;
            }
        }
    }
}

}  // namespace swk

#endif  /* SW_STRIP_CUH_ */
