/*
 * sw_locate.cu -- begin and end coordinates of the best local alignment of selected (query row, subject)
 * pairs (sw_locate_db), and its CIGAR (sw_align_db).  Locate runs two score-only passes per pair, with no
 * traceback storage (DESIGN.md section 5.7):
 *   forward  -- the recurrence over the whole pair, keeping the first cell in (column, row) order whose
 *               diagonal value M reaches the pair's maximum S: the end cell (q_end, s_end);
 *   reverse  -- the same recurrence over reverse(query[0:q_end]) x reverse(subject[0:s_end]), stopping at
 *               the first cell in (column, row) order whose M reaches S: (a, b) gives the begin.
 * Align adds a third pass of the same recurrence over the located rectangle query[q_begin:q_end] x
 * subject[s_begin:s_end] that stores 4 direction bits per cell, then walks back from the end (section 5.8).
 * One thread per pair, shaped like score32_kernel (sw_kernels.cu): the query is walked in strips of 16 rows
 * held in registers, the subject's 2-bit record gives the columns, and the (H, G) row between strips is parked
 * per column in global scratch laid out [column][thread].  32-bit arithmetic, exact for every score.
 */
#include "sw_strip.cuh"
#include "sw_kernels.h"

#include <stdint.h>

#define SW_DEVERR_LOCATE 64u   /* the reverse pass did not reach the forward pass's score */
#define SW_DEVERR_ALIGN 128u   /* the walk left the rectangle, did not end at (1, 1) in M or did not score S; or an
                                  index into the direction buffer or an op slot was out of range */

namespace swk {

constexpr int kLR = 16;        // query rows per strip

enum LocateMode { kForward, kReverse, kTrace };

// direction bits of one cell of the trace pass (one nibble, row r of a strip at bits 4r .. 4r+3)
constexpr uint32_t kDirHFromI = 1;    // H came from I (M < I); clear: from M
constexpr uint32_t kDirULeft = 2;     // I came from the left, G(i, j-1) (G(i-1, j) < G(i, j-1)); clear: from up
constexpr uint32_t kDirGExtend = 4;   // G was an extend, I + ge (M + goe < I + ge); clear: an open, M + goe

struct LocateArgs {
    const uint8_t *raw; const uint64_t *off; const uint32_t *len; uint32_t ns; size_t raw_bytes;
    const uint8_t *qpacked; const uint32_t *qoff; const uint32_t *qlen; int nq; size_t q_bytes;
    const uint2 *pairs; uint32_t npairs;
    int32_t *score; uint4 *coord; size_t out_elems;
    int32_t *scratch; uint32_t max_cols;
    int match, mismatch, goe, ge;
    unsigned *dev_err;
};

// 2-bit code of base k of a packed record (byte k / 4, bits 2 * (k % 4)); `base` is the record's byte offset in
// a buffer of `bytes` bytes (bounds-check build).
__device__ __forceinline__ int locate_code(const uint8_t *buf, uint64_t base, int k, size_t bytes, unsigned bit,
                                       const LocateArgs &a)
{
    SW_CHECK(base + (uint64_t)(k >> 2) < bytes, bit, a);
    return (buf[base + (k >> 2)] >> ((k & 3) * 2)) & 3;
}

// Query / subject position of row / column k of a pass: kTrace runs over the rectangle at (a.q0, a.s0).
template <int MODE, class Args>
__device__ __forceinline__ int row_base(const Args &a, int k)
{
    if constexpr (MODE == kTrace) return a.q0 + k; else return k;
}
template <int MODE, class Args>
__device__ __forceinline__ int col_base(const Args &a, int k)
{
    if constexpr (MODE == kTrace) return a.s0 + k; else return k;
}

// One pass over m query rows x n subject columns.  kForward: rows are query[0..m), columns subject[0..n);
// returns the largest M in *bm and its first cell in (column, row) order in (*bi, *bj), 1-based.
// kReverse: rows are query[m-1], query[m-2], ..., columns subject[n-1], subject[n-2], ...; returns in (*bi, *bj)
// the first cell in (column, row) order whose M reaches `target`, and *bm = target (0 and (0, 0) if none does).
// kTrace (Args = TraceArgs): rows are query[a.q0..a.q0+m), columns subject[a.s0..a.s0+n); writes the direction
// bits of strip k, column j to a.trace[k * n + j] and returns nothing useful.
template <int MODE, class Args>
__device__ __forceinline__ void locate_pass(uint64_t qbase, int m, uint64_t sbase, int n, int target, int32_t *Hb,
                                            int32_t *Gb, size_t nthreads, const Args &a, int *bm, int *bi, int *bj)
{
    constexpr bool REV = MODE == kReverse;
    const int gb = a.goe > a.ge ? a.goe : a.ge;
    int best = 0, best_i = 0, best_j = 0;
    int ncols = n;                                      // REV: columns a later strip can still win in
    for (int j = 0; j < ncols; ++j) {
        SW_CHECK((uint32_t)j < a.max_cols, SW_DEVERR_BND, a);
        Hb[(size_t)j * nthreads] = 0; Gb[(size_t)j * nthreads] = gb;
    }
    for (int r0 = 0; r0 < m && ncols > 0; r0 += kLR) {
        const int nr = (m - r0 < kLR) ? (m - r0) : kLR;
        uint32_t qw = 0;                                // 2-bit codes of the strip's rows
        for (int r = 0; r < nr; ++r) {
            const int i = r0 + r;
            qw |= (uint32_t)locate_code(a.qpacked, qbase, row_base<MODE>(a, REV ? m - 1 - i : i), a.q_bytes, SW_DEVERR_PROF, a) << (2 * r);
        }
        int H[kLR], Gv[kLR];
#pragma unroll
        for (int r = 0; r < kLR; ++r) { H[r] = 0; Gv[r] = gb; }
        int hd_top = 0;                                 // H(r0-1, j-1)
        int nx_h = Hb[0], nx_g = Gb[0];
        int sbest = 0, sbest_r = 0, sbest_j = 0;        // forward: this strip's best M and its first cell
        for (int j = 0; j < ncols; ++j) {
            const int tj = locate_code(a.raw, sbase, col_base<MODE>(a, REV ? n - 1 - j : j), a.raw_bytes, SW_DEVERR_TP, a);
            const int top_h = nx_h, top_g = nx_g;       // H, G of row r0-1 in this column
            if (j + 1 < ncols) {
                SW_CHECK((uint32_t)(j + 1) < a.max_cols, SW_DEVERR_BND, a);
                nx_h = Hb[(size_t)(j + 1) * nthreads]; nx_g = Gb[(size_t)(j + 1) * nthreads];
            }
            int diag = hd_top, gu = top_g;
            unsigned reached = 0;                       // REV: rows of this column whose M reaches target
            uint64_t dirs = 0;                          // kTrace: this column's nibbles
#pragma unroll
            for (int r = 0; r < kLR; ++r) {
                if (r < nr) {
                    const int sc = ((int)((qw >> (2 * r)) & 3) == tj) ? a.match : a.mismatch;
                    const int mm = __viaddmax_s32(diag, sc, 0);               // M = max(0, H(i-1, j-1) + s)
                    const int ii = Gv[r] > gu ? Gv[r] : gu;                   // I = max(G(i, j-1), G(i-1, j))
                    if constexpr (MODE == kTrace) {
                        const uint32_t d = (mm < ii ? kDirHFromI : 0u) | (gu < Gv[r] ? kDirULeft : 0u) |
                                           (mm + a.goe < ii + a.ge ? kDirGExtend : 0u);
                        dirs |= (uint64_t)d << (4 * r);
                    }
                    diag = H[r];
                    gu = __viaddmax_s32(mm, a.goe, ii + a.ge);                // G = max(M + go + ge, I + ge)
                    Gv[r] = gu;
                    H[r] = mm > ii ? mm : ii;                                 // H = max(M, I)
                    if (REV) {
                        reached |= (mm >= target ? 1u : 0u) << r;
                    } else if (mm > sbest) {
                        sbest = mm; sbest_r = r; sbest_j = j;
                    }
                }
            }
            hd_top = top_h;
            Hb[(size_t)j * nthreads] = H[kLR - 1];     // used only below full strips
            Gb[(size_t)j * nthreads] = Gv[kLR - 1];
            if constexpr (MODE == kTrace) {
                const uint64_t w = (uint64_t)(r0 / kLR) * (uint64_t)n + (uint64_t)j;
                SW_CHECK(w < a.trace_words, SW_DEVERR_ALIGN, a);
                a.trace[w] = dirs;
            }
            if (REV && reached) {
                // first row of the first column in this strip; a later strip can only win at a smaller column
                best = target; best_i = r0 + __ffs(reached); best_j = j + 1;
                ncols = j;
                break;
            }
        }
        // strips run one after another: a strip's cell wins on a larger M, or on the same M at a smaller column
        // (every earlier strip's rows are smaller)
        if (!REV && (sbest > best || (sbest == best && sbest > 0 && sbest_j + 1 < best_j))) {
            best = sbest; best_i = r0 + sbest_r + 1; best_j = sbest_j + 1;
        }
    }
    *bm = best; *bi = best_i; *bj = best_j;
}

__global__ void __launch_bounds__(128) locate_kernel(const LocateArgs a)
{
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int32_t *Hb = a.scratch + tid;                      // Hb[j * nthreads]: H(strip bottom, j)
    int32_t *Gb = a.scratch + (size_t)a.max_cols * nthreads + tid;
    for (size_t job = tid; job < a.npairs; job += nthreads) {
        const uint2 p = a.pairs[job];                   // {query row, shard-local subject}
        SW_CHECK(p.x < (uint32_t)a.nq && p.y < a.ns, SW_DEVERR_OUT, a);
        const int m = (int)a.qlen[p.x], n = (int)a.len[p.y];
        const uint64_t qbase = a.qoff[p.x], sbase = a.off[p.y];
        int S = 0, qe = 0, se = 0;
        locate_pass<kForward>(qbase, m, sbase, n, 0, Hb, Gb, nthreads, a, &S, &qe, &se);
        uint4 c = make_uint4(0u, 0u, 0u, 0u);
        if (S > 0) {
            int found = 0, ra = 0, rb = 0;
            locate_pass<kReverse>(qbase, qe, sbase, se, S, Hb, Gb, nthreads, a, &found, &ra, &rb);
            SW_CHECK(found == S, SW_DEVERR_LOCATE, a);
            c = make_uint4((unsigned)(qe - ra), (unsigned)qe, (unsigned)(se - rb), (unsigned)se);
        }
        SW_CHECK(job < a.out_elems, SW_DEVERR_OUT, a);
        a.score[job] = S;
        a.coord[job] = c;
    }
}

// the trace pass's view of one pair: the launch's arguments plus the rectangle's origin and direction region
struct TraceArgs : LocateArgs {
    int q0, s0;
    uint64_t *trace; uint64_t trace_words;
};

struct AlignArgs {
    LocateArgs loc;                    // pairs, located score and coord (inputs here), (H, G) scratch
    uint32_t job0, job1;               // this round: pairs [job0, job1)
    const uint64_t *trace_off;         // per pair: first word of its direction region in trace
    uint64_t *trace; uint64_t trace_words;
    const uint64_t *ops_off;           // per pair: first entry of its op slot, (q_end-q_begin) + (s_end-s_begin) - 1 long
    uint32_t *ops; uint64_t ops_elems;
    uint32_t *nops;                    // per pair: ops written to its slot
};

// Trace pass over the located rectangle, then the walk of DESIGN.md section 5.8 from (m, n) in state M to (1, 1),
// run-length encoded as BAM ops (len << 4 | op) in the pair's slot.
__global__ void __launch_bounds__(128) align_kernel(const AlignArgs A)
{
    const LocateArgs &a = A.loc;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int32_t *Hb = a.scratch + tid;
    int32_t *Gb = a.scratch + (size_t)a.max_cols * nthreads + tid;
    for (size_t job = A.job0 + tid; job < A.job1; job += nthreads) {
        SW_CHECK(job < a.out_elems, SW_DEVERR_OUT, a);
        const int S = a.score[job];
        if (S <= 0) { A.nops[job] = 0; continue; }
        const uint2 p = a.pairs[job];
        SW_CHECK(p.x < (uint32_t)a.nq && p.y < a.ns, SW_DEVERR_OUT, a);
        const uint4 c = a.coord[job];
        const int qb = (int)c.x, m = (int)(c.y - c.x), sb = (int)c.z, n = (int)(c.w - c.z);
        const uint64_t qbase = a.qoff[p.x], sbase = a.off[p.y];
        const uint64_t toff = A.trace_off[job];
        SW_CHECK(toff + (uint64_t)((m + kLR - 1) / kLR) * (uint64_t)n <= A.trace_words, SW_DEVERR_ALIGN, a);
        const uint64_t tw = A.trace_words - toff;
        uint64_t *tr = A.trace + toff;
        TraceArgs t;
        static_cast<LocateArgs &>(t) = a;
        t.q0 = qb; t.s0 = sb; t.trace = tr; t.trace_words = tw;
        int unused_m, unused_i, unused_j;
        locate_pass<kTrace>(qbase, m, sbase, n, 0, Hb, Gb, nthreads, t, &unused_m, &unused_i, &unused_j);

        const uint64_t slot_cap = (uint64_t)m + (uint64_t)n - 1;
        SW_CHECK(A.ops_off[job] + slot_cap <= A.ops_elems, SW_DEVERR_ALIGN, a);
        uint32_t *slot = A.ops + A.ops_off[job];
        enum { kM, kI, kDiag, kGap };                  // kDiag / kGap: just arrived, the cell's bits give the state
        int i = m, j = n, st = kM, got = 0;
        bool ended = false;
        uint32_t run_op = 0, run_len = 0, k = 0;
        for (;;) {
            if (i < 1 || j < 1) break;                 // left the rectangle
            const uint64_t w = (uint64_t)((i - 1) / kLR) * (uint64_t)n + (uint64_t)(j - 1);
            SW_CHECK(w < tw, SW_DEVERR_ALIGN, a);
            const uint32_t d = (uint32_t)(tr[w] >> (4 * ((i - 1) % kLR))) & 15u;
            if (st == kDiag) {
                st = (d & kDirHFromI) ? kI : kM;
            } else if (st == kGap) {
                if (d & kDirGExtend) st = kI;
                else { st = kM; got += a.goe - a.ge; }   // the gap run opened here: go once, ge per column
            }
            uint32_t op;
            if (st == kM) {
                const bool eq = locate_code(a.qpacked, qbase, qb + i - 1, a.q_bytes, SW_DEVERR_PROF, a) ==
                                locate_code(a.raw, sbase, sb + j - 1, a.raw_bytes, SW_DEVERR_TP, a);
                op = eq ? 7u : 8u;                     // '=' / 'X'
                got += eq ? a.match : a.mismatch;
                ended = i == 1 && j == 1;
                --i; --j; st = kDiag;
            } else {
                if (d & kDirULeft) { op = 2u; --j; }   // 'D': a subject base against a gap
                else { op = 1u; --i; }                 // 'I': a query base against a gap
                got += a.ge; st = kGap;
            }
            if (op != run_op) {
                if (run_len) {
                    SW_CHECK(k < slot_cap, SW_DEVERR_ALIGN, a);
                    if (k < slot_cap) slot[k++] = run_len << 4 | run_op;
                }
                run_op = op; run_len = 0;
            }
            ++run_len;
            if (ended) break;
        }
        SW_CHECK(k < slot_cap, SW_DEVERR_ALIGN, a);
        if (k < slot_cap) slot[k++] = run_len << 4 | run_op;
        for (uint32_t x = 0, y = k - 1; x < y; ++x, --y) { const uint32_t t = slot[x]; slot[x] = slot[y]; slot[y] = t; }
        SW_CHECK(ended && got == S, SW_DEVERR_ALIGN, a);
        A.nops[job] = k;
    }
}

}  // namespace swk

namespace {

swk::LocateArgs locate_args(const SwLocateLaunch &L)
{
    swk::LocateArgs a{};
    a.raw = L.db.raw; a.off = L.db.off; a.len = L.db.len; a.ns = L.db.ns; a.raw_bytes = L.raw_bytes;
    a.qpacked = L.q.packed; a.qoff = L.q.off; a.qlen = L.q.len; a.nq = L.q.nq; a.q_bytes = L.q_bytes;
    a.pairs = L.pairs; a.npairs = L.npairs;
    a.score = L.score; a.coord = L.coord; a.out_elems = L.out_elems;
    a.scratch = L.scratch; a.max_cols = L.max_cols;
    a.match = L.sc.match; a.mismatch = L.sc.mismatch; a.goe = L.sc.goe; a.ge = L.sc.ge;
    a.dev_err = L.dev_err;
    return a;
}

}  // namespace

cudaError_t sw_launch_locate(cudaStream_t st, const SwLocateLaunch &L)
{
    const int bt = 128;
    const int grid = L.threads_total / bt;
    if (grid <= 0 || L.npairs == 0) return cudaErrorInvalidValue;
    swk::locate_kernel<<<grid, bt, 0, st>>>(locate_args(L));
    return cudaGetLastError();
}

cudaError_t sw_launch_align(cudaStream_t st, const SwAlignLaunch &L)
{
    const int bt = 128;
    const int grid = L.loc.threads_total / bt;
    if (grid <= 0 || L.job1 <= L.job0 || L.job1 > L.loc.npairs) return cudaErrorInvalidValue;
    swk::AlignArgs a{};
    a.loc = locate_args(L.loc);
    a.job0 = L.job0; a.job1 = L.job1;
    a.trace_off = L.trace_off; a.trace = L.trace; a.trace_words = L.trace_words;
    a.ops_off = L.ops_off; a.ops = L.ops; a.ops_elems = L.ops_elems;
    a.nops = L.nops;
    swk::align_kernel<<<grid, bt, 0, st>>>(a);
    return cudaGetLastError();
}
