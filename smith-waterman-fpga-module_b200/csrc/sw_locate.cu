/*
 * sw_locate.cu -- begin and end coordinates of the best local alignment of selected (query row, subject)
 * pairs (sw_locate_db).  Two score-only passes per pair, no traceback storage (DESIGN.md section 5.7):
 *   forward  -- the recurrence over the whole pair, keeping the first cell in (column, row) order whose
 *               diagonal value M reaches the pair's maximum S: the end cell (q_end, s_end);
 *   reverse  -- the same recurrence over reverse(query[0:q_end]) x reverse(subject[0:s_end]), stopping at
 *               the first cell in (column, row) order whose M reaches S: (a, b) gives the begin.
 * One thread per pair, shaped like score32_kernel (sw_kernels.cu): the query is walked in strips of 16 rows
 * held in registers, the subject's 2-bit record gives the columns, and the (H, G) row between strips is parked
 * per column in global scratch laid out [column][thread].  32-bit arithmetic, exact for every score.
 */
#include "sw_strip.cuh"
#include "sw_kernels.h"

#include <stdint.h>

#define SW_DEVERR_LOCATE 64u   /* the reverse pass did not reach the forward pass's score */

namespace swk {

constexpr int kLR = 16;        // query rows per strip

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

// One pass over m query rows x n subject columns.  REV = false: rows are query[0..m), columns subject[0..n);
// returns the largest M in *bm and its first cell in (column, row) order in (*bi, *bj), 1-based.
// REV = true: rows are query[m-1], query[m-2], ..., columns subject[n-1], subject[n-2], ...; returns in (*bi, *bj)
// the first cell in (column, row) order whose M reaches `target`, and *bm = target (0 and (0, 0) if none does).
template <bool REV>
__device__ __forceinline__ void locate_pass(uint64_t qbase, int m, uint64_t sbase, int n, int target, int32_t *Hb,
                                            int32_t *Gb, size_t nthreads, const LocateArgs &a, int *bm, int *bi, int *bj)
{
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
            qw |= (uint32_t)locate_code(a.qpacked, qbase, REV ? m - 1 - i : i, a.q_bytes, SW_DEVERR_PROF, a) << (2 * r);
        }
        int H[kLR], Gv[kLR];
#pragma unroll
        for (int r = 0; r < kLR; ++r) { H[r] = 0; Gv[r] = gb; }
        int hd_top = 0;                                 // H(r0-1, j-1)
        int nx_h = Hb[0], nx_g = Gb[0];
        int sbest = 0, sbest_r = 0, sbest_j = 0;        // forward: this strip's best M and its first cell
        for (int j = 0; j < ncols; ++j) {
            const int tj = locate_code(a.raw, sbase, REV ? n - 1 - j : j, a.raw_bytes, SW_DEVERR_TP, a);
            const int top_h = nx_h, top_g = nx_g;       // H, G of row r0-1 in this column
            if (j + 1 < ncols) {
                SW_CHECK((uint32_t)(j + 1) < a.max_cols, SW_DEVERR_BND, a);
                nx_h = Hb[(size_t)(j + 1) * nthreads]; nx_g = Gb[(size_t)(j + 1) * nthreads];
            }
            int diag = hd_top, gu = top_g;
            unsigned reached = 0;                       // REV: rows of this column whose M reaches target
#pragma unroll
            for (int r = 0; r < kLR; ++r) {
                if (r < nr) {
                    const int sc = ((int)((qw >> (2 * r)) & 3) == tj) ? a.match : a.mismatch;
                    const int mm = __viaddmax_s32(diag, sc, 0);               // M = max(0, H(i-1, j-1) + s)
                    const int ii = Gv[r] > gu ? Gv[r] : gu;                   // I = max(G(i, j-1), G(i-1, j))
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
        locate_pass<false>(qbase, m, sbase, n, 0, Hb, Gb, nthreads, a, &S, &qe, &se);
        uint4 c = make_uint4(0u, 0u, 0u, 0u);
        if (S > 0) {
            int found = 0, ra = 0, rb = 0;
            locate_pass<true>(qbase, qe, sbase, se, S, Hb, Gb, nthreads, a, &found, &ra, &rb);
            SW_CHECK(found == S, SW_DEVERR_LOCATE, a);
            c = make_uint4((unsigned)(qe - ra), (unsigned)qe, (unsigned)(se - rb), (unsigned)se);
        }
        SW_CHECK(job < a.out_elems, SW_DEVERR_OUT, a);
        a.score[job] = S;
        a.coord[job] = c;
    }
}

}  // namespace swk

cudaError_t sw_launch_locate(cudaStream_t st, const SwLocateLaunch &L)
{
    const int bt = 128;
    const int grid = L.threads_total / bt;
    if (grid <= 0 || L.npairs == 0) return cudaErrorInvalidValue;
    swk::LocateArgs a{};
    a.raw = L.db.raw; a.off = L.db.off; a.len = L.db.len; a.ns = L.db.ns; a.raw_bytes = L.raw_bytes;
    a.qpacked = L.q.packed; a.qoff = L.q.off; a.qlen = L.q.len; a.nq = L.q.nq; a.q_bytes = L.q_bytes;
    a.pairs = L.pairs; a.npairs = L.npairs;
    a.score = L.score; a.coord = L.coord; a.out_elems = L.out_elems;
    a.scratch = L.scratch; a.max_cols = L.max_cols;
    a.match = L.sc.match; a.mismatch = L.sc.mismatch; a.goe = L.sc.goe; a.ge = L.sc.ge;
    a.dev_err = L.dev_err;
    swk::locate_kernel<<<grid, bt, 0, st>>>(a);
    return cudaGetLastError();
}
