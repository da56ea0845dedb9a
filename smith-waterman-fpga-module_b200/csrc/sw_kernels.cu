/*
 * sw_kernels.cu -- the kernels around the strip kernel (sw_strip.cuh): code-stream builder, 32-bit
 * scorer / overflow fix-up, best-hit and top-k merge; the variant table and the launchers.
 */
#include "sw_variants.h"
#include "sw_wave.cuh"

#include <stdint.h>

#include <algorithm>
#include <vector>

namespace swk {

// ------------------------------------------------------------------------------------------
// Column code stream builder: one byte per column of a pair (codes 0..20, see kHiEndedCode /
// kPadCode), four columns per 32-bit word, word k of the 32 pairs of a tile contiguous.
// One warp per tile: lane = pair slot, loop over words -> coalesced 128-byte stores.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t load8_bases(const uint8_t *rec, uint32_t len, uint32_t k)
{
    // the 4 bases of columns 4k .. 4k+3 (one packed byte), 0 past the end of the record
    return (k < ((len + 3) >> 2)) ? rec[k] : 0u;
}

__global__ void __launch_bounds__(256) build_tp_kernel(const uint8_t *raw, const uint64_t *off,
                                                      const uint32_t *len, const uint32_t *pair_subj,
                                                      const uint32_t *pair_len, const uint64_t *tile_woff,
                                                      uint32_t *tp, uint32_t ntiles)
{
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (warp >= ntiles) return;
    const uint64_t w0 = tile_woff[warp], w1 = tile_woff[warp + 1];
    const uint32_t kmax = (uint32_t)((w1 - w0) >> 5);
    const uint32_t pair = warp * 32 + lane;
    const uint32_t slo = pair_subj[2 * pair], shi = pair_subj[2 * pair + 1];
    const uint32_t nlo = pair_len[2 * pair], nhi = pair_len[2 * pair + 1];
    const uint8_t *rlo = (slo != SW_NO_SUBJECT) ? raw + off[slo] : nullptr;
    const uint8_t *rhi = (shi != SW_NO_SUBJECT) ? raw + off[shi] : nullptr;
    for (uint32_t k = 0; k < kmax; ++k) {
        const uint32_t a = rlo ? load8_bases(rlo, nlo, k) : 0u;
        const uint32_t b = rhi ? load8_bases(rhi, nhi, k) : 0u;
        tp[w0 + (uint64_t)k * 32 + lane] = make_code_word(a, b, k, nlo, nhi);
    }
}

// ------------------------------------------------------------------------------------------
// 32-bit scorer: one thread per (query, subject) job, any length, any score range, W-bit mode.
// The recurrence is symmetric in its two sequences, so the SHORTER one is walked as columns and
// the longer one in strips of 16 rows held in registers (their 2-bit codes fit one word); the
// bottom row (H, G) of a strip is parked per column in global scratch laid out [column][thread],
// so a warp touches one 128-byte line per access and a cell costs 4/16 memory operations -- and
// the scratch is bounded by min(longest query, longest subject) columns per thread.
// Explicit form of SW_ProcessingElement_v1.0.v (M, I = max(G_left, G_up), ...).
// mode 0: all jobs; mode 1: matrix entries flagged SW_OVERFLOW_SENTINEL; mode 2: overflow list.
// ------------------------------------------------------------------------------------------
constexpr int kGR = 16;

struct Score32Args {
    const uint8_t *raw; const uint64_t *off; const uint32_t *len; uint32_t ns;
    const uint8_t *qpacked; const uint32_t *qoff; const uint32_t *qlen; int q0, q1;
    void *out; size_t out_stride; int out_mode;
    int32_t *scratch; uint32_t max_cols;
    int match, mismatch, goe, ge, limit, mode;
    const unsigned *list_count; const uint2 *list; unsigned list_cap; int32_t *list_score;
    unsigned long long wave32_min_cells;
    unsigned wave32_limit;
};

__device__ __forceinline__ int score32_pair(const uint8_t *rp, int m, const uint8_t *cp, int n, int32_t *Hb,
                                            int32_t *Gb, size_t nthreads, const Score32Args &a)
{
    // rows = (rp, m), columns = (cp, n), n <= max_cols
    const int gb = a.goe > a.ge ? a.goe : a.ge;
    for (int j = 0; j < n; ++j) { Hb[(size_t)j * nthreads] = 0; Gb[(size_t)j * nthreads] = gb; }
    int best = 0;
    for (int r0 = 0; r0 < m; r0 += kGR) {
        const int nr = (m - r0 < kGR) ? (m - r0) : kGR;
        uint32_t qw = 0;                               // 2-bit codes of the strip's rows
        for (int r = 0; r < nr; ++r) {
            const int i = r0 + r;
            qw |= (uint32_t)((rp[i >> 2] >> ((i & 3) * 2)) & 3) << (2 * r);
        }
        int H[kGR], Gv[kGR];
#pragma unroll
        for (int r = 0; r < kGR; ++r) { H[r] = 0; Gv[r] = gb; }
        int hd_top = 0;                                // H(r0-1, j-1)
        int nx_h = n ? Hb[0] : 0, nx_g = n ? Gb[0] : gb;
        for (int j = 0; j < n; ++j) {
            const int tj = (cp[j >> 2] >> ((j & 3) * 2)) & 3;
            const int top_h = nx_h, top_g = nx_g;      // H, G of row r0-1 in this column
            if (j + 1 < n) { nx_h = Hb[(size_t)(j + 1) * nthreads]; nx_g = Gb[(size_t)(j + 1) * nthreads]; }
            int diag = hd_top, gu = top_g;
#pragma unroll
            for (int r = 0; r < kGR; ++r) {
                if (r < nr) {
                    const int sc = ((int)((qw >> (2 * r)) & 3) == tj) ? a.match : a.mismatch;
                    int mm = diag + sc;                             // v1.0.v:287
                    mm = mm > 0 ? mm : 0;                           // v1.0.v:288
                    if (a.limit && mm > a.limit) mm = 0;            // W-bit wrap-then-clamp
                    const int ii = Gv[r] > gu ? Gv[r] : gu;         // v1.0.v:126-129, 291
                    diag = H[r];
                    const int a1 = mm + a.goe, a2 = ii + a.ge;
                    gu = a1 > a2 ? a1 : a2;
                    Gv[r] = gu;
                    H[r] = mm > ii ? mm : ii;
                    best = H[r] > best ? H[r] : best;               // v1.0.v:411-420
                }
            }
            hd_top = top_h;
            Hb[(size_t)j * nthreads] = H[kGR - 1];                  // used only below full strips
            Gb[(size_t)j * nthreads] = Gv[kGR - 1];
        }
    }
    return best;
}

__global__ void __launch_bounds__(128) score32_kernel(const Score32Args a)
{
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int32_t *Hb = a.scratch + tid;                          // Hb[j * nthreads]: H(strip bottom, j)
    int32_t *Gb = a.scratch + (size_t)a.max_cols * nthreads + tid;
    size_t njobs;
    if (a.mode == 2) {
        const unsigned c = *a.list_count;
        njobs = c < a.list_cap ? c : a.list_cap;
    } else {
        njobs = (size_t)a.ns * (size_t)(a.q1 - a.q0);
    }
    for (size_t job = tid; job < njobs; job += nthreads) {
        uint32_t s; int q;
        if (a.mode == 2) { q = (int)a.list[job].x; s = a.list[job].y; }
        else { s = (uint32_t)(job % a.ns); q = a.q0 + (int)(job / a.ns); }
        if (a.mode == 1) {
            const bool flagged = a.out_mode == SW_OUT_I16 ? ((const int16_t *)a.out)[(size_t)q * a.out_stride + s] == SW_OVERFLOW_SENTINEL
                                                          : ((const int32_t *)a.out)[(size_t)q * a.out_stride + s] == SW_OVERFLOW_SENTINEL;
            if (!flagged) continue;
        }
        const int m = (int)a.qlen[q], n = (int)a.len[s];
        // long entries at the head of the list belong to the band-pipelined 32-bit scorer
        if (a.mode == 2 && a.wave32_min_cells && wave32_takes((unsigned)job, (uint32_t)m, (uint32_t)n, a.wave32_min_cells, a.wave32_limit)) continue;
        const uint8_t *qp = a.qpacked + a.qoff[q];
        const uint8_t *tpk = a.raw + a.off[s];
        const int best = (n <= m) ? score32_pair(qp, m, tpk, n, Hb, Gb, nthreads, a)
                                  : score32_pair(tpk, n, qp, m, Hb, Gb, nthreads, a);
        if (a.mode == 2 && a.list_score) a.list_score[job] = best;
        if (a.out) {
            // a 16-bit matrix keeps the sentinel for scores it cannot hold (they are on the list)
            if (a.out_mode == SW_OUT_I16) { if (best <= 32767) ((int16_t *)a.out)[(size_t)q * a.out_stride + s] = (int16_t)best; }
            else ((int32_t *)a.out)[(size_t)q * a.out_stride + s] = best;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Per-query best hit (the bank's never-driven max / vld_max, ScoreBank_v2.v:42-43).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) best_kernel(const int32_t *scores, size_t stride, uint32_t ns,
                                                    int32_t *best_score, uint32_t *best_index)
{
    const int q = blockIdx.x;
    const int32_t *row = scores + (size_t)q * stride;
    // key = (score << 32) | ~index : max key = highest score, lowest index
    unsigned long long key = 0;
    for (uint32_t s = threadIdx.x; s < ns; s += blockDim.x) {
        const unsigned long long k = ((unsigned long long)(uint32_t)row[s] << 32) | (uint32_t)(~s);
        key = k > key ? k : key;
    }
    __shared__ unsigned long long sk[32];
    for (int o = 16; o >= 1; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o);
        key = other > key ? other : key;
    }
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x < 32) {
        key = (threadIdx.x < (blockDim.x >> 5)) ? sk[threadIdx.x] : 0ull;
        for (int o = 16; o >= 1; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o);
            key = other > key ? other : key;
        }
        if (threadIdx.x == 0) {
            best_score[q] = ns ? (int32_t)(key >> 32) : 0;
            best_index[q] = ns ? ~(uint32_t)(key & 0xFFFFFFFFu) : 0u;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Top-k merge: one block per query folds the per-block lists of the strip epilogue (nlists x k
// keys, descending) and the recomputed overflow entries of this query into out_keys[q][0..k).
// Keys are unique (they contain the subject index), so "largest key below the previous pick"
// enumerates them in order: k rounds of a block-wide max.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) topk_merge_kernel(const unsigned long long *keys, int nlists, int nq, int k,
                                                        const unsigned *ovf_count, const uint2 *ovf_list,
                                                        const int32_t *ovf_score, unsigned ovf_cap,
                                                        unsigned long long *out_keys)
{
    const int q = blockIdx.x;
    __shared__ unsigned long long s_red[8];
    __shared__ unsigned long long s_pick;
    const unsigned novf = ovf_count ? min(*ovf_count, ovf_cap) : 0u;
    unsigned long long prev = ~0ull;
    for (int round = 0; round < k; ++round) {
        unsigned long long best = 0;
        for (int i = threadIdx.x; i < nlists * k; i += blockDim.x) {
            const unsigned long long v = keys[((size_t)(i / k) * nq + q) * k + (i % k)];
            if (v < prev && v > best) best = v;
        }
        for (unsigned i = threadIdx.x; i < novf; i += blockDim.x) {
            if ((int)ovf_list[i].x != q) continue;
            const unsigned long long v = ((unsigned long long)(uint32_t)ovf_score[i] << 32) | (uint32_t)(~ovf_list[i].y);
            if (v < prev && v > best) best = v;
        }
        for (int o = 16; o >= 1; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, best, o);
            best = other > best ? other : best;
        }
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long b = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) b = s_red[w] > b ? s_red[w] : b;
            s_pick = b;
            out_keys[(size_t)q * k + round] = b;
        }
        __syncthreads();
        prev = s_pick;
        if (prev == 0) {                       // nothing left: the remaining slots stay empty
            for (int r = round + 1 + threadIdx.x; r < k; r += blockDim.x) out_keys[(size_t)q * k + r] = 0;
            break;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Variant table (assembled from the translation units that hold the instances)
// ------------------------------------------------------------------------------------------
static const std::vector<VariantEntry> &variants()
{
    static const std::vector<VariantEntry> all = [] {
        std::vector<VariantEntry> v;
        const VariantPart parts[] = {sw_variants_part_a(), sw_variants_part_b(), sw_variants_part_c(),
                                     sw_variants_part_d(), sw_variants_part_e(), sw_variants_part_f(),
                                     sw_variants_part_g(), sw_variants_part_h()};
        for (const VariantPart &p : parts) v.insert(v.end(), p.v, p.v + p.n);
        return v;
    }();
    return all;
}

}  // namespace swk

using namespace swk;

// dynamic + static shared memory must stay below 48 KB unless the kernel opts in; the strip kernel has
// a few KB of static shared memory (work item, top-k candidates), so opt in from 32 KB of dynamic on
static const size_t kSmemOptIn = 32 * 1024;

static bool g_no_fixed = false;     // testing: force the run-time-penalty instance
void sw_strip_disable_fixed(bool off) { g_no_fixed = off; }

int sw_strip_variant_count(void) { return (int)variants().size(); }

const SwStripVariant *sw_strip_variant(int idx)
{
    return (idx >= 0 && idx < (int)variants().size()) ? &variants()[idx].info : nullptr;
}

size_t sw_strip_smem_bytes(int idx, int chunk_passes)
{
    const SwStripVariant *v = sw_strip_variant(idx);
    if (!v) return 0;
    const int rs = v->R / v->S;
    return (size_t)chunk_passes * v->G * v->S * ((rs + 1) / 2) * kCodesPerRow * sizeof(uint2);
}

cudaError_t sw_strip_occupancy(int idx, size_t smem_bytes, int *blocks_per_sm)
{
    const SwStripVariant *v = sw_strip_variant(idx);
    if (!v) return cudaErrorInvalidValue;
    const void *fn = (const void *)variants()[idx].fn;
    if (smem_bytes > kSmemOptIn) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
        if (e != cudaSuccess) return e;
    }
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, v->block_threads, smem_bytes);
}

static StripFn pick_instance(const SwStripLaunch &L, const char **kind)
{
    const VariantEntry &v = variants()[L.vidx];
    const SwScoring &sc = L.sc;
    if (L.direct) { *kind = "direct"; return sc.limit ? nullptr : v.fn_direct; }
    if (sc.limit) { *kind = "w12"; return v.fn_w12; }
    if (!g_no_fixed && v.fn_fixed && sc.goe == kFixedGoe && sc.ge == kFixedGe) { *kind = "fixed"; return v.fn_fixed; }
    if (!g_no_fixed && v.fn_fixed2 && sc.goe == kFixed2Goe && sc.ge == kFixed2Ge) { *kind = "fixed"; return v.fn_fixed2; }
    *kind = "runtime";
    return v.fn;
}

const char *sw_strip_instance_kind(const SwStripLaunch &L)
{
    if (L.vidx < 0 || L.vidx >= (int)variants().size()) return "none";
    if (L.jit_kernel && !L.direct && !L.sc.limit) return "jit";
    const char *kind = "none";
    pick_instance(L, &kind);
    return kind;
}

cudaError_t sw_launch_strip(cudaStream_t st, const SwStripLaunch &L)
{
    if (L.vidx < 0 || L.vidx >= (int)variants().size()) return cudaErrorInvalidValue;
    const VariantEntry &v = variants()[L.vidx];
    const char *kind = "none";
    StripFn fn = pick_instance(L, &kind);
    if (fn == nullptr) return cudaErrorInvalidValue;
    const int ppb = v.info.block_threads / v.info.G;
    const SwScoring &sc = L.sc;
    StripArgs a{};
    a.tp = L.db.tp; a.tile_woff = L.db.tile_woff; a.pair_len = L.db.pair_len; a.pair_subj = L.db.pair_subj;
    a.npairs = L.db.npairs; a.npb = (L.db.npairs + ppb - 1) / ppb; a.superblock = L.superblock;
    a.qpacked = L.q.packed; a.qoff = L.q.off; a.qlen = L.q.len; a.qidx = L.qidx; a.q0 = L.q0; a.nql = L.nql;
    a.out = L.out; a.out_stride = L.out_stride; a.out_mode = L.out_mode;
    a.bnd = L.bnd; a.bnd_cols = L.bnd_cols; a.counter = L.counter; a.sticky = (L.counter && L.sticky > 0 && L.nql > 1) ? L.sticky : 0;
    a.chunk_passes = L.chunk_passes;
    const bool split = L.nparts > 1 && L.part_done && L.part_best && L.part_passes > 0 && L.part_passes % L.chunk_passes == 0 && !L.direct;
    a.nparts = split ? L.nparts : 0; a.part_passes = split ? L.part_passes : 0;
    a.part_done = split ? L.part_done : nullptr; a.part_best = split ? L.part_best : nullptr;
    if (L.nparts > 1 && !split) return cudaErrorInvalidValue;
    a.match = sc.match; a.mismatch = sc.mismatch; a.goe = sc.goe; a.ge = sc.ge; a.limit = sc.limit;
    a.goe2 = ((uint32_t)sc.goe & 0xFFFFu) * 0x10001u; a.ge2 = ((uint32_t)sc.ge & 0xFFFFu) * 0x10001u;
    a.ovf_limit = 32767 - sc.match - 1;
    a.zero = 0;
    a.raw = L.db.raw; a.off = L.db.off; a.pair_desc = L.db.pair_desc;
    a.ovf_count = L.ovf_count; a.ovf_list = L.ovf_list; a.ovf_cap = L.ovf_cap;
    a.topk_keys = L.topk_keys; a.topk_k = L.topk_k; a.topk_nq = L.topk_nq;
    a.hits = L.hits.keys; a.hits_score = L.hits.score; a.hits_count = L.hits.count; a.hits_cap = L.hits.cap;
    a.min_score = L.hits.min_score; a.hits_shift = L.hits.shift;
    a.dev_err = L.dev_err;
    a.done_count = L.done_count; a.done_flag = L.done_flag; a.done_seq = L.done_seq;
#ifdef SW_BOUNDS_CHECK
    a.tp_words = L.db.tp_words; a.bnd_elems = L.bnd_elems; a.out_elems = L.out_elems;
#endif
    if (L.out_mode == SW_OUT_TOPK && (L.topk_k < 1 || L.topk_k > kMaxTopK || !L.topk_keys)) return cudaErrorInvalidValue;
    if (L.out_mode == SW_OUT_HITS && (L.direct || (L.hits.keys && (!L.hits.score || !L.hits.count)))) return cudaErrorInvalidValue;
    const size_t smem = sw_strip_smem_bytes(L.vidx, L.chunk_passes);
    if (L.jit_kernel && !L.direct && !sc.limit) {
        void *params[] = {&a};
        cudaKernel_t k = (cudaKernel_t)L.jit_kernel;
        if (smem > kSmemOptIn) {
            cudaError_t e = cudaFuncSetAttribute((const void *)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        return cudaLaunchKernel((const void *)k, dim3(L.grid), dim3(v.info.block_threads), params, smem, st);
    }
    if (smem > kSmemOptIn) {
        cudaError_t e = cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    fn<<<L.grid, v.info.block_threads, smem, st>>>(a);
    return cudaGetLastError();
}

// ---- band-pipelined kernel ---------------------------------------------------------------------
// Four instances (measured over few-long-pair shapes, profiles/r02_wave_instance_ab2.txt, r02_wave_vs_strip_mid.txt):
//   0  R8x2        bands of 512 rows, one column per step, four pairs per block: many pairs (the
//                  GPU is full of pair-bands; throughput-bound)
//   1  R8x1 C4     bands of 256 rows, four columns per step, ONE pair per block: a few dozen to a
//                  few hundred pairs
//   2  R8x1 C2     bands of 256 rows, two columns per step, one pair per block: a handful of pairs
//                  down to a single one (latency-bound: one warp per band; with one pair per block
//                  the active warps spread over the four schedulers of an SM instead of all being
//                  warp 0 of a four-warp block)
//   3  R8x2 C2     bands of 512 rows, two columns per step, four pairs per block: many pairs of long
//                  subjects (>= 1 kb on average: +2-6 % over instance 0; the doubled skew of 126
//                  columns per band costs more than that on shorter ones)
namespace {
typedef void (*WaveFn)(const WaveArgs);
struct WaveInstance { int rows, bt; size_t smem; WaveFn fn, fn_fixed; const char *name; };
constexpr size_t wave_smem(int rs, int s) { return (size_t)32 * s * ((rs + 1) / 2) * kWaveCodes * sizeof(uint2); }
#define SW_WAVE(RS, S, BT, MINB, BLK, C, LS, NAME) \
    {RS * S * 32, BT, wave_smem(RS, S), sw_wave_kernel<RS, S, ArithS16, BT, MINB, 0, 0, BLK, C, LS>, \
     sw_wave_kernel<RS, S, ArithS16, BT, MINB, kFixedGoe, kFixedGe, BLK, C, LS>, NAME}
const WaveInstance g_wave[] = {
    SW_WAVE(8, 2, 128, 4, 32, 1, false, "wave_s16x2_R8x2_G32"),
    SW_WAVE(8, 1, 32, 8, 32, 4, false, "wave_s16x2_R8x1_G32_C4"),
    SW_WAVE(8, 1, 32, 16, 32, 2, true, "wave_s16x2_R8x1_G32_C2"),
    SW_WAVE(8, 2, 128, 3, 32, 2, false, "wave_s16x2_R8x2_G32_C2"),
    // measured and dropped (profiles/r02_wave_instance_ab.jsonl, r02_wave_instance_ab2.txt): 16-column
    // blocks, 128-row bands (R4x1 with 1 / 2 / 4 columns per step, R4x2), R8x1 with one column per
    // step, four-pair blocks for the multi-column instances
};
constexpr int kNumWave = sizeof(g_wave) / sizeof(g_wave[0]);
inline int wave_index(int inst) { return (inst >= 0 && inst < kNumWave) ? inst : 0; }
}  // namespace

const char *sw_wave_kernel_name(int inst) { return g_wave[wave_index(inst)].name; }
int sw_wave_rows_per_band(int inst) { return g_wave[wave_index(inst)].rows; }
int sw_wave_instance_count(void) { return kNumWave; }
int sw_wave_pairs_per_block(int inst) { return g_wave[wave_index(inst)].bt / 32; }

cudaError_t sw_wave_occupancy(int inst, int *blocks_per_sm)
{
    const WaveInstance &w = g_wave[wave_index(inst)];
    cudaError_t e = cudaFuncSetAttribute((const void *)w.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w.smem);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, (const void *)w.fn, w.bt, w.smem);
}

cudaError_t sw_launch_wave(cudaStream_t st, const SwWaveLaunch &L)
{
    const SwScoring &sc = L.sc;
    if (sc.limit) return cudaErrorInvalidValue;            // exact arithmetic only
    const WaveInstance &w = g_wave[wave_index(L.instance)];
    WaveFn fn = (!g_no_fixed && sc.goe == kFixedGoe && sc.ge == kFixedGe) ? w.fn_fixed : w.fn;
    WaveArgs a{};
    a.tp = L.db.tp; a.tile_woff = L.db.tile_woff; a.pair_len = L.db.pair_len; a.pair_subj = L.db.pair_subj;
    a.npairs = L.db.npairs; a.npb = (L.db.npairs + (uint32_t)(w.bt / 32) - 1u) / (uint32_t)(w.bt / 32);
    a.qpacked = L.q.packed; a.qoff = L.q.off; a.qlen = L.q.len; a.q = L.query; a.npass = L.npass;
    a.out_row = L.out_row >= 0 ? L.out_row : L.query;
    a.out = L.out; a.out_stride = L.out_stride; a.out_mode = L.out_mode;
    a.bnd = (ulonglong2 *)L.bnd; a.cols_stride = L.cols_stride; a.epoch = L.epoch; a.best = L.best; a.done = L.done; a.counter = L.counter;
    a.match = sc.match; a.mismatch = sc.mismatch; a.goe = sc.goe; a.ge = sc.ge;
    a.goe2 = ((uint32_t)sc.goe & 0xFFFFu) * 0x10001u; a.ge2 = ((uint32_t)sc.ge & 0xFFFFu) * 0x10001u;
    a.ovf_limit = 32767 - sc.match - 1;
    a.zero = 0;
    a.ovf_count = L.ovf_count; a.ovf_list = L.ovf_list; a.ovf_cap = L.ovf_cap;
    a.dev_err = L.dev_err;
    a.spin_limit = 1u << 24;
    a.tp_words = L.db.tp_words; a.bnd_elems = L.bnd_elems; a.out_elems = L.out_elems;
    cudaError_t e = cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w.smem);
    if (e != cudaSuccess) return e;
    fn<<<L.grid, w.bt, w.smem, st>>>(a);
    return cudaGetLastError();
}

static_assert(SW_WAVE32_MAX_ENTRIES == kWave32MaxEntries && SW_WAVE32_ROWS == kWave32Rows, "sw_kernels.h / sw_wave.cuh");
namespace {
constexpr int kWave32MinBlocks = 16;
const auto g_wave32 = sw_wave32_kernel<8, 2, kWave32MinBlocks>;
}

cudaError_t sw_wave32_occupancy(int *blocks_per_sm)
{
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, (const void *)g_wave32, 32, 0);
}

cudaError_t sw_launch_wave32(cudaStream_t st, const SwWave32Launch &L)
{
    if (L.sc.limit || L.grid <= 0 || L.nslots == 0) return cudaErrorInvalidValue;    // exact arithmetic only
    Wave32Args a{};
    a.raw = L.db.raw; a.off = L.db.off; a.len = L.db.len;
    a.qpacked = L.q.packed; a.qoff = L.q.off; a.qlen = L.q.len;
    a.list_count = L.list_count; a.list = L.list; a.list_cap = L.list_cap; a.list_score = L.list_score;
    a.entry_base = L.entry_base; a.entry_limit = L.entry_limit;
    a.out = L.out; a.out_stride = L.out_stride; a.out_mode = L.out_mode; a.out_elems = L.out_elems;
    a.bnd = (ulonglong2 *)L.bnd; a.cols_stride = L.cols_stride; a.nslots = L.nslots; a.epoch = L.epoch; a.bnd_elems = L.bnd_elems;
    a.best = (int *)L.state; a.done = L.state + kWave32MaxEntries; a.flag = L.state + 2 * kWave32MaxEntries;
    a.counter = L.counter; a.maxb = L.maxb ? L.maxb : 1u; a.min_cells = L.min_cells;
    a.match = L.sc.match; a.mismatch = L.sc.mismatch; a.goe = L.sc.goe; a.ge = L.sc.ge;
    a.dev_err = L.dev_err;
    a.spin_limit = 1u << 24;
    g_wave32<<<L.grid, 32, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t sw_launch_score32(cudaStream_t st, const SwScore32Launch &L)
{
    const int bt = 128;
    const int grid = L.threads_total / bt;
    if (grid <= 0) return cudaErrorInvalidValue;
    Score32Args a{};
    a.raw = L.db.raw; a.off = L.db.off; a.len = L.db.len; a.ns = L.db.ns;
    a.qpacked = L.q.packed; a.qoff = L.q.off; a.qlen = L.q.len; a.q0 = L.q0; a.q1 = L.q1;
    a.out = L.out; a.out_stride = L.out_stride; a.out_mode = L.out_mode;
    a.scratch = L.scratch; a.max_cols = L.max_cols;
    a.match = L.sc.match; a.mismatch = L.sc.mismatch; a.goe = L.sc.goe; a.ge = L.sc.ge; a.limit = L.sc.limit;
    a.mode = L.mode; a.list_count = L.list_count; a.list = L.list; a.list_cap = L.list_cap; a.list_score = L.list_score;
    a.wave32_min_cells = L.wave32_min_cells; a.wave32_limit = L.wave32_limit;
    score32_kernel<<<grid, bt, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t sw_launch_build_tp(cudaStream_t st, const SwDevDb &db)
{
    const uint32_t ntiles = (db.npairs + 31) / 32;
    if (ntiles == 0) return cudaSuccess;
    const int bt = 256;
    const uint32_t grid = (ntiles * 32 + bt - 1) / bt;
    build_tp_kernel<<<grid, bt, 0, st>>>(db.raw, db.off, db.len, db.pair_subj, db.pair_len, db.tile_woff,
                                         db.tp, ntiles);
    return cudaGetLastError();
}

cudaError_t sw_launch_best(cudaStream_t st, const int32_t *scores, size_t stride, uint32_t ns, int nq,
                           int32_t *best_score, uint32_t *best_index)
{
    if (nq <= 0) return cudaSuccess;
    best_kernel<<<nq, 1024, 0, st>>>(scores, stride, ns, best_score, best_index);
    return cudaGetLastError();
}

namespace {
// k rounds of a block-wide max over the unique keys (score << 32 | ~subject) of one score row
__global__ void __launch_bounds__(256) topk_row_kernel(const int32_t *row, uint32_t n, int k, unsigned long long *out)
{
    __shared__ unsigned long long s_red[8];
    __shared__ unsigned long long s_pick;
    unsigned long long prev = ~0ull;
    for (int round = 0; round < k; ++round) {
        unsigned long long best = 0;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            const int32_t v = row[i];
            if (v < 0) continue;                                   // not scored here (empty subject, overflow sentinel)
            const unsigned long long key = ((unsigned long long)(uint32_t)v << 32) | (uint32_t)(~i);
            if (key < prev && key > best) best = key;
        }
        for (int o = 16; o >= 1; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, best, o);
            best = other > best ? other : best;
        }
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long b = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) b = s_red[w] > b ? s_red[w] : b;
            s_pick = b;
            out[round] = b;
        }
        __syncthreads();
        prev = s_pick;
        if (prev == 0) break;                                      // fewer than k entries: the rest stays 0
    }
}
}  // namespace

cudaError_t sw_launch_topk_row(cudaStream_t st, const int32_t *row, uint32_t n, int q, int k, unsigned long long *keys)
{
    if (k <= 0) return cudaSuccess;
    topk_row_kernel<<<1, 256, 0, st>>>(row, n, k, keys + (size_t)q * k);
    return cudaGetLastError();
}

namespace {
// hit-list entries of one materialised score row (the band-pipelined kernel's) / of the overflow list; grid-stride,
// so a warp's lanes look at consecutive entries and the warp appends with one atomicAdd (hits_slots)
__global__ void __launch_bounds__(256) hits_row_kernel(const int32_t *row, uint32_t n, int q, const SwHitList hl)
{
    const unsigned long long key_row = (unsigned long long)(unsigned)q << hl.shift;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i0 = blockIdx.x * blockDim.x; i0 < n; i0 += stride) {       // warp-uniform trip count
        const uint32_t i = i0 + threadIdx.x;
        const int32_t v = i < n ? row[i] : -1;
        const bool take = v >= 0 && v >= hl.min_score;                         // < 0: not scored here / sentinel
        unsigned long long p = 0, unused = 0;
        if (hits_slots(hl.count, take, false, p, unused) && take && p < hl.cap) { hl.keys[p] = key_row | i; hl.score[p] = v; }
    }
}

__global__ void __launch_bounds__(256) hits_ovf_kernel(const unsigned *ovf_count, const uint2 *ovf_list, const int32_t *ovf_score,
                                                       unsigned ovf_cap, const SwHitList hl)
{
    const unsigned c = *ovf_count, n = c < ovf_cap ? c : ovf_cap;
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned i0 = blockIdx.x * blockDim.x; i0 < n; i0 += stride) {
        const unsigned i = i0 + threadIdx.x;
        const bool take = i < n && ovf_score[i] >= hl.min_score;
        unsigned long long p = 0, unused = 0;
        if (hits_slots(hl.count, take, false, p, unused) && take && p < hl.cap) {
            hl.keys[p] = ((unsigned long long)ovf_list[i].x << hl.shift) | ovf_list[i].y;
            hl.score[p] = ovf_score[i];
        }
    }
}
}  // namespace

cudaError_t sw_launch_hits_row(cudaStream_t st, const int32_t *row, uint32_t n, int q, const SwHitList &hl)
{
    if (n == 0 || !hl.keys) return cudaSuccess;
    const uint32_t grid = std::min<uint32_t>((n + 255) / 256, 1024);
    hits_row_kernel<<<grid, 256, 0, st>>>(row, n, q, hl);
    return cudaGetLastError();
}

cudaError_t sw_launch_hits_ovf(cudaStream_t st, const unsigned *ovf_count, const uint2 *ovf_list, const int32_t *ovf_score,
                               unsigned ovf_cap, const SwHitList &hl)
{
    if (!hl.keys) return cudaSuccess;
    hits_ovf_kernel<<<std::max<unsigned>(1, std::min<unsigned>((ovf_cap + 255) / 256, 256)), 256, 0, st>>>(ovf_count, ovf_list, ovf_score, ovf_cap, hl);
    return cudaGetLastError();
}

cudaError_t sw_launch_topk_merge(cudaStream_t st, const unsigned long long *keys, int nlists, int nq, int k,
                                 const unsigned *ovf_count, const uint2 *ovf_list, const int32_t *ovf_score,
                                 unsigned ovf_cap, unsigned long long *out_keys)
{
    if (nq <= 0 || k <= 0) return cudaSuccess;
    topk_merge_kernel<<<nq, 256, 0, st>>>(keys, nlists, nq, k, ovf_count, ovf_list, ovf_score, ovf_cap, out_keys);
    return cudaGetLastError();
}
