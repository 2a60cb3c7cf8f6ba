/*
 * cg_device.cu — sm_100a kernels and the C ABI of include/crumble_gpu.h.
 *
 * Kernel chain of one cg_run() (DESIGN.md §pipeline):
 *   k_prep_read -> scan(pileup flag) -> k_prep_keys -> scan(prefix max of end keys)
 *   -> k_gap -> scan(sum of zero-coverage gaps, + island compaction) -> k_finish_read
 *   -> k_tile_index -> k_column (pileup + consensus + column heuristics; the hot kernel)
 *   -> scan(flagged columns -> ordered list) -> k_flagged (indel spectrum, STR extents)
 *   -> [depth scans -> k_epochs -> k_deep]   (only when the over-depth test can fire)
 *   -> k_chain -> k_paint -> k_rewrite (per-read replay + P-block) -> scan(BED events)
 *
 * No tensor cores: the path is integer/byte work plus in-order FP64 sums (SURVEY §8d).
 * There is no CPU fallback in this file: without a device every entry point fails.
 */
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "cg_host.h"
#include "cg_column_lean.h"

#define CG_CHECK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    snprintf(ctx->err, sizeof ctx->err, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    return CG_ERR_CUDA; } } while (0)

/* ============================== scan primitive ======================================== */
#define SCAN_THREADS 256
#define SCAN_ITEMS   16
#define SCAN_CHUNK   (SCAN_THREADS * SCAN_ITEMS)

struct OpSum { template <class T> __device__ static T apply(T a, T b) { return a + b; } };
struct OpMax { template <class T> __device__ static T apply(T a, T b) { return a > b ? a : b; } };

template <class T, class Op>
__device__ __forceinline__ T block_scan_incl(T v, T ident, T *sh /* >= 32 */, T *block_total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = Op::apply(u, v);
    }
    if (lane == 31) sh[w] = v;
    __syncthreads();
    if (w == 0) {
        T s = lane < (SCAN_THREADS / 32) ? sh[lane] : ident;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            T u = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s = Op::apply(u, s);
        }
        sh[lane] = s;
    }
    __syncthreads();
    if (w > 0) v = Op::apply(sh[w - 1], v);
    *block_total = sh[SCAN_THREADS / 32 - 1];
    __syncthreads();
    return v;
}

template <class T, class Op, class Load>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(Load ld, int64_t n, T ident, T *aggr) {
    __shared__ T sh[32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_CHUNK;
    T acc = ident;
#pragma unroll 4
    for (int k = 0; k < SCAN_ITEMS; k++) {
        int64_t i = base + (int64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n) acc = Op::apply(acc, ld(i));
    }
    T tot;
    block_scan_incl<T, Op>(acc, ident, sh, &tot);
    if (threadIdx.x == 0) aggr[blockIdx.x] = tot;
}

template <class T, class Op>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_aggr(T *aggr, int nb, T ident, T *total) {
    __shared__ T sh[32];
    T carry = ident;
    for (int b0 = 0; b0 < nb; b0 += SCAN_THREADS) {
        int b = b0 + threadIdx.x;
        T v = b < nb ? aggr[b] : ident;
        T tot;
        T inc = block_scan_incl<T, Op>(v, ident, sh, &tot);
        /* exclusive = carry (+) inclusive of the previous element */
        T prev = __shfl_up_sync(0xffffffffu, inc, 1);
        __shared__ T edge[SCAN_THREADS / 32];
        if ((threadIdx.x & 31) == 31) edge[threadIdx.x >> 5] = inc;
        __syncthreads();
        T ex;
        if (threadIdx.x == 0) ex = ident;
        else if ((threadIdx.x & 31) == 0) ex = edge[(threadIdx.x >> 5) - 1];
        else ex = prev;
        if (b < nb) aggr[b] = Op::apply(carry, ex);
        carry = Op::apply(carry, tot);
        __syncthreads();
    }
    if (threadIdx.x == 0 && total) *total = carry;
}

/* st(i, inclusive, exclusive) */
template <class T, class Op, class Load, class Store>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(Load ld, Store st, int64_t n, T ident, const T *aggr_excl) {
    __shared__ T sh[32];
    __shared__ T edge[SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_CHUNK;
    T carry = aggr_excl[blockIdx.x];
    for (int k = 0; k < SCAN_ITEMS; k++) {
        int64_t i = base + (int64_t)k * SCAN_THREADS + threadIdx.x;
        T v = i < n ? ld(i) : ident;
        T tot;
        T inc = block_scan_incl<T, Op>(v, ident, sh, &tot);
        T prev = __shfl_up_sync(0xffffffffu, inc, 1);
        if ((threadIdx.x & 31) == 31) edge[threadIdx.x >> 5] = inc;
        __syncthreads();
        T ex;
        if (threadIdx.x == 0) ex = ident;
        else if ((threadIdx.x & 31) == 0) ex = edge[(threadIdx.x >> 5) - 1];
        else ex = prev;
        if (i < n) st(i, Op::apply(carry, inc), Op::apply(carry, ex));
        carry = Op::apply(carry, tot);
        __syncthreads();
    }
}

/* ============================== functors ============================================== */
struct LdPileFlag { const int32_t *rspan; __device__ int32_t operator()(int64_t i) const { return rspan[i] != 0; } };
struct StJmap { int32_t *jmap; __device__ void operator()(int64_t i, int32_t, int32_t ex) const { jmap[i] = ex; } };
struct LdI32 { const int32_t *p; __device__ int32_t operator()(int64_t i) const { return p[i]; } };
struct LdI64 { const int64_t *p; __device__ int64_t operator()(int64_t i) const { return p[i]; } };
struct StI64Incl { int64_t *p; __device__ void operator()(int64_t i, int64_t inc, int64_t) const { p[i] = inc; } };
struct LdIslandFlag { const int64_t *gapraw; __device__ int32_t operator()(int64_t j) const { return j == 0 || gapraw[j] > 0; } };
struct StIsland {
    CgIsland *isl; const int64_t *ks; const int64_t *gapsum; const int64_t *gapraw;
    __device__ void operator()(int64_t j, int32_t, int32_t ex) const {
        if (j == 0 || gapraw[j] > 0) {
            CgIsland I; I.col_start = (int32_t)(ks[j] - ks[0] - gapsum[j]); I.tid = (int32_t)(ks[j] >> 32);
            I.pos_start = (int32_t)(ks[j] & 0xffffffff); I.pad = 0; isl[ex] = I;
        }
    }
};
struct LdPad8 { const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return ((int64_t)lq[i] + 7) & ~(int64_t)7; } };
struct LdNCig { const uint16_t *nc; __device__ int32_t operator()(int64_t i) const { return (int32_t)nc[i]; } };
struct StExcl64 { int64_t *p; __device__ void operator()(int64_t i, int64_t, int64_t ex) const { p[i] = ex; } };
struct StExcl32 { int32_t *p; __device__ void operator()(int64_t i, int32_t, int32_t ex) const { p[i] = ex; } };
/* ---- compact planes of the per-record arrays (cg_batch.meta_planes, include/crumble_gpu.h) -> tid / pos / l_qseq / n_cigar / cigar ---- */
struct LdD8 { const uint8_t *d; __device__ uint32_t operator()(int64_t i) const { const uint32_t v = d[i]; return v == 255u ? 0u : v; } };
struct StInclU32 { uint32_t *p; __device__ void operator()(int64_t i, uint32_t inc, uint32_t) const { p[i] = inc; } };
struct LdNcx { const uint8_t *nc8; __device__ int32_t operator()(int64_t i) const { const int v = nc8[i]; return v == 255 ? 0 : v; } };
/* running sum of the position deltas at every listed record */
__global__ void k_meta_gather(const uint64_t *__restrict__ pos_abs, int64_t n_abs, const uint32_t *__restrict__ S, uint32_t *__restrict__ absS) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_abs) absS[k] = S[pos_abs[k] >> 32];
}
/* last entry of a (record index << 32 | value) list whose index is <= i (entry 0 has index 0) */
__device__ __forceinline__ int64_t meta_find(const uint64_t *__restrict__ list, int64_t n, int64_t i) {
    int64_t lo = 0, hi = n;
    while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)(list[mid] >> 32) <= i) lo = mid; else hi = mid; }
    return lo;
}
__global__ void __launch_bounds__(256) k_meta_expand(int64_t n, const uint64_t *__restrict__ tid_runs, int64_t n_runs, const uint64_t *__restrict__ pos_abs, int64_t n_abs,
                                                    const uint32_t *__restrict__ absS, const uint8_t *__restrict__ lq8, const int32_t *__restrict__ lq_dict,
                                                    const uint8_t *__restrict__ nc8, int32_t *tid, int32_t *pos /* in: running sums, out: positions */,
                                                    int32_t *lq, uint16_t *nc) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    lq[i] = lq_dict[lq8[i]];
    const int v = nc8[i];
    nc[i] = (uint16_t)(v == 255 ? 1 : v);
    tid[i] = (int32_t)(uint32_t)tid_runs[meta_find(tid_runs, n_runs, i)];
    const int64_t k = meta_find(pos_abs, n_abs, i);
    pos[i] = (int32_t)((uint32_t)pos_abs[k] + ((uint32_t)pos[i] - absS[k]));
}
__global__ void __launch_bounds__(256) k_meta_cigar(int64_t n, const uint8_t *__restrict__ nc8, const int32_t *__restrict__ lq, const int32_t *__restrict__ coff,
                                                   const int32_t *__restrict__ xoff, const uint32_t *__restrict__ cigar_x, uint32_t *cigar,
                                                   int64_t cigar_cap, int64_t n_cigar_x) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int v = nc8[i];
    /* planes that do not add up stay inside the buffers here and are rejected by the totals check that follows */
    if ((int64_t)coff[i] + (v == 255 ? 1 : v) > cigar_cap || (v != 255 && (int64_t)xoff[i] + v > n_cigar_x)) return;
    if (v == 255) cigar[coff[i]] = (uint32_t)lq[i] << 4;                       /* one M of l_qseq bases */
    else for (int k = 0; k < v; k++) cigar[coff[i] + k] = cigar_x[xoff[i] + k];
}

struct LdEvFlag { const uint16_t *ev; uint16_t mask; __device__ int32_t operator()(int64_t c) const { return (ev[c] & mask) != 0; } };
struct StCompact { int32_t *out; const uint16_t *ev; uint16_t mask; __device__ void operator()(int64_t c, int32_t, int32_t ex) const { if (ev[c] & mask) out[ex] = (int32_t)c; } };
struct LdDepthCounted { const uint32_t *depth; const uint16_t *ev; __device__ int64_t operator()(int64_t c) const { return (ev[c] & CG_EV_COUNTED) ? (int64_t)depth[c] : 0; } };
struct LdCounted { const uint16_t *ev; __device__ int32_t operator()(int64_t c) const { return (ev[c] & CG_EV_COUNTED) != 0; } };
struct StI32Incl { int32_t *p; __device__ void operator()(int64_t i, int32_t inc, int32_t) const { p[i] = inc; } };
struct LdEvCount { const uint16_t *ev; __device__ int32_t operator()(int64_t c) const { return __popc(cg_event_bits(ev[c])); } };
struct StEvents {
    cg_bed_event *out; const uint16_t *ev; CgDev D; int64_t cap;
    __device__ void operator()(int64_t c, int32_t, int32_t ex) const {
        int bits = cg_event_bits(ev[c]);
        if (!bits) return;
        int is = cg_island_of(&D, (int)c);
        int tid = D.isl[is].tid, pos = D.isl[is].pos_start + ((int)c - D.isl[is].col_start);
        for (int t = 0; t < 5; t++) if (bits >> t & 1) { if (ex < cap) { cg_bed_event e; e.tid = tid; e.pos = pos; e.tag = t; out[ex] = e; } ex++; }
    }
};

/* ============================== kernels ================================================ */
__global__ void k_prep_read(const __grid_constant__ CgDev D) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < D.n_reads) cg_prep_read(&D, r);
}
__global__ void k_prep_keys(const __grid_constant__ CgDev D) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < D.n_reads) cg_prep_keys(&D, r);
}
/* raw gap per pileup read (needs the prefix max of end keys) */
__global__ void k_gap(const __grid_constant__ CgDev D, const int32_t *n_pile, int64_t *gapraw) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < *n_pile) gapraw[j] = cg_gap_of(&D, j);
}
__global__ void k_finish_read(const __grid_constant__ CgDev D, const int32_t *n_pile, int32_t *n_cols) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int np = *n_pile;
    if (j < np) {
        cg_finish_read(&D, j, D.ks[0]);
        if (j == np - 1) *n_cols = D.pmaxcol[j];
        if (D.glist && !(D.rd[j].rf & CG_RF_SIMPLE)) D.glist[atomicAdd(D.n_glist, 1)] = j;   /* k_cells_general's work list */
    }
    if (j == 0 && np == 0) *n_cols = 0;
}
/* device scalars -> MAPPED pinned host memory, written by the SMs: a cudaMemcpy would queue behind the bulk quality
 * downloads on the D2H copy engine and stall the host's per-slice sync by a whole chunk */
__global__ void k_publish(const int32_t *src, int32_t *dst_mapped, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst_mapped[i] = src[i];
    __threadfence_system();
}
__global__ void k_fill_i32(int32_t *p, int64_t n, int32_t v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void k_tile_index(const __grid_constant__ CgDev D) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < D.n_pile) cg_tile_index(&D, j);
}

/* the plain body, out of line: mode A (-q) columns are recomputed from the records */
__device__ __noinline__ CgColOut col_body_plain(const CgDev *D, int c) { return cg_column_body(D, c); }

/* ============================== column stage ============================================
 * Two kernels (cell format and per-lane bodies: cg_cells.h, cg_column_lean.h; DESIGN.md §3.1):
 *
 *  k_cells    read-major pre-pass: every pileup read is decoded ONCE into a row of 16-bit cells, one per reference column it covers,
 *             in groups of 8 cells = 16 bytes aligned to the dense column axis.  Four lanes per read, one group per lane and step:
 *             two aligned 64-bit quality loads and two 32-bit sequence loads funnel-shifted into place, the eight nt16 codes mapped
 *             to bases in one SIMD-within-register pass, quality x mapq through the effective-quality table.  Reads with a
 *             non-trivial CIGAR (a few percent) are left to k_cells_general: one warp per read, lane = column.
 *  k_column   one lane per dense column, one warp per 32-column tile, warps independent (no block barrier in the loop) and
 *             scheduled dynamically (a global tile counter), so a 1000x amplicon tile occupies one warp while the others move on.
 *             Per chunk of COL_R candidate reads: the tile's four groups of every row arrive by 16-byte cp.async (zero-filled where
 *             the read does not reach), double-buffered: the next chunk is in flight while this one is walked.  Each lane then walks
 *             its column down the rows (cg_rank_rows): one 16-bit LDS per cell, the per-quality constants from a 32-byte
 *             shared-memory row addressed by the cell's own bits, six in-order FP64 adds in rank space.  The tile ends with the
 *             lean finalisation (cg_cons_finalize_lean) and the column decisions (cg_column_finish). */
#define COL_WARPS    4
#ifndef COL_MINB
#define COL_MINB     5          /* resident blocks per SM the register allocation is sized for */
#endif
#ifndef COL_R
#define COL_R        60         /* rows per staged chunk: (COL_R + 1) x 64 B must hold the 15 x 32 doubles of the un-permute scratch */
#endif

struct __align__(16) ColSmem {
    uint16_t cell[COL_WARPS][2][COL_R + 1][32];     /* + 1: the column loop looks one row ahead */
    double rare[COL_WARPS][9][32];
    ColTabRow tab[104];
    unsigned cntw[COL_WARPS][32];
};
static_assert((COL_R + 1) * 64 >= 15 * 32 * 8, "un-permute scratch must fit one cell buffer");

__device__ __forceinline__ void cp_async16(void *dst_shared, const void *src, unsigned src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;\n" :: "r"((unsigned)__cvta_generic_to_shared(dst_shared)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

/* cell-matrix row records: ngrp per read -> exclusive scan -> first group of every row */
struct LdNgrp { const CgRead *rd; __device__ int64_t operator()(int64_t j) const { return (int64_t)cg_cell_ngroups(rd[j].col0, rd[j].span); } };
struct StCellRec {
    CgCellRec *crec; const CgRead *rd;
    __device__ void operator()(int64_t j, int64_t, int64_t ex) const {
        CgCellRec r; r.cpos8 = (uint32_t)ex; r.col0 = rd[j].col0; r.span = rd[j].span; r.ngrp = cg_cell_ngroups(r.col0, r.span);
        crec[j] = r;
    }
};

/* pileup reads [j_begin, j_end): 4 lanes per read */
__global__ void __launch_bounds__(256) k_cells(const __grid_constant__ CgDev D, int j_begin, int j_end) {
    const int j = j_begin + (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 2);
    if (j >= j_end) return;
    const uint4 h = __ldg(reinterpret_cast<const uint4 *>(D.rd + j));             /* off8, col0, span, pk */
    if (!(h.w & ((uint32_t)CG_RF_SIMPLE << 24))) return;                          /* k_cells_general */
    const CgCellRec cr = D.crec[j];
    CgRead q; q.off8 = h.x; q.col0 = (int32_t)h.y; q.span = (int32_t)h.z; q.mapq = (uint8_t)(h.w >> 16); q.rf = (uint8_t)(h.w >> 24);
    const int doB = D.P.min_qual_B != 0;
    uint4 *row = reinterpret_cast<uint4 *>(D.cells) + cr.cpos8;
    for (uint32_t k = threadIdx.x & 3; k < cr.ngrp; k += 4) {
        uint32_t o[4];
        cg_cells8_simple(&D, &q, 8 * (int)k - (q.col0 & 7), doB, o);
        row[k] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}
/* reads with a non-trivial CIGAR (listed by k_finish_read, a few percent of all): one warp per read, lane = column; the list is in no
 * particular order, a launch takes the entries inside its range of pileup reads */
__global__ void __launch_bounds__(256) k_cells_general(const __grid_constant__ CgDev D, int j_begin, int j_end) {
    const int lane = threadIdx.x & 31;
    const int nw = (int)((gridDim.x * (unsigned)blockDim.x) >> 5), total = *D.n_glist;
    const int doB = D.P.min_qual_B != 0;
    for (int gi = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5); gi < total; gi += nw) {
        const int g = D.glist[gi];
        if (g < j_begin || g >= j_end) continue;
        const CgRead q = D.rd[g];
        const CgCellRec cr = D.crec[g];
        uint16_t *row = D.cells + (size_t)cr.cpos8 * 8;
        const int n = (int)cr.ngrp * 8, lead = q.col0 & 7;
        for (int x = lane; x < n; x += 32) row[x] = (uint16_t)cg_cell_general(&D, &q, x - lead, doB);
    }
}

/* asm volatile: the load is issued where it is written (ahead of the column loop), not sunk to its first use */
__device__ __forceinline__ CgCellRec ld_crec(const CgCellRec *p) {
    CgCellRec r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];\n" : "=r"(r.cpos8), "=r"(r.col0), "=r"(r.span), "=r"(r.ngrp) : "l"(p));
    return r;
}

/* Stage rows [j0, j0 + n) of the read window for tile t into buf: lane l owns rows l and 32 + l (their records were loaded ahead) */
__device__ __forceinline__ void col_issue(const CgDev &D, uint16_t (*buf)[32], int tile_c0, int n, const CgCellRec &ra, const CgCellRec &rb, int lane) {
    const uint4 *cells = reinterpret_cast<const uint4 *>(D.cells);
#pragma unroll
    for (int s = 0; s < 2; s++) {
        const CgCellRec &r = s ? rb : ra;
        const int row = s * 32 + lane;
        if (row < n) {
            const int g0 = (tile_c0 - (r.col0 & ~7)) >> 3;                  /* the tile's first group inside this row (may be negative) */
#pragma unroll
            for (int p = 0; p < 4; p++) {
                const bool ok = (unsigned)(g0 + p) < r.ngrp;
                cp_async16(&buf[row][8 * p], cells + (ok ? (size_t)r.cpos8 + (size_t)(g0 + p) : (size_t)0), ok ? 16u : 0u);
            }
        }
    }
    cp_async_commit();
}

__global__ void __launch_bounds__(COL_WARPS * 32, COL_MINB) k_column(const __grid_constant__ CgDev D, int t_begin, int t_end, int *tile_counter) {
    __shared__ ColSmem S;
    const CgTables *T = D.T;
    const CgDevParams *P = &D.P;
    for (int i = threadIdx.x; i < 104; i += blockDim.x) {
        int q = i > 100 ? 100 : i;
        ColTabRow r; r.MM = T->MM[q]; r.hM = T->_M[q]; r.om = T->omq2p[q]; r.pad = 0;
        S.tab[i] = r;
    }
    S.cntw[threadIdx.x >> 5][threadIdx.x & 31] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int lean = P->min_qual_B != 0 && P->min_qual_A == 0;
    const uint32_t tab = (uint32_t)__cvta_generic_to_shared(S.tab);
    double *rare = &S.rare[w][0][lane];
    int depth_max = 0;
    unsigned long long items_ub = 0;
    const CgCellRec zrec = { 0u, 0, 0, 0u };

    /* Work items: (tile, chunk of its read window).  Tiles are claimed from a global counter THREE ahead: the atomic of tile i+3 is
     * issued when tile i starts and read when it ends, the window bounds of tile i+2 are loaded then and used a tile later, so
     * neither latency is ever waited for.  t = current tile, nt = next (bounds loaded), n2 = after that (bounds in flight). */
    int pend = 0;
    auto claim_issue = [&]() { if (lane == 0) pend = t_begin + atomicAdd(tile_counter, 1); };
    auto claim_read = [&]() -> int { return __shfl_sync(0xffffffffu, pend, 0); };
    claim_issue(); int t = claim_read();
    if (t >= t_end) return;
    claim_issue(); int nt = claim_read();
    claim_issue(); int n2 = claim_read();
    int lo = D.tile_lo[t], hi = D.tile_start[t + 1];
    int nlo = 0, nhi = 0, n2lo = 0, n2hi = 0;
    if (nt < t_end) { nlo = D.tile_lo[nt]; nhi = D.tile_start[nt + 1]; }
    if (n2 < t_end) { n2lo = D.tile_lo[n2]; n2hi = D.tile_start[n2 + 1]; }
    int j0 = lo, cur = 0;
    {   /* prologue: first chunk of the first tile */
        const int n = hi - j0 < COL_R ? hi - j0 : COL_R;
        const CgCellRec ra = lane < n ? ld_crec(D.crec + j0 + lane) : zrec, rb = 32 + lane < n ? ld_crec(D.crec + j0 + 32 + lane) : zrec;
        col_issue(D, S.cell[w][0], t * 32, n, ra, rb, lane);
    }
    CgRankAcc A;
    cg_rank_init<32>(&A, rare);
    claim_issue();
    for (;;) {
        const int n = hi - j0 < COL_R ? hi - j0 : COL_R;          /* rows of the current item (<= 0 for an empty window) */
        const bool last = j0 + COL_R >= hi;
        /* the item after this one: next chunk of the same tile, or the first chunk of the next tile */
        int xt = t, xj0 = j0 + COL_R, xhi = hi;
        if (last) { xt = nt; xj0 = nlo; xhi = nhi; }
        const bool more = xt < t_end;
        int xn = 0;
        CgCellRec ra = zrec, rb = zrec;
        if (more) {                                               /* its row records: requested now, used after this item's rows have been walked */
            xn = xhi - xj0 < COL_R ? xhi - xj0 : COL_R;
            if (lane < xn) ra = ld_crec(D.crec + xj0 + lane);
            if (32 + lane < xn) rb = ld_crec(D.crec + xj0 + 32 + lane);
        }
        cp_async_wait_all();
        __syncwarp();
        const uint16_t *col = &S.cell[w][cur][0][lane];
        if (n > 0) {
            cg_rank_peek<32>(&A, col, n);
            cg_rank_rows<32, 32>(&A, rare, col, n, tab);
        }
        if (more) col_issue(D, S.cell[w][cur ^ 1], xt * 32, xn, ra, rb, lane);
        if (last) {
            const int c = t * 32 + lane;
            CgColOut o; o.cnt = 0; o.n_plp = 0; o.items = 0;
            if (c < D.n_cols) {
                if (!lean) o = col_body_plain(&D, c);                                        /* mode A (-q): the plain body */
                else {
                    double *dump = reinterpret_cast<double *>(&S.cell[w][cur][0][0]) + lane;  /* the walked buffer is dead: lane-private scratch */
                    int rk[5];
                    CgConsAcc C;
                    cg_rank_of_bases(A.pi, A.nseen, rk);
                    cg_rank_dump_S<32, 32>(&A, rare, dump); cg_rank_unpermute_S<32>(dump, rk, C.S);
                    cg_rank_dump_C<32, 32>(&A, rare, dump); cg_rank_unpermute_C<32>(dump, rk, C.sumsC);
                    CgColStats st; st.cp = 0; st.n_plp = A.n_plp; st.n_skip = A.n_skip; st.low_mq = A.low_mq; st.had_indel = A.indel_cnt > 0; st.indel_cnt = A.indel_cnt;
                    st.clipped = A.clipped; st.n_overlap = A.n_overlap; st.ins_seen = A.ins_seen != 0;
                    CgCons cB;
                    cg_cons_finalize_lean(T, &C, A.n_plp - A.n_skip - A.n_none, A.nN, &cB);
                    o = cg_column_finish(&D, c, lo, hi, &st, (CgConsAcc *)0, &cB);
                }
            }
            /* counters: per warp in shared memory, flushed once when the warp runs out of tiles */
            unsigned un = __reduce_or_sync(0xffffffffu, o.cnt);
            while (un) {
                int b = __ffs(un) - 1; un &= un - 1;
                unsigned m = __ballot_sync(0xffffffffu, (o.cnt >> b) & 1);
                if (lane == 0) S.cntw[w][b] += __popc(m);
            }
            int mx = __reduce_max_sync(0xffffffffu, o.n_plp);
            depth_max = mx > depth_max ? mx : depth_max;
            items_ub += (unsigned)__reduce_add_sync(0xffffffffu, o.items);
            if (!more) break;
            cg_rank_init<32>(&A, rare);
            const int n3 = claim_read();
            t = nt; lo = nlo; hi = nhi; j0 = lo;
            nt = n2; nlo = n2lo; nhi = n2hi;
            n2 = n3;
            if (n2 < t_end) { n2lo = D.tile_lo[n2]; n2hi = D.tile_start[n2 + 1]; }
            claim_issue();
        } else j0 += COL_R;
        cur ^= 1;
    }
    __syncwarp();
    if (lane < CG_N_COUNTERS && S.cntw[w][lane]) atomicAdd(&D.counters[lane], (unsigned long long)S.cntw[w][lane]);
    if (lane == 0 && depth_max > 0) atomicMax(D.maxdepth, depth_max);
    if (lane == 0 && items_ub) atomicAdd(D.item_bound, items_ub);
}

/* Options outside the hand-tuned kernels (-S, -k/-K/-y, -N, -R; cg_params_generic): one column / one record per thread
 * through the plain bodies of cg_pipeline.h.  Same results as the reference, lower throughput. */
__global__ void __launch_bounds__(128) k_column_generic(const __grid_constant__ CgDev D, int t_begin, int t_end) {
    const int c = t_begin * 32 + blockIdx.x * blockDim.x + threadIdx.x;
    const int c_end = t_end * 32 < D.n_cols ? t_end * 32 : D.n_cols;
    CgColOut o; o.cnt = 0; o.n_plp = 0; o.items = 0;
    if (c < c_end) o = cg_column_body(&D, c);
    const unsigned it = (unsigned)__reduce_add_sync(0xffffffffu, o.items);
    if ((threadIdx.x & 31) == 0 && it) atomicAdd(D.item_bound, (unsigned long long)it);
    unsigned un = __reduce_or_sync(0xffffffffu, o.cnt);
    while (un) {
        const int b = __ffs(un) - 1; un &= un - 1;
        const unsigned m = __ballot_sync(0xffffffffu, (o.cnt >> b) & 1);
        if ((threadIdx.x & 31) == 0) atomicAdd(&D.counters[b], (unsigned long long)__popc(m));
    }
    const int mx = __reduce_max_sync(0xffffffffu, o.n_plp);
    if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(D.maxdepth, mx);
}
__global__ void __launch_bounds__(128) k_rewrite_generic(const __grid_constant__ CgDev D, int64_t rec_begin, int64_t rec_end) {
    const int64_t r = rec_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < rec_end) cg_rewrite(&D, r, D.n_flagged);
}

/* Flagged columns (had an indel / may open a keep window): the decisions of cg_flagged (cg_pipeline.h;
 * snp_score.c:1690-1762, 1775-1819) in two kernels.
 *  k_flagged    one WARP per column, lanes over the column's reads: indel count, insertion-size spectrum tests, and
 *               which reads trigger.  What the reference computes read by read is order-free except for two things,
 *               both recovered from the index of the LAST triggering read of each type (jI, jS): the running STR
 *               extents as seen by that read (PI/QI, PS/QS = min/max over the triggering reads up to it) and the
 *               column variable `indel`.  Every triggering read becomes one work item (flagged entry, read, query
 *               position, type) appended to the slice's item list; the list is unordered, its order does not matter.
 *  k_str_items  one THREAD per work item: mask_LC_regions + find_STR of one read at one column in the bit-parallel form
 *               (cg_mask_lc_bits, cg_core.h: the window as 2-bit codes in 64-bit words, period tests and extensions as word
 *               arithmetic, a 16-entry ring instead of the repeat list, scan cut at rpos + add + 15); the only loop left runs over
 *               candidate positions, so the lanes of a warp stay together; extents are folded into the trigger record with atomics. */
#define FL_WARPS 4
__global__ void __launch_bounds__(FL_WARPS * 32) k_flagged(const __grid_constant__ CgDev D, int k_begin, int k_end) {
    __shared__ int hist[FL_WARPS][104];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int gw = blockIdx.x * FL_WARPS + w, nw = gridDim.x * FL_WARPS;
    const CgDevParams *P = &D.P;
    const unsigned FULL = 0xffffffffu;
    for (int k = k_begin + gw; k < k_end; k += nw) {
        const int c = D.fcol[k];
        const int t = c >> 5;
        const int lo = D.tile_lo[t], hi = D.tile_start[t + 1];
        const uint16_t ev = D.ev[c];
        const int n_plp = (int)D.depth[c];
        const int had_indel = (ev & CG_EV_HADINDEL) != 0, lowscore = (ev & CG_EV_LOWSCORE) != 0, strall = (ev & CG_EV_STRALL) != 0;
        const int is = cg_island_of(&D, c);
        const int tid = D.isl[is].tid, pos = D.isl[is].pos_start + (c - D.isl[is].col_start);
        for (int i = lane; i < 104; i += 32) hist[w][i] = 0;
        __syncwarp();
        /* indel count, insertion-size spectrum, last triggering read of each type, `indel` */
        int indel_cnt = 0, jI = -1, jS = -1, maxsz = 0, nIq = 0;
        for (int j = lo + lane; j < hi; j += 32) {
            const CgRead q = D.rd[j]; CgCell cell;
            if (!cg_cell(&D, &q, c, &cell)) continue;
            if (cell.indel || cell.is_del) indel_cnt++;
            if (cell.is_refskip) continue;                                     /* 1696-1697 */
            const int is_indel = (cell.indel || cell.is_del);
            if (!cell.is_head && !cell.is_tail && (cell.indel > 0 || had_indel)) {     /* 1708-1713 */
                if (cell.indel > maxsz) maxsz = cell.indel;
                if (cell.indel >= 0) atomicAdd(&hist[w][cell.indel < 99 ? cell.indel : 99], 1);
            }
            if ((is_indel || strall) && lowscore) {                            /* 1718-1720 */
                if (is_indel) { jI = j; nIq++; } else jS = j;
            }
        }
        indel_cnt = __reduce_add_sync(FULL, indel_cnt); nIq = __reduce_add_sync(FULL, nIq);
        jI = __reduce_max_sync(FULL, jI); jS = __reduce_max_sync(FULL, jS); maxsz = __reduce_max_sync(FULL, maxsz);
        const int gate = indel_cnt >= n_plp * P->indel_fract;                  /* 1732: no STR search below the indel fraction */
        int vall = 0, vafter = 0;
        if (jI >= 0 || jS >= 0) {
            for (int j0 = lo; j0 < hi; j0 += 32) {
                const int j = j0 + lane;
                int emit = 0, rpos = 0, isi = 0;
                if (j < hi) {
                    const CgRead q = D.rd[j]; CgCell cell;
                    if ((unsigned)(c - q.col0) < (unsigned)q.span) D.r_bf[j] = 1;  /* every read of a trigger column is back-filled (1870-1879) */
                    if (cg_cell(&D, &q, c, &cell) && !cell.is_refskip) {
                        isi = (cell.indel || cell.is_del);
                        if (isi) {
                            const int v = (cell.indel < 0 ? -cell.indel : cell.indel) + cell.is_del;
                            if (v > vall) vall = v;
                            if (j > jS && v > vafter) vafter = v;
                        }
                        emit = gate && (isi || strall) && q.l_qseq > 0;        /* lowscore holds: a trigger exists */
                        rpos = cell.qpos + 1;
                    }
                }
                const unsigned em = __ballot_sync(FULL, emit);
                if (em) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd(D.n_sitem, __popc(em));
                    base = __shfl_sync(FULL, base, 0) + __popc(em & ((1u << lane) - 1u));
                    if (emit) {
                        if (base < D.sitem_cap) { CgStrItem it; it.k = k; it.j = j; it.rpos = rpos; it.is_indel = isi; D.sitem[base] = it; }
                        else *D.err = CG_ERR_OVERFLOW;                          /* cannot happen: the list is sized from the columns' own bound */
                    }
                }
            }
            vall = __reduce_max_sync(FULL, vall); vafter = __reduce_max_sync(FULL, vafter);
        }
        __syncwarp();
        if (lane == 0) {
            CgTrig tr; tr.tid = tid; tr.pos = pos; tr.col = c;
            tr.hasI = jI >= 0; tr.hasS = jS >= 0; tr.jI = jI; tr.jS = jS;
            tr.PI = tr.QI = tr.PS = tr.QS = tr.A = tr.B = pos;                /* k_str_items widens them */
            tr.indel = tr.hasS ? (vafter > 1 ? vafter : 1) : vall;             /* 1725-1730: a SNP-type trigger resets it to 1 */
            D.trig[k] = tr;
            uint32_t cnt = 0;
            if (nIq) cnt |= 1u << CG_CNT_INDEL_QUAL;                           /* 1762 */
            uint16_t ev_add = 0; int keep = 0;
            const int indel_sz = maxsz < 100 ? maxsz : 100;
            if (indel_sz) {                                                    /* 1777-1819 */
                int qd1 = 0, qd2 = 0, ov = 0;
                for (int i = 0; i <= indel_sz && i < 100; i++) {
                    int d = hist[w][i];
                    if (!d) continue;
                    ov += d;
                    if (qd1 < d) { qd2 = qd1; qd1 = d; } else if (qd2 < d) qd2 = d;
                }
                if ((ov - qd1 - qd2) > P->ins_len_perc * (ov + .1)) { ev_add |= CG_EV_INDEL_LEN; keep = 1; cnt |= 1u << CG_CNT_INS_LEN_PERC; }
                if ((double)ov < P->indel_ov_perc * n_plp) { ev_add |= CG_EV_INDEL_COV; keep = 1; cnt |= 1u << CG_CNT_INDEL_OV_PERC; }
            }
            if (tr.hasI || tr.hasS) ev_add |= CG_EV_TRIGGER;
            if (ev_add) D.ev[c] = (uint16_t)(ev | ev_add);
            if (keep) D.cb[c] |= CG_CB_KEEP;
            if (ev & CG_EV_REPLAY) cnt = 0;                                      /* counted by the previous call of the chain */
            while (cnt) { int b = __ffs(cnt) - 1; cnt &= cnt - 1; atomicAdd(&D.counters[b], 1ULL); }
        }
        __syncwarp();
    }
}

#ifndef STR_THREADS
#define STR_THREADS 128
#endif
__global__ void __launch_bounds__(STR_THREADS) k_str_items(const __grid_constant__ CgDev D) {
    __shared__ uint64_t W[16 * STR_THREADS];                                   /* the read window as 2-bit codes; word-major: lane-adjacent threads use adjacent words */
    __shared__ uint32_t ring[16 * STR_THREADS];                                /* live repeats (start, end) */
    const CgDevParams *P = &D.P;
    const int total = *D.n_sitem;
    for (int it = blockIdx.x * STR_THREADS + threadIdx.x; it < total; it += gridDim.x * STR_THREADS) {
        const CgStrItem im = D.sitem[it];
        CgTrig *tr = &D.trig[im.k];
        const int pos = tr->pos, jI = tr->jI, jS = tr->jS, j = im.j;
        const CgRead q = D.rd[j];
        const int phantom = (q.l_qseq & 1) ? (D.seq[(CG_OFF(&q) >> 1) + (q.l_qseq >> 1)] & 0xf)
                                           : (cg_cap_qual(D.qual[CG_OFF(&q)], P, D.T) >> 4);
        int lo_r = pos, hi_r = pos;                                            /* 1732-1739: the two calls are identical in effect */
        cg_mask_lc_bits<STR_THREADS, STR_THREADS>(D.seq + (CG_OFF(&q) >> 1), q.l_qseq, phantom, D.cigar + q.cig_off, q.n_cigar, q.pos,
                                                  im.rpos, im.is_indel ? P->iSTR_add : P->sSTR_add, W + threadIdx.x, ring + threadIdx.x, &lo_r, &hi_r);
        if (lo_r < pos) { atomicMin(&tr->A, lo_r); if (j <= jI) atomicMin(&tr->PI, lo_r); if (j <= jS) atomicMin(&tr->PS, lo_r); }
        if (hi_r > pos) { atomicMax(&tr->B, hi_r); if (j <= jI) atomicMax(&tr->QI, hi_r); if (j <= jS) atomicMax(&tr->QS, hi_r); }
    }
}

/* depth-average epochs (snp_score.c:1478-1491,1684-1687): sequential over contigs and the
 * ~n_cols/524289 halving points only; everything per-column is a prefix-sum lookup */
struct CgEpoch { int32_t col_begin; int32_t pad; int64_t td_base, tc_base, d_off, c_off; };
/* what a slice of columns hands to the next one: the contig whose running sums are open, and the prefix sums so far */
struct CgEpochCarry { int32_t tid, valid; int64_t td, tc, d_off, c_off; int64_t dsum_last; int32_t csum_last, n_ep; };

/* first index in [lo, hi) with csum[index] >= want, by the whole warp: 32-way splits instead of halving (the dependent global loads of
 * a one-thread binary search were most of this kernel's time, and the kernel sits on the serial path between region shards) */
__device__ __forceinline__ int epoch_lower_bound(const int32_t *csum, int lo, int hi, int64_t want) {
    const int lane = threadIdx.x & 31;
    while (hi - lo > 32) {
        const int step = (hi - lo + 31) >> 5;
        const int i = lo + lane * step;                      /* lane probes the first element of its part */
        const bool ge = i < hi ? (int64_t)csum[i] >= want : true;
        const unsigned m = __ballot_sync(0xffffffffu, ge);   /* parts whose first element already reaches want */
        const int f = m ? __ffs(m) - 1 : 32;                 /* the answer lies in part f - 1 (after its first element) or is part f's first element */
        if (f == 0) return lo;
        const int nlo = lo + (f - 1) * step + 1, nhi = f < 32 ? lo + f * step : hi;
        lo = nlo; hi = nhi < hi ? nhi : hi;
    }
    const int i = lo + lane;
    const unsigned m = __ballot_sync(0xffffffffu, i < hi ? (int64_t)csum[i] >= want : true);
    const int f = m ? __ffs(m) - 1 : 32;                     /* exactly 32 left and none reaches want: hi */
    return lo + f < hi ? lo + f : hi;
}

__global__ void k_epochs(const __grid_constant__ CgDev D, CgEpoch *ep, CgEpochCarry *carry, int cap, int cb, int ce) {
    if (blockIdx.x || threadIdx.x >= 32) return;             /* one warp: lanes take part in the searches, lane 0's state is the state */
    int ne = carry->n_ep;
    int is = cg_island_of(&D, cb);
    while (is < D.n_islands && D.isl[is].col_start < ce) {
        const int tid = D.isl[is].tid; int is2 = is;
        while (is2 + 1 < D.n_islands && D.isl[is2 + 1].tid == tid) is2++;
        const int c0 = D.isl[is].col_start > cb ? D.isl[is].col_start : cb;
        const int c1_true = (is2 + 1 < D.n_islands) ? D.isl[is2 + 1].col_start : D.n_cols;
        const int c1 = c1_true < ce ? c1_true : ce;
        int64_t d_off, c_off, td, tc; int s = c0;
        if (carry->valid && carry->tid == tid) {
            td = carry->td; tc = carry->tc; d_off = carry->d_off; c_off = carry->c_off;
            if (ne == 0) {                                  /* resumed from an earlier call (cg_process_window): its epoch list is gone */
                if (ne < cap) { CgEpoch e; e.col_begin = s; e.pad = 0; e.td_base = td; e.tc_base = tc; e.d_off = d_off; e.c_off = c_off; ep[ne] = e; }
                ne++;
            }
        } else {
            d_off = c0 ? D.dsum[c0 - 1] : 0; c_off = c0 ? D.csum[c0 - 1] : 0; td = tc = 0;
            if (ne < cap) { CgEpoch e; e.col_begin = s; e.pad = 0; e.td_base = td; e.tc_base = tc; e.d_off = d_off; e.c_off = c_off; ep[ne] = e; }
            ne++;
        }
        for (;;) {
            /* first column in [s,c1) whose counted index makes total_col exceed 2^20 */
            int64_t want = c_off + (1024 * 1024 + 1 - tc);
            int c = epoch_lower_bound(D.csum, s, c1, want);
            while (c < c1 && !((D.ev[c] & CG_EV_PROCESSED) && (D.ev[c] & CG_EV_COUNTED))) c++;
            if (c >= c1) break;
            td = (td + (D.dsum[c] - d_off)) >> 1;
            tc = (tc + ((int64_t)D.csum[c] - c_off)) >> 1;
            d_off = D.dsum[c]; c_off = D.csum[c]; s = c + 1;
            if (s >= c1_true) break;
            if (ne < cap) { CgEpoch e; e.col_begin = s; e.pad = 0; e.td_base = td; e.tc_base = tc; e.d_off = d_off; e.c_off = c_off; ep[ne] = e; }
            ne++;
            if (s >= c1) break;
        }
        carry->tid = tid; carry->valid = 1; carry->td = td; carry->tc = tc; carry->d_off = d_off; carry->c_off = c_off;
        is = is2 + 1;
    }
    carry->n_ep = ne;
    if (ce > cb) { carry->dsum_last = D.dsum[ce - 1]; carry->csum_last = D.csum[ce - 1]; }
    if (ne > cap) *D.err = CG_ERR_OVERFLOW;
}

__global__ void k_deep(const __grid_constant__ CgDev D, const CgEpoch *ep, const CgEpochCarry *carry, int cb, int ce) {
    int c = cb + blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t cnt = 0;
    if (c < ce && (D.ev[c] & CG_EV_PROCESSED)) {
        int lo = 0, hi = carry->n_ep - 1;
        while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (ep[mid].col_begin <= c) lo = mid; else hi = mid - 1; }
        const CgEpoch e = ep[lo];
        int64_t td = e.td_base + (D.dsum[c] - e.d_off), tc = e.tc_base + ((int64_t)D.csum[c] - e.c_off);
        cnt = cg_deep_test(&D, c, td, tc);
    }
    unsigned m = __ballot_sync(0xffffffffu, cnt != 0);
    if (m && (threadIdx.x & 31) == 0) atomicAdd(&D.counters[CG_CNT_OVER_DEPTH], (unsigned long long)__popc(m));
}

/* Keep-window chain (snp_score.c:1508-1511,1741-1755) in parallel.  The state (min_pos..max_pos2) is reset whenever
 * a trigger lies beyond max_pos2, so the chain falls into independent segments; a segment head is recognised without
 * knowing the state from an UPPER BOUND of max_pos2: windows only grow with the running STR maximum, so
 *   max_pos2 after trigger i  <=  U_i = max_{i' <= i} ceil( pos_i' + (Bmax_i' - pos_i') * mul + add ),  Bmax = prefix max of B
 * (both prefix maxima restricted to the contig by packing tid into the high word).  pos_k > U_{k-1} proves a reset at k;
 * each proven head then replays its segment sequentially (unproven resets inside are found by the replay itself). */
struct CgChainCarry { int64_t bkey, ukey; CgWin w; int32_t has, wtid; };    /* state after the last trigger of the previous slice (wtid = its contig) */
struct LdTrigB {
    const CgTrig *t; const CgChainCarry *cy;
    __device__ int64_t operator()(int64_t k) const {
        const CgTrig x = t[k];
        const int64_t v = ((int64_t)x.tid << 32) | (uint32_t)((x.hasI || x.hasS) ? (x.B > 0 ? x.B : 0) : 0);
        return v > cy->bkey ? v : cy->bkey;
    }
};
struct LdTrigU {
    const CgTrig *t; const int64_t *bmax; const CgChainCarry *cy; double mul, add;
    __device__ int64_t operator()(int64_t k) const {
        const CgTrig x = t[k];
        uint32_t u = 0;
        if (x.hasI || x.hasS) {
            const double M = (double)(uint32_t)bmax[k];
            double f = (double)x.pos + (M - x.pos) * mul + add + 2.0;
            if (f < 0) f = 0;
            u = f >= 2147483647.0 ? 0x7fffffffu : (uint32_t)f;
        }
        const int64_t v = ((int64_t)x.tid << 32) | u;
        return v > cy->ukey ? v : cy->ukey;
    }
};
__device__ __forceinline__ bool chain_is_head(const CgTrig &x, int k, int k_begin, const int64_t *umax, const CgChainCarry *cy) {
    const int64_t u = k == k_begin ? cy->ukey : umax[k - 1];
    return (int32_t)(u >> 32) != x.tid || (uint32_t)x.pos > (uint32_t)u;
}
/* umax is indexed by flagged entry (global); the thread of the slice's first entry also continues an open segment */
__global__ void k_chain(const __grid_constant__ CgDev D, const int64_t *umax, const CgChainCarry *cy, int k_begin, int k_end) {
    int k0 = k_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (k0 >= k_end) return;
    CgTrig t = D.trig[k0];
    CgWin w; cg_win_reset(&w);
    if (k0 == k_begin) {
        while (!(t.hasI || t.hasS)) { if (++k0 >= k_end) return; t = D.trig[k0]; }
        if (!chain_is_head(t, k0, k_begin, umax, cy) && cy->has) w = cy->w;
    } else if (!(t.hasI || t.hasS) || !chain_is_head(t, k0, k_begin, umax, cy)) return;
    for (int k = k0;;) {
        cg_win_step(&w, &t, &D.P);
        D.twin[k] = w;
        for (k++; k < k_end; k++) { t = D.trig[k]; if (t.hasI || t.hasS) break; }
        if (k >= k_end || chain_is_head(t, k, k_begin, umax, cy)) break;
    }
}
__global__ void k_chain_carry(const __grid_constant__ CgDev D, const int64_t *bmax, const int64_t *umax, CgChainCarry *cy, int k_begin, int k_end) {
    if (threadIdx.x || blockIdx.x || k_end <= k_begin) return;
    cy->bkey = bmax[k_end - 1]; cy->ukey = umax[k_end - 1];
    for (int k = k_end - 1; k >= k_begin; k--) {
        const CgTrig *t = &D.trig[k];
        if (t->hasI || t->hasS) { cy->w = D.twin[k]; cy->has = 1; cy->wtid = t->tid; break; }
    }
}
__global__ void k_paint(const __grid_constant__ CgDev D, int k_begin, int k_end) {
    int k = k_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (k < k_end) cg_paint(&D, k, k_end);
}
/* ---- chained calls (cg_process_window) ----
 * What one call hands to the next: both carries as they stand before the next call's first column, with the depth
 * carry's prefix-sum offsets rebased so that the next call's prefix sums may start from zero. */
struct CgSavedCarry { CgChainCarry cc; CgEpochCarry ec; };
__global__ void k_carry_save(const CgChainCarry *cc, const CgEpochCarry *ec, CgSavedCarry *out) {
    if (threadIdx.x || blockIdx.x) return;
    CgSavedCarry s; s.cc = *cc; s.ec = *ec;
    s.ec.d_off -= s.ec.dsum_last; s.ec.c_off -= s.ec.csum_last; s.ec.dsum_last = 0; s.ec.csum_last = 0; s.ec.n_ep = 0;
    *out = s;
}
__global__ void k_find_col(const __grid_constant__ CgDev D, int tid, int pos, int32_t *out) {
    if (threadIdx.x || blockIdx.x) return;
    *out = cg_find_col(&D, tid, pos);
}
/* the keep window the previous call left open stays active from this call's first column up to its max_pos2 */
__global__ void k_paint_carry(const __grid_constant__ CgDev D, const CgChainCarry *cy, int lo_tid, int lo_pos) {
    if (threadIdx.x || blockIdx.x) return;
    if (cy->has && cy->wtid == lo_tid && cy->w.min_pos != INT_MAX && cy->w.max_pos2 >= lo_pos) cg_paint_range(&D, lo_tid, lo_pos, cy->w.max_pos2);
}

/* Per-read quality rewrite.  A block owns RW_READS consecutive records; their quality strings, packed sequences
 * and the column bytes under them are three CONTIGUOUS ranges.  The column bytes (read at arbitrary offsets) come in
 * with one bulk async copy (TMA, cp.async.bulk + mbarrier) into shared memory; qualities and sequences are read
 * word by word, in order, in phase A2, so they go from global memory straight to registers (one step ahead), and the
 * rewritten words are collected in shared memory for the P-block pass and the bulk store.  Then
 *   phase A1 (thread per read):  whole-read facts from the staged column bytes (any keep_qual column, head column
 *            processed) and the word map: which read each staged 8-byte quality word belongs to;
 *   phase A2 (thread per WORD, all lanes busy whatever the read length): single-M reads without back-fill are
 *            rewritten SIMD-within-register, 8 bases per word: kept / match / binning are byte-parallel mask
 *            arithmetic on the 64-bit quality word, the 64-bit column word and the 8 expanded nt16 codes;
 *   phase A3 (warp per read): reads with indels, clips or back-fill are replayed op by op;
 *   phase B  (thread per read): P-block, a sequential greedy scan, in place, one 8-byte word per step where the word
 *            holds a single value (nearly all words after the rewrite), byte by byte elsewhere;
 *   phase C: one bulk async store of the block's output range (8-byte edges by the owning threads).
 * Blocks whose ranges do not fit the staging buffers (long reads) run the one-thread-per-read body (cg_rewrite). */
#ifndef RW_THREADS
#define RW_THREADS 128
#endif
#define RW_READS   RW_THREADS
#define RW_QCAP    (RW_READS * 168)     /* staged quality bytes (152 per padded 150-base read) */
#define RW_CCAP    3072                 /* staged column bytes */
#define RW_GORIG   176                  /* general path: reads up to this length keep their originals in shared memory */
#define RW_L_M     0x000fffffu          /* RwMeta.lk: L | kind << 20 | keep << 22 | init80 << 23 | tail_unreached << 24 */
#define RW_KIND_SH 20
#define RW_KEEP    (1u << 22)
#define RW_INIT    (1u << 23)
#define RW_TAILU   (1u << 24)

struct __align__(16) RwMeta { int32_t qoff, coff; uint32_t lk; int32_t j; };   /* offsets inside the staging buffers */
struct __align__(128) RwSmem {
    uint8_t q[RW_QCAP + 32];
    uint8_t c[RW_CCAP + 32];
    uint8_t wmap[RW_QCAP / 8 + 8];      /* read slot of every staged quality word, 0xff = none, 0xfe = read on the general path */
    RwMeta  m[RW_READS];
    uint8_t glist[RW_READS];            /* slots taking the general path */
    uint8_t gorig[RW_THREADS / 32][RW_GORIG];   /* general path: the read's original qualities, one buffer per warp */
    int     n_general;
    unsigned long long bar;
    long long red[4][4];
    long long rng[6];                   /* qa, qbytes, sa, sbytes, ca, cbytes (cbytes < 0: fallback) */
};

struct RwK { uint32_t QH, QL, cut, capadd; int mode; };   /* mode 0: mismatches keep their value, 1: -> qlow, 2: binary */

/* four quality bytes: byte-parallel form of cg_visit for reads whose bytes are < 0x80 and <= qcap */
__device__ __forceinline__ uint32_t rw_swar4(uint32_t q, uint32_t cb, uint32_t nib, uint32_t init80, const RwK &K) {
    const uint32_t kept = (((cb & 0x70707070u) + 0x70707070u) | init80) & 0x80808080u;     /* unproc | preserve | active | low mapq */
    const uint32_t m = nib & cb & 0x0f0f0f0fu;
    const uint32_t nzm = (m + 0x0f0f0f0fu) & 0x10101010u;                                    /* base inside the call set */
    const uint32_t h = nib & ((nib | 0x10101010u) - 0x01010101u) & 0x0f0f0f0fu;
    const uint32_t nzh = (h + 0x0f0f0f0fu) & 0x10101010u;                                    /* ambiguity code: never equal to a call */
    const uint32_t M = ((nzm & ~nzh) >> 4) * 0xffu;
    const uint32_t Kp = (kept >> 7) * 0xffu;
    uint32_t low = q;
    if (K.mode == 1) low = K.QL;
    else if (K.mode == 2) { const uint32_t G = (((q + K.cut) & 0x80808080u) >> 7) * 0xffu; low = (K.QH & G) | (K.QL & ~G); }
    return ((q & Kp) | (~Kp & ((K.QH & M) | (~M & low)))) & 0x7f7f7f7fu;
}

/* scalar form for the same 8 bytes (any byte >= 0x80 or above -U) */
__device__ __noinline__ uint64_t rw_visit8_scalar(uint64_t q8, uint64_t cb8, uint32_t s4, uint8_t init_or, int keep, const CgDevParams *P, const CgTables *T) {
    uint64_t out = 0;
    for (int k = 0; k < 8; k++) {
        const uint8_t qin = (uint8_t)(q8 >> (8 * k)), cbv = (uint8_t)(cb8 >> (8 * k));
        const int nib = (int)((s4 >> (8 * (k >> 1) + ((k & 1) ? 0 : 4))) & 0xf);
        const uint8_t oc = cg_cap_qual(qin, P, T);
        const uint8_t v = keep ? oc : cg_visit((uint8_t)(qin | init_or), cbv, oc, nib, P, T);
        out |= (uint64_t)(v & 0x7f) << (8 * k);
    }
    return out;
}

/* P-block (pblock, snp_score.c:803-834) on an 8-byte aligned string in shared memory, in run-length form: equal
 * neighbouring bytes cannot move the running min/max, so only the positions where the value CHANGES are visited
 * (chg = one bit per byte, built word-parallel by the whole block beforehand).  After the rewrite most of a read is
 * one value, so a thread steps through a handful of positions instead of 150 bytes, and the divergent part of the
 * warp's work shrinks with it.  Runs are filled with masked word stores, and only when the fill changes a byte. */
__device__ __forceinline__ void rw_fill(uint8_t *q, int j, int i, int mid) {
    const uint64_t mw = (uint64_t)(uint32_t)mid * 0x0101010101010101ULL;
    int k0 = j & ~7;
    if (k0 < j) {                                                  /* ragged first word: masked read-modify-write */
        uint64_t mask = ~0ULL << (8 * (j - k0));
        if (k0 + 8 > i) mask &= ~0ULL >> (8 * (k0 + 8 - i));
        uint64_t *p = reinterpret_cast<uint64_t *>(q + k0);
        *p = (*p & ~mask) | (mw & mask);
        k0 += 8;
    }
    for (; k0 + 8 <= i; k0 += 8) *reinterpret_cast<uint64_t *>(q + k0) = mw;   /* whole words: plain stores */
    if (k0 < i) {                                                  /* ragged last word */
        const uint64_t mask = ~0ULL >> (8 * (k0 + 8 - i));
        uint64_t *p = reinterpret_cast<uint64_t *>(q + k0);
        *p = (*p & ~mask) | (mw & mask);
    }
}
__device__ __forceinline__ void rw_pblock_rle(uint8_t *q, const uint8_t *chg, int len, int level, int qcap) {
    level *= 2;
    int qmin = q[0], qmax = qmin, j = 0;
    const int nw = (len + 7) >> 3;
    for (int g = 0; g < nw; g += 4) {
        uint32_t m = chg[g];
        if (g + 1 < nw) m |= (uint32_t)chg[g + 1] << 8;
        if (g + 2 < nw) m |= (uint32_t)chg[g + 2] << 16;
        if (g + 3 < nw) m |= (uint32_t)chg[g + 3] << 24;
        if (g == 0) m &= ~1u;
        const int rem = len - 8 * g;
        if (rem < 32) m &= (1u << rem) - 1u;
        while (m) {
            const int i = 8 * g + __ffs(m) - 1; m &= m - 1;
            const int v = q[i];
            int nmin = qmin < v ? qmin : v, nmax = qmax > v ? qmax : v;
            if (nmax - nmin > level) {
                int mid = (qmin + qmax) / 2;
                if (mid > qcap) mid = qcap;
                if (qmin != qmax || mid != qmin) rw_fill(q, j, i, mid);
                nmin = nmax = v; j = i;
            }
            qmin = nmin; qmax = nmax;
        }
    }
    if (qmin != qmax) rw_fill(q, j, len, (qmin + qmax) / 2);      /* the last run is not capped (832-833) */
}

__device__ __forceinline__ void rw_mbar_init(unsigned long long *bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" :: "r"((unsigned)__cvta_generic_to_shared(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void rw_bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 :: "r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void rw_mbar_expect(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rw_mbar_wait(unsigned long long *bar, uint32_t phase) {
    /* bounded: a bulk copy that never completes must end in a reported fault, not in a hung device */
    unsigned ok = 0;
    for (int spin = 0; spin < (1 << 22) && !ok; spin++)
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(phase) : "memory");
    if (!ok) __trap();
}

__global__ void __launch_bounds__(RW_THREADS) k_rewrite(const __grid_constant__ CgDev D, int64_t rec_begin, int64_t rec_end) {
    __shared__ RwSmem S;
    const CgDevParams *P = &D.P;
    const CgTables *T = D.T;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t base = rec_begin + (int64_t)blockIdx.x * RW_READS;
    const int nf = D.n_flagged;

    /* ---- phase 0: per-read facts, block ranges, bulk loads ---- */
    if (threadIdx.x == 0) { rw_mbar_init(&S.bar); S.n_general = 0; }
    int64_t off = 0; int L = 0, kind = 0, col0 = 0, span = 0, j = -1; uint32_t init_mq = 0, tail_unreached = 0;
    {
        const int64_t r = base + threadIdx.x;
        if (r < rec_end) { L = D.l_qseq[r]; off = D.off[r]; }
        if (L > 0) {
            kind = 1;
            if (D.rspan[r]) {
                j = D.jmap[r];
                const CgRead q = D.rd[j];
                col0 = q.col0; span = q.span;
                tail_unreached = (P->region_tid >= 0 && q.pos + q.span - 1 >= P->region_end);
                init_mq = q.mapq <= P->min_mqual;
                kind = ((q.rf & CG_RF_SIMPLE) && q.span == L && !D.r_bf[j]) ? 2 : 3;
            }
        }
        long long v0 = L > 0 ? off : LLONG_MAX, v1 = L > 0 ? off + L : LLONG_MIN;
        long long v2 = kind >= 2 ? col0 : LLONG_MAX, v3 = kind >= 2 ? (long long)col0 + span : LLONG_MIN;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            long long u0 = __shfl_xor_sync(0xffffffffu, v0, o), u1 = __shfl_xor_sync(0xffffffffu, v1, o);
            long long u2 = __shfl_xor_sync(0xffffffffu, v2, o), u3 = __shfl_xor_sync(0xffffffffu, v3, o);
            v0 = u0 < v0 ? u0 : v0; v1 = u1 > v1 ? u1 : v1; v2 = u2 < v2 ? u2 : v2; v3 = u3 > v3 ? u3 : v3;
        }
        if (lane == 0) { S.red[w][0] = v0; S.red[w][1] = v1; S.red[w][2] = v2; S.red[w][3] = v3; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long lo = LLONG_MAX, hi = LLONG_MIN, clo = LLONG_MAX, chi = LLONG_MIN;
        for (int i = 0; i < RW_THREADS / 32; i++) {
            lo = S.red[i][0] < lo ? S.red[i][0] : lo; hi = S.red[i][1] > hi ? S.red[i][1] : hi;
            clo = S.red[i][2] < clo ? S.red[i][2] : clo; chi = S.red[i][3] > chi ? S.red[i][3] : chi;
        }
        long long qa = 0, qb = 0, sa = 0, sb = 0, ca = 0, cbn = 0;
        if (hi > lo) {
            qa = lo & ~15LL; qb = ((hi + 15) & ~15LL) - qa;
            sa = (lo >> 1) & ~15LL; sb = ((((hi + 1) >> 1) + 15) & ~15LL) - sa;
            if (chi > clo) { ca = clo & ~15LL; cbn = ((chi + 15) & ~15LL) - ca; }
            if (qb > RW_QCAP + 16 || sb > RW_QCAP / 2 + 16 || cbn > RW_CCAP + 16) cbn = -1;
            else {
                rw_mbar_expect(&S.bar, (uint32_t)cbn);
                if (cbn > 0) rw_bulk_g2s(S.c, D.cb + ca, (uint32_t)cbn, &S.bar);
            }
        }
        S.rng[0] = qa; S.rng[1] = qb; S.rng[2] = sa; S.rng[3] = sb; S.rng[4] = ca; S.rng[5] = cbn;
        S.red[0][0] = lo; S.red[0][1] = hi;
    }
    __syncthreads();
    const long long qa = S.rng[0], qbytes = S.rng[1], ca = S.rng[4], cbytes = S.rng[5];
    if (qbytes == 0) return;                                   /* nothing but empty records */
    if (cbytes < 0) {                                          /* ranges too long for the staging buffers */
        const int64_t r = base + threadIdx.x;
        if (r < rec_end) cg_rewrite(&D, r, nf);
        return;
    }
    const int nwords = (int)(qbytes >> 3);
    for (int i = threadIdx.x; i < (nwords + 3) >> 2; i += RW_THREADS) reinterpret_cast<uint32_t *>(S.wmap)[i] = 0xffffffffu;
    __syncthreads();
    rw_mbar_wait(&S.bar, 0);

    /* ---- phase A1: whole-read facts, word map ---- */
    {
        const int qoff = (int)(off - qa), coff = (int)(col0 - ca);
        uint32_t lk = (uint32_t)L | ((uint32_t)kind << RW_KIND_SH) | (tail_unreached ? RW_TAILU : 0u);
        if (kind >= 2) {
            /* OR of the column bytes under the read: aligned words, ragged ends masked */
            const int a0 = coff & ~7, e = coff + span;
            uint32_t acc = 0;
            {   /* first word: bytes before the read's first column masked off (and those past its last one, for short reads) */
                uint64_t v = *reinterpret_cast<const uint64_t *>(S.c + a0);
                v &= ~0ULL << (8 * (coff - a0));
                if (a0 + 8 > e) v &= ~0ULL >> (8 * (a0 + 8 - e));
                acc = (uint32_t)v | (uint32_t)(v >> 32);
            }
            int a = a0 + 8;
            for (; a + 8 <= e; a += 8) { const uint2 v = *reinterpret_cast<const uint2 *>(S.c + a); acc |= v.x | v.y; }
            if (a < e) {                                         /* last word: bytes past the read's last column masked off */
                uint64_t v = *reinterpret_cast<const uint64_t *>(S.c + a);
                v &= ~0ULL >> (8 * (a + 8 - e));
                acc |= (uint32_t)v | (uint32_t)(v >> 32);
            }
            if ((acc & 0x80808080u) && !tail_unreached) lk |= RW_KEEP;          /* keep_qual on any covered column (1847, 1939-1940) */
            if (init_mq && !(S.c[coff] & CG_CB_UNPROC)) lk |= RW_INIT;          /* head column processed and mapq <= -m (1852-1859) */
        }
        RwMeta m; m.qoff = qoff; m.coff = coff; m.lk = lk; m.j = j;
        S.m[threadIdx.x] = m;
        if (kind == 1 || kind == 2) {
            const int w0 = qoff >> 3, nwr = (L + 7) >> 3;
            for (int i = 0; i < nwr; i++) S.wmap[w0 + i] = (uint8_t)threadIdx.x;
        } else if (kind == 3) {
            S.glist[atomicAdd(&S.n_general, 1)] = (uint8_t)threadIdx.x;
            const int w0 = qoff >> 3, nwr = (L + 7) >> 3;
            for (int i = 0; i < nwr; i++) S.wmap[w0 + i] = 0xfeu;              /* phase A2 leaves these words to phase A3 */
        }
    }
    __syncthreads();

    /* ---- phase A2: one staged quality word per thread and step ---- */
    RwK K;
    K.QH = (uint32_t)(P->qhigh & 0xff) * 0x01010101u; K.QL = (uint32_t)(P->qlow & 0xff) * 0x01010101u;
    K.mode = !P->reduce_qual ? 0 : (P->binary_qual ? 2 : 1);
    { int cq = P->qcutoff < 0 ? 0 : (P->qcutoff > 128 ? 128 : P->qcutoff); K.cut = (uint32_t)((128 - cq) & 0xff) * 0x01010101u; }
    K.capadd = P->qcap >= 127 ? 0u : (uint32_t)(127 - (P->qcap < 0 ? 0 : P->qcap)) * 0x01010101u;
    const bool swar_ok = !P->any_preserve_qual;
    const uint64_t *gq = reinterpret_cast<const uint64_t *>(D.qual + qa);      /* qa is a multiple of 16, and so is the buffer's base */
    const uint32_t *gs = reinterpret_cast<const uint32_t *>(D.seq + (qa >> 1));
    uint64_t q8n = 0; uint32_t s4n = 0;
    if ((int)threadIdx.x < nwords) { q8n = __ldg(gq + threadIdx.x); s4n = __ldg(gs + threadIdx.x); }
    for (int wi = threadIdx.x; wi < nwords; wi += RW_THREADS) {
        const uint32_t slot = S.wmap[wi];
        const uint64_t q8 = q8n; const uint32_t s4 = s4n;
        if (wi + RW_THREADS < nwords) { q8n = __ldg(gq + wi + RW_THREADS); s4n = __ldg(gs + wi + RW_THREADS); }   /* next step's words are in flight during this one */
        if (slot == 0xfeu) continue;
        if (slot == 0xffu) { *reinterpret_cast<uint64_t *>(S.q + wi * 8) = q8; continue; }   /* bytes of no record travel unchanged */
        const RwMeta m = S.m[slot];
        const int x0 = wi * 8 - m.qoff, nv = (int)(m.lk & RW_L_M) - x0;         /* nv >= 1 */
        const uint64_t vm = nv >= 8 ? ~0ULL : ((1ULL << (8 * nv)) - 1);
        uint64_t res;
        if (((m.lk >> RW_KIND_SH) & 3u) == 1u) res = q8 & 0x7f7f7f7f7f7f7f7fULL;  /* never in the pileup: strip bit 7 only (P-block follows) */
        else {
            /* column bytes [coff + x0, +8): two aligned words, funnel-shifted */
            const int cpos = m.coff + x0;
            const uint2 *cw = reinterpret_cast<const uint2 *>(S.c + (cpos & ~7));
            const uint2 w0 = cw[0], w1 = cw[1];
            const int sh = cpos & 7;
            const uint32_t Wa = (sh & 4) ? w0.y : w0.x, Wb = (sh & 4) ? w1.x : w0.y, Wc = (sh & 4) ? w1.y : w1.x;
            const uint32_t clo = __funnelshift_r(Wa, Wb, (sh & 3) * 8), chi = __funnelshift_r(Wb, Wc, (sh & 3) * 8);
            const int keep = (m.lk & RW_KEEP) != 0;
            const uint32_t qlo = (uint32_t)q8, qhi = (uint32_t)(q8 >> 32);
            const uint32_t bad = (((((qlo & 0x7f7f7f7fu) + K.capadd) | qlo) & (uint32_t)vm) | ((((qhi & 0x7f7f7f7fu) + K.capadd) | qhi) & (uint32_t)(vm >> 32))) & 0x80808080u;
            if (swar_ok && !bad) {
                if (keep) res = q8;                             /* memcpy of the (uncapped: <= -U) originals, snp_score.c:1939-1940 */
                else {
                    const uint32_t init80 = (m.lk & RW_INIT) ? 0x80808080u : 0u;
                    const uint32_t t0 = __byte_perm(s4, 0, 0x1100), t1 = __byte_perm(s4, 0, 0x3322);
                    const uint32_t n0 = ((t0 >> 4) & 0x000f000fu) | (t0 & 0x0f000f00u), n1 = ((t1 >> 4) & 0x000f000fu) | (t1 & 0x0f000f00u);
                    res = (uint64_t)rw_swar4(qlo, clo, n0, init80, K) | ((uint64_t)rw_swar4(qhi, chi, n1, init80, K) << 32);
                }
            } else {
                res = rw_visit8_scalar(q8, (uint64_t)clo | ((uint64_t)chi << 32), s4, (m.lk & RW_INIT) ? 0x80 : 0, keep, P, T);
            }
        }
        *reinterpret_cast<uint64_t *>(S.q + wi * 8) = (res & vm) | (q8 & ~vm);
    }

    /* ---- phase A3: general path, warp per read: replay inside the slot.  The slot still holds the staged originals (phase A2
     * skips these reads); they move to the warp's side buffer first, and bases come from the staged sequence, so the replay's
     * inner loops touch shared memory only (reads longer than the side buffer take originals from global memory). ---- */
    for (int gi = w; gi < S.n_general; gi += RW_THREADS / 32) {
        const RwMeta m = S.m[S.glist[gi]];
        uint8_t *sl = S.q + m.qoff;
        const int Lr = (int)(m.lk & RW_L_M);
        const uint8_t *cbp = S.c + m.coff;
        const uint8_t init_or = (m.lk & RW_INIT) ? 0x80 : 0;
        const int keep = (m.lk & RW_KEEP) != 0;
        const CgRead q = D.rd[m.j];
        const uint32_t *cig = D.cigar + q.cig_off;
        const uint8_t *qin = D.qual + (qa + m.qoff);
        const uint8_t *ss = D.seq + ((qa + m.qoff) >> 1);            /* qoff is a multiple of 8 */
        if (Lr <= RW_GORIG) {
            __syncwarp();
            for (int x = lane; x < ((Lr + 7) & ~7); x += 32) S.gorig[w][x] = qin[x];      /* with the padding of the last word */
            qin = S.gorig[w];
        }
        __syncwarp();
        for (int x = lane; x < ((Lr + 7) & ~7); x += 32) sl[x] = x < Lr ? (uint8_t)(qin[x] | init_or) : qin[x];   /* the slot starts empty: padding travels unchanged */
        __syncwarp();
#define RW_NIB(x_) ((ss[(x_) >> 1] >> ((~(x_) & 1) << 2)) & 0xf)
        int c = 0, y = 0;
        for (int k = 0; k < q.n_cigar; k++) {
            const int op = cg_cig_op(cig[k]), l = cg_cig_len(cig[k]);
            if (cg_is_mop(op)) {
                for (int ii = lane; ii < l; ii += 32) {
                    int x = y + ii;
                    if (x < Lr) sl[x] = cg_visit(sl[x], cbp[c + ii], cg_cap_qual(qin[x], P, T), RW_NIB(x), P, T);
                }
                c += l; y += l;
            } else if (op == 2 || op == 3) {
                if (lane == 0 && y < Lr) {
                    uint8_t oc = cg_cap_qual(qin[y], P, T); int nib = RW_NIB(y); uint8_t v = sl[y];
                    for (int ii = 0; ii < l; ii++) v = cg_visit(v, cbp[c + ii], oc, nib, P, T);
                    sl[y] = v;
                }
                c += l;
            } else if (op == 1 || op == 4) y += l;
            __syncwarp();
        }
#undef RW_NIB
        if (D.r_bf[m.j]) {
            for (int k = cg_trig_lower_bound(&D, nf, q.col0); k < nf && D.fcol[k] < q.col0 + q.span; k++) {
                const CgTrig *t = &D.trig[k];
                if (!(t->hasI || t->hasS)) continue;
                CgCell cell;
                if (!cg_cell(&D, &q, t->col, &cell)) continue;
                int xs = cg_ref2query_pos(cig, q.n_cigar, q.pos, D.twin[k].min_pos2);
                for (int x = xs + lane; x <= cell.qpos && x < Lr; x += 32) sl[x] = (uint8_t)(cg_cap_qual(qin[x], P, T) | 0x80);
            }
            __syncwarp();
        }
        for (int x = lane; x < Lr; x += 32) sl[x] = (keep ? cg_cap_qual(qin[x], P, T) : sl[x]) & 0x7f;
    }
    __syncthreads();
    /* ---- phase B: P-block: change bits of every staged word (word map storage reused), then thread per read ---- */
    if (P->pblock) {
        if (!P->any_preserve_qual) {
            for (int wi = threadIdx.x; wi < nwords; wi += RW_THREADS) {
                const uint2 v = *reinterpret_cast<const uint2 *>(S.q + wi * 8);
                const uint32_t prev = wi ? S.q[wi * 8 - 1] : 0u;
                const uint32_t dx = v.x ^ ((v.x << 8) | prev), dy = v.y ^ __funnelshift_l(v.x, v.y, 8);
                const uint32_t tx = ((((dx & 0x7f7f7f7fu) + 0x7f7f7f7fu) | dx) & 0x80808080u) >> 7;
                const uint32_t ty = ((((dy & 0x7f7f7f7fu) + 0x7f7f7f7fu) | dy) & 0x80808080u) >> 7;
                S.wmap[wi] = (uint8_t)(((tx * 0x01020408u) >> 24) | (((ty * 0x01020408u) >> 24) << 4));
            }
            __syncthreads();
        }
        const RwMeta m = S.m[threadIdx.x];
        if ((m.lk >> RW_KIND_SH) & 3u) {
            if (P->any_preserve_qual) cg_pblock_t<1>(S.q + m.qoff, (int)(m.lk & RW_L_M), P->pblock, P->qcap, T);
            else rw_pblock_rle(S.q + m.qoff, S.wmap + (m.qoff >> 3), (int)(m.lk & RW_L_M), P->pblock, P->qcap);
        }
    }
    /* ---- phase C: the block's output range ---- */
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    __syncthreads();
    {
        const long long lo = S.red[0][0], hi8 = (S.red[0][1] + 7) & ~7LL;            /* 8-aligned: record offsets are */
        const long long ilo = (lo + 15) & ~15LL, ihi = hi8 & ~15LL;
        if (threadIdx.x == 0 && ihi > ilo) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n"
                         :: "l"(D.qual_out + ilo), "r"((unsigned)__cvta_generic_to_shared(S.q + (ilo - qa))), "r"((uint32_t)(ihi - ilo)) : "memory");
            asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
        }
        if (threadIdx.x == 1 && lo < ilo && lo < hi8) *(uint64_t *)(D.qual_out + lo) = *(const uint64_t *)(S.q + (lo - qa));
        if (threadIdx.x == 2 && ihi < hi8 && ihi >= ilo) *(uint64_t *)(D.qual_out + ihi) = *(const uint64_t *)(S.q + (ihi - qa));
        if (threadIdx.x == 0 && ihi > ilo) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    }
}
__global__ void k_dump_flags(const __grid_constant__ CgDev D) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= D.n_cols) return;
    cg_column z = D.coldump[c];
    if (z.tid < 0) return;
    uint8_t cb = D.cb[c]; uint16_t ev = D.ev[c];
    if (cb & CG_CB_ACTIVE) z.flags |= 4;
    if (cb & CG_CB_KEEP) z.flags |= 2;
    if (ev & CG_EV_TRIGGER) z.flags |= 16;
    if (ev & CG_EV_HADINDEL) z.flags |= 32;
    z.flags |= (uint32_t)(ev & CG_EV_BEDMASK) << 8;
    D.coldump[c] = z;
}

/* ---- compact planes (cg_batch.seq2 / qualp, include/crumble_gpu.h) -> the 4-bit / 8-bit working arrays --------------------------
 * One thread per 8 positions [8g, 8g + 8): 2 bytes of 2-bit bases become 4 bytes of nt16 codes (high nibble first), 2 or 4 bytes of
 * dictionary codes become 8 quality bytes through byte permutes of the dictionary held in registers. */
struct CgDict { uint32_t w[4]; };
__global__ void __launch_bounds__(256) k_unpack(const uint8_t *__restrict__ seq2, const uint8_t *__restrict__ qualp, uint8_t *__restrict__ seq, uint8_t *__restrict__ qual,
                                                int64_t g_begin, int64_t g_end, int bits, const __grid_constant__ CgDict dict) {
    const int64_t g = g_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= g_end) return;
    const uint32_t s = reinterpret_cast<const uint16_t *>(seq2)[g];
    uint32_t out = 0;
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
        const uint32_t hi = 1u << ((s >> (2 * k)) & 3u), lo = 1u << ((s >> (2 * k + 2)) & 3u);   /* nt16: A=1 C=2 G=4 T=8 */
        out |= ((hi << 4) | lo) << (4 * k);
    }
    reinterpret_cast<uint32_t *>(seq)[g] = out;
    if (bits == 2) {
        const uint32_t c = reinterpret_cast<const uint16_t *>(qualp)[g];
        /* 2-bit codes -> byte selectors of one permute per four positions */
        const uint32_t x0 = c & 0xffu, x1 = c >> 8;
        const uint32_t s0 = ((x0 & 0xc0u) << 6) | ((x0 & 0x30u) << 4) | ((x0 & 0x0cu) << 2) | (x0 & 0x03u);
        const uint32_t s1 = ((x1 & 0xc0u) << 6) | ((x1 & 0x30u) << 4) | ((x1 & 0x0cu) << 2) | (x1 & 0x03u);
        reinterpret_cast<uint2 *>(qual)[g] = make_uint2(__byte_perm(dict.w[0], 0, s0), __byte_perm(dict.w[0], 0, s1));
    } else if (bits == 4) {
        const uint32_t c = reinterpret_cast<const uint32_t *>(qualp)[g];
        uint32_t r[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t x = (c >> (16 * h)) & 0xffffu;                 /* four 4-bit codes */
            const uint32_t sel = x & 0x7777u, hi8 = x & 0x8888u;           /* selector inside an 8-byte half, and which half */
            const uint32_t a = __byte_perm(dict.w[0], dict.w[1], sel), b = __byte_perm(dict.w[2], dict.w[3], sel);
            /* byte mask from bit 3 of every nibble */
            const uint32_t m = ((hi8 >> 3) & 1u) * 0xffu | ((hi8 >> 7) & 1u) * 0xff00u | ((hi8 >> 11) & 1u) * 0xff0000u | ((hi8 >> 15) & 1u) * 0xff000000u;
            r[h] = (a & ~m) | (b & m);
        }
        reinterpret_cast<uint2 *>(qual)[g] = make_uint2(r[0], r[1]);
    }
}
/* the positions whose base is not A/C/G/T: patch the nibble (two exceptions may share a byte, never a nibble) */
__global__ void __launch_bounds__(256) k_unpack_exc(const uint64_t *__restrict__ exc, int64_t e_begin, int64_t e_end, uint8_t *seq) {
    const int64_t i = e_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e_end) return;
    const uint64_t v = exc[i];
    const int64_t pos = (int64_t)(v >> 4); const uint32_t code = (uint32_t)(v & 15u);
    const int64_t byte = pos >> 1;
    uint32_t *word = reinterpret_cast<uint32_t *>(seq + (byte & ~(int64_t)3));
    const int sh = (int)(byte & 3) * 8 + ((pos & 1) ? 0 : 4);
    atomicAnd(word, ~(0xfu << sh));
    atomicOr(word, code << sh);
}

/* ============================== context ================================================ */
/* the staging loads of k_column / k_rewrite read whole aligned words around a read: pad both ends of seq and qual */
#define CG_FRONT_PAD 256
struct dbuf { void *p; size_t cap; };

#define CG_MAX_CHUNKS 32
struct CgBounds { int64_t rb[CG_MAX_CHUNKS]; int32_t n; };
struct CgSlice { int t0, t1, c0, c1, jb, je, kb, ke, chunk, save_after; int64_t r0, r1; };   /* see slice_A / slice_B */

/* The device scalar block (b_scal): the chain's scalars and counters, both carries, the chunk bounds and a scratch carry; run_prep
 * zeroes it.  Its head is mirrored into mapped pinned memory (cg_ctx::h_dims), copied there at the host's synchronisations or written
 * there directly by k_publish and k_find_col.  Every field keeps a fixed byte offset, checked below. */
struct CgScalHead {
    int32_t n_pile;               /* pileup reads */
    int32_t n_cols;
    int32_t n_islands;
    int32_t n_flagged;            /* of the slice */
    int32_t maxdepth;
    int32_t err;                  /* device-side error code */
    int32_t n_events;             /* BED events */
    int32_t pad7;
    int32_t beyond;               /* CgDev::beyond */
    int32_t window_max;           /* most candidate reads of one tile */
    int32_t n_sitem;              /* STR items of the slice */
    int32_t next_col;             /* in the mirror only: the next call's first column (k_find_col) */
    int64_t qual_total;           /* a packed batch: padded quality bytes */
    int32_t cigar_total;          /* a packed batch: CIGAR operations */
    int32_t pad15;
    int64_t cell_groups;          /* cell matrix */
    struct { int32_t tile_counter, pad; unsigned long long item_bound; } slice;   /* reset before each column stage: k_column's tile counter, STR item bound */
    int32_t pad22[2];
};
struct CgScalars {
    CgScalHead h;
    int32_t n_glist;              /* reads with a non-trivial CIGAR */
    int32_t pad25[7];
    unsigned long long counters[CG_N_COUNTERS];
    char pad_counters[512 - 128 - 8 * CG_N_COUNTERS];
    CgChainCarry chain;
    char pad_chain[640 - 512 - sizeof(CgChainCarry)];
    CgEpochCarry epoch;
    char pad_epoch[768 - 640 - sizeof(CgEpochCarry)];
    int64_t bounds[3 * CG_MAX_CHUNKS];                     /* k_bounds */
    char pad_bounds[1600 - 768 - 8 * 3 * CG_MAX_CHUNKS];
    CgChainCarry chain_import;    /* cg_shard_end paints from the carry the shard imported */
    char pad_import[1664 - 1600 - sizeof(CgChainCarry)];
    struct CgStreamScal {         /* cg_stream_device: the cut of the call and what it holds back, read at its one synchronisation */
        CgStreamRed red;
        CgStreamCut cut;
        int64_t held_n, held_padded, held_cig, held_qual, held_seq;   /* totals of the keep-flag scans */
    } stream;
    char pad_end[2048 - 1664 - sizeof(CgStreamScal)];
};
#define CG_SCAL_AT(f, off) static_assert(offsetof(CgScalars, f) == (off), "scalar block: " #f " must stay at byte " #off)
CG_SCAL_AT(h.n_pile, 0); CG_SCAL_AT(h.n_cols, 4); CG_SCAL_AT(h.n_islands, 8); CG_SCAL_AT(h.n_flagged, 12);
CG_SCAL_AT(h.maxdepth, 16); CG_SCAL_AT(h.err, 20); CG_SCAL_AT(h.n_events, 24); CG_SCAL_AT(h.beyond, 32);
CG_SCAL_AT(h.window_max, 36); CG_SCAL_AT(h.n_sitem, 40); CG_SCAL_AT(h.next_col, 44); CG_SCAL_AT(h.qual_total, 48);
CG_SCAL_AT(h.cigar_total, 56); CG_SCAL_AT(h.cell_groups, 64); CG_SCAL_AT(h.slice.tile_counter, 72); CG_SCAL_AT(h.slice.item_bound, 80);
CG_SCAL_AT(n_glist, 96); CG_SCAL_AT(counters, 128); CG_SCAL_AT(chain, 512); CG_SCAL_AT(epoch, 640); CG_SCAL_AT(bounds, 768);
CG_SCAL_AT(chain_import, 1600); CG_SCAL_AT(stream, 1664);
#undef CG_SCAL_AT
static_assert(sizeof(CgScalHead) == 96, "the mirrored head is 24 int32 slots");
static_assert(sizeof(CgScalars) == 2048, "scalar block size");

struct cg_ctx {
    int device; cudaStream_t stream; int own_stream;
    cg_params params; CgTables *hT; CgTables *dT;
    char err[512];
    /* device buffers */
    dbuf b_tid, b_pos, b_flag, b_mapq, b_lq, b_nc, b_off, b_coff, b_cigar, b_seq, b_qual, b_qout;
    dbuf b_jmap, b_rspan, b_rd, b_ks, b_ke, b_gap, b_gapraw, b_pmax, b_orig, b_rbf, b_glist;
    dbuf b_tlo, b_tstart, b_isl, b_cb, b_ev, b_depth, b_dump, b_dsum, b_csum, b_fcol, b_trig, b_twin;
    dbuf b_aggr, b_scal, b_scratch, b_epoch, b_events, b_chain, b_items, b_bed, b_bedpm, b_crec, b_cells, b_seq2, b_qualp, b_exc;
    dbuf b_truns, b_pabs, b_pd8, b_lq8, b_nc8, b_cigx, b_lqd, b_xoff, b_absS;   /* compact planes of the per-record arrays and what their expansion needs */
    dbuf b_qsrc, b_ssrc, b_dvsum;  /* cg_process_device: where each record starts in the caller's arrays, the sums checked on the host */
    /* cg_stream_device: the held store (records kept for later calls, in the padded working layout) and the keep-flag scans that fill it */
    dbuf b_htid, b_hpos, b_hflag, b_hmapq, b_hlq, b_hnc, b_hcig, b_hqual, b_hseq, b_keep, b_kidx, b_koff, b_kcig;
    int st_open, st_unplaced, st_has_key; uint64_t st_kmax;            /* an open stream; the sort order across its chunks */
    int64_t st_n, st_e0, st_padded, st_cig, st_qual, st_seq;          /* held records (the first st_e0 already emitted) and their sizes */
    cg_window st_win;                                                  /* first / lo_tid / lo_pos / cnt_pos of the next call */
    CgScalars::CgStreamScal *h_stream;                                 /* pinned */
    int has_meta; int64_t n_truns, n_pabs, n_cigx;
    int generic;                  /* cg_params_generic(): column and rewrite stages through the plain bodies */
    /* host mirrors */
    CgScalHead *d_hdims;          /* device alias of h_dims (mapped pinned memory) */
    CgScalHead *h_dims;           /* pinned, mapped: the head of the scalar block */
    unsigned long long *h_counters;
    CgDev D;
    int resident; int dump_columns;
    int64_t qual_bytes, cigar_total, events_cap_dev;
    int need_depth, epoch_cap, nf_total;
    int64_t chunk_bytes;
    int win_on, have_saved, depth_matters; cg_window win; dbuf b_saved;
    int has_planes, qual_bits; CgDict dict;                                     /* compact planes travel instead of seq / qual */
    int packed, offsets_ready; int64_t h2d_bytes;                           /* offsets rebuilt on the device; bytes copied up by the last call */       /* chained calls: this call's window, the carries of the previous one */
    cudaStream_t s_h2d, s_d2h; cudaEvent_t ev_up[32], ev_done[32], ev_misc;
    char h_carry_init[64];
    char *h_carry_io;                                           /* pinned: [0, 128) the state a shard imported, [128, 256) the one it exports */
    CgSlice sl[2 * CG_MAX_CHUNKS + 2]; int n_sl, shard_state, shard_next, shard_save_end, shard_timed; const cg_batch *shard_in;
    cudaEvent_t ev[CG_N_TIMERS][2];
    float ms[CG_N_TIMERS];
    int64_t launches;
};

/* while a stream is open (cg_stream_device) the working buffers, the window state and the stream belong to it */
static int stream_busy(cg_ctx *ctx) {
    if (!ctx->st_open) return 0;
    snprintf(ctx->err, sizeof ctx->err, "a stream is open on this context: finish it with cg_stream_device(last = 1) first");
    return CG_ERR_STATE;
}

static int ensure(cg_ctx *ctx, dbuf *b, size_t bytes) {
    if (bytes <= b->cap) return 0;
    if (b->p) cudaFree(b->p);
    size_t nc = bytes + (bytes >> 3) + 256;
    b->p = NULL; b->cap = 0;
    CG_CHECK(cudaMalloc(&b->p, nc));
    b->cap = nc;
    return 0;
}

/* grow a buffer whose contents must survive (lists appended to slice after slice) */
static int ensure_keep(cg_ctx *ctx, dbuf *b, size_t bytes) {
    if (bytes <= b->cap) return 0;
    size_t nc = bytes * 2 + 4096;
    void *np_ = NULL;
    CG_CHECK(cudaMalloc(&np_, nc));
    if (b->p) {
        CG_CHECK(cudaMemcpyAsync(np_, b->p, b->cap, cudaMemcpyDeviceToDevice, ctx->stream));
        CG_CHECK(cudaStreamSynchronize(ctx->stream));
        cudaFree(b->p);
    }
    b->p = np_; b->cap = nc;
    return 0;
}

static void *pinned_alloc(size_t n) { void *p = NULL; if (cudaHostAlloc(&p, n, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return NULL; } return p; }
static void pinned_free(void *p) { cudaFreeHost(p); }

extern "C" int cg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static void install_hooks(void) {
    if (cg_device_count() > 0) { cg_pinned_alloc_hook = pinned_alloc; cg_pinned_free_hook = pinned_free; }
}

extern "C" int cg_enable_pinned(void) { install_hooks(); return cg_pinned_alloc_hook != NULL; }

extern "C" int cg_set_params(cg_ctx *ctx, const cg_params *p) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    const char *why = NULL;
    int e = cg_params_check(p, &why);
    if (e) { snprintf(ctx->err, sizeof ctx->err, "not implemented on the device path: %s", why); return e; }
    ctx->params = *p;
    ctx->generic = cg_params_generic(p);
    cg_tables_init(ctx->hT, p);
    CG_CHECK(cudaMemcpyAsync(ctx->dT, ctx->hT, sizeof(CgTables), cudaMemcpyHostToDevice, ctx->stream));
    if (p->nbed > 0) {                                          /* -R regions and the prefix max cg_bed_hit searches */
        int64_t *pm = (int64_t *)malloc(sizeof(int64_t) * (size_t)p->nbed);
        if (!pm) return CG_ERR_NOMEM;
        cg_bed_prefix_max(p->bed, p->nbed, pm);
        if ((e = ensure(ctx, &ctx->b_bed, sizeof(cg_bed_reg) * (size_t)p->nbed)) || (e = ensure(ctx, &ctx->b_bedpm, sizeof(int64_t) * (size_t)p->nbed))) { free(pm); return e; }
        cudaMemcpyAsync(ctx->b_bed.p, p->bed, sizeof(cg_bed_reg) * (size_t)p->nbed, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(ctx->b_bedpm.p, pm, sizeof(int64_t) * (size_t)p->nbed, cudaMemcpyHostToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        free(pm);
        ctx->params.bed = NULL;                                 /* borrowed pointer: not kept */
    }
    CG_CHECK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" cg_ctx *cg_create(const cg_params *p, int device, int *err) {
    int n = cg_device_count();
    if (n <= 0 || device < 0 || device >= n) { if (err) *err = CG_ERR_NO_DEVICE; return NULL; }
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); if (err) *err = CG_ERR_NO_DEVICE; return NULL; }
    install_hooks();
    cg_ctx *ctx = (cg_ctx *)calloc(1, sizeof(cg_ctx));
    if (!ctx) { if (err) *err = CG_ERR_NOMEM; return NULL; }
    ctx->device = device;
    int e = 0;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) e = CG_ERR_CUDA;
    ctx->own_stream = 1;
    ctx->hT = (CgTables *)malloc(sizeof(CgTables));
    if (!e && cudaMalloc((void **)&ctx->dT, sizeof(CgTables)) != cudaSuccess) e = CG_ERR_CUDA;
    if (!e && cudaHostAlloc((void **)&ctx->h_dims, sizeof(CgScalHead), cudaHostAllocMapped) != cudaSuccess) e = CG_ERR_CUDA;
    if (!e && cudaHostGetDevicePointer((void **)&ctx->d_hdims, ctx->h_dims, 0) != cudaSuccess) e = CG_ERR_CUDA;
    if (!e && cudaHostAlloc((void **)&ctx->h_counters, sizeof(unsigned long long) * 32, cudaHostAllocDefault) != cudaSuccess) e = CG_ERR_CUDA;
    if (!e && cudaHostAlloc((void **)&ctx->h_carry_io, 2 * CG_CARRY_BYTES, cudaHostAllocDefault) != cudaSuccess) e = CG_ERR_CUDA;
    for (int i = 0; i < CG_N_TIMERS && !e; i++)
        for (int k = 0; k < 2; k++) if (cudaEventCreate(&ctx->ev[i][k]) != cudaSuccess) e = CG_ERR_CUDA;
    if (!e) e = cg_set_params(ctx, p);
    if (e) { if (err) *err = e; cudaGetLastError(); cg_destroy(ctx); return NULL; }
    if (err) *err = 0;
    return ctx;
}

extern "C" void cg_destroy(cg_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    dbuf *all[] = { &ctx->b_tid, &ctx->b_pos, &ctx->b_flag, &ctx->b_mapq, &ctx->b_lq, &ctx->b_nc, &ctx->b_off, &ctx->b_coff, &ctx->b_cigar,
        &ctx->b_seq, &ctx->b_qual, &ctx->b_qout, &ctx->b_jmap, &ctx->b_rspan, &ctx->b_rd, &ctx->b_ks, &ctx->b_ke, &ctx->b_gap, &ctx->b_gapraw,
        &ctx->b_pmax, &ctx->b_orig, &ctx->b_rbf, &ctx->b_glist, &ctx->b_tlo, &ctx->b_tstart, &ctx->b_isl, &ctx->b_cb, &ctx->b_ev, &ctx->b_depth, &ctx->b_dump,
        &ctx->b_dsum, &ctx->b_csum, &ctx->b_fcol, &ctx->b_trig, &ctx->b_twin, &ctx->b_aggr, &ctx->b_scal, &ctx->b_scratch, &ctx->b_epoch, &ctx->b_events, &ctx->b_chain, &ctx->b_items, &ctx->b_bed, &ctx->b_bedpm, &ctx->b_saved, &ctx->b_crec, &ctx->b_cells, &ctx->b_seq2, &ctx->b_qualp, &ctx->b_exc,
        &ctx->b_truns, &ctx->b_pabs, &ctx->b_pd8, &ctx->b_lq8, &ctx->b_nc8, &ctx->b_cigx, &ctx->b_lqd, &ctx->b_xoff, &ctx->b_absS,
        &ctx->b_qsrc, &ctx->b_ssrc, &ctx->b_dvsum, &ctx->b_htid, &ctx->b_hpos, &ctx->b_hflag, &ctx->b_hmapq, &ctx->b_hlq, &ctx->b_hnc,
        &ctx->b_hcig, &ctx->b_hqual, &ctx->b_hseq, &ctx->b_keep, &ctx->b_kidx, &ctx->b_koff, &ctx->b_kcig };
    for (size_t i = 0; i < sizeof(all) / sizeof(all[0]); i++) if (all[i]->p) cudaFree(all[i]->p);
    if (ctx->dT) cudaFree(ctx->dT);
    if (ctx->h_dims) cudaFreeHost(ctx->h_dims);
    if (ctx->h_counters) cudaFreeHost(ctx->h_counters);
    if (ctx->h_carry_io) cudaFreeHost(ctx->h_carry_io);
    if (ctx->h_stream) cudaFreeHost(ctx->h_stream);
    for (int i = 0; i < CG_N_TIMERS; i++) for (int k = 0; k < 2; k++) if (ctx->ev[i][k]) cudaEventDestroy(ctx->ev[i][k]);
    if (ctx->s_h2d) { cudaStreamDestroy(ctx->s_h2d); cudaStreamDestroy(ctx->s_d2h); for (int i = 0; i < 32; i++) { cudaEventDestroy(ctx->ev_up[i]); cudaEventDestroy(ctx->ev_done[i]); } cudaEventDestroy(ctx->ev_misc); }
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    free(ctx->hT);
    free(ctx);
}

extern "C" const char *cg_last_error(const cg_ctx *ctx) { return ctx ? ctx->err : "no context"; }
extern "C" int cg_set_stream(cg_ctx *ctx, void *s) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)s; ctx->own_stream = 0;
    return 0;
}
extern "C" int cg_set_chunk_bytes(cg_ctx *ctx, int64_t bytes) { ctx->chunk_bytes = bytes; return 0; }
extern "C" int cg_sync(cg_ctx *ctx) { CG_CHECK(cudaStreamSynchronize(ctx->stream)); return 0; }
extern "C" float cg_last_ms(const cg_ctx *ctx, int which) { return (which >= 0 && which < CG_N_TIMERS) ? ctx->ms[which] : -1.f; }
extern "C" int64_t cg_last_launches(const cg_ctx *ctx) { return ctx->launches; }
extern "C" int64_t cg_last_h2d_bytes(const cg_ctx *ctx) { return ctx->h2d_bytes; }
extern "C" int64_t cg_n_columns(const cg_ctx *ctx) { return ctx->D.n_cols; }

#define T0(i) cudaEventRecord(ctx->ev[i][0], st)
#define T1(i) cudaEventRecord(ctx->ev[i][1], st)

/* ---------------------------------------------------------------------------------------- */
static int alloc_inputs(cg_ctx *ctx, const cg_batch *in) {
    const int64_t n = in->n_reads;
    if (n < 0 || in->qual_bytes < 0) return CG_ERR_BAD_ARG;
    if (n > 0x7fffff00LL || in->n_cigar_total > 0x7fffff00LL || in->qual_bytes >= (1LL << 35)) { snprintf(ctx->err, sizeof ctx->err, "batch too large: split it"); return CG_ERR_BAD_ARG; }
    if (n > 0 && in->packed != 1) {
        /* a caller's own layout: every kernel takes record i's bytes at [off[i], off[i] + l_qseq[i]) and k_rewrite / the streamed driver move whole
         * byte RANGES of consecutive records, so the layout must be 8-aligned, ascending and non-overlapping (gaps are fine) */
        for (int64_t i = 0; i < n; i++) {
            const int64_t o = in->off[i], nx = i + 1 < n ? in->off[i + 1] : in->qual_bytes;
            const int64_t c = in->cigar_off[i], cn = i + 1 < n ? in->cigar_off[i + 1] : in->n_cigar_total;
            if (o < 0 || (o & 7) || in->l_qseq[i] < 0 || o + in->l_qseq[i] > nx || nx > in->qual_bytes || c < 0 || c + in->n_cigar[i] > cn || cn > in->n_cigar_total) {
                snprintf(ctx->err, sizeof ctx->err, "record %lld: off[] / cigar_off[] must be 8-aligned (off), ascending and non-overlapping, inside qual_bytes / n_cigar_total", (long long)i);
                return CG_ERR_BAD_ARG;
            }
        }
        if (in->seq_bytes < (in->qual_bytes + 1) / 2) { snprintf(ctx->err, sizeof ctx->err, "seq_bytes must cover qual_bytes / 2"); return CG_ERR_BAD_ARG; }
    }
    size_t n1 = (size_t)n + 1;
    int e;
    if ((e = ensure(ctx, &ctx->b_tid, n1 * 4)) || (e = ensure(ctx, &ctx->b_pos, n1 * 4)) || (e = ensure(ctx, &ctx->b_flag, n1 * 2)) ||
        (e = ensure(ctx, &ctx->b_mapq, n1)) || (e = ensure(ctx, &ctx->b_lq, n1 * 4)) || (e = ensure(ctx, &ctx->b_nc, n1 * 2)) ||
        (e = ensure(ctx, &ctx->b_off, n1 * 8)) || (e = ensure(ctx, &ctx->b_coff, n1 * 4)) ||
        (e = ensure(ctx, &ctx->b_cigar, ((size_t)in->n_cigar_total + 1) * 4)) || (e = ensure(ctx, &ctx->b_seq, (size_t)in->seq_bytes + 128 + CG_FRONT_PAD)) ||
        (e = ensure(ctx, &ctx->b_qual, (size_t)in->qual_bytes + 128 + CG_FRONT_PAD)) || (e = ensure(ctx, &ctx->b_qout, (size_t)in->qual_bytes + 16))) return e;
    CgDev *D = &ctx->D;
    memset(D, 0, sizeof(*D));
    D->n_reads = n; D->n_cigar_total = in->n_cigar_total;
    D->tid = (const int32_t *)ctx->b_tid.p; D->pos = (const int32_t *)ctx->b_pos.p; D->flag = (const uint16_t *)ctx->b_flag.p;
    D->mapq = (const uint8_t *)ctx->b_mapq.p; D->l_qseq = (const int32_t *)ctx->b_lq.p; D->n_cigar = (const uint16_t *)ctx->b_nc.p;
    D->off = (const int64_t *)ctx->b_off.p; D->cigar_off = (const int32_t *)ctx->b_coff.p; D->cigar = (const uint32_t *)ctx->b_cigar.p;
    D->seq = (const uint8_t *)ctx->b_seq.p + CG_FRONT_PAD; D->qual = (const uint8_t *)ctx->b_qual.p + CG_FRONT_PAD; D->qual_out = (uint8_t *)ctx->b_qout.p;
    ctx->has_planes = in->seq2 != NULL; ctx->qual_bits = ctx->has_planes ? in->qual_bits : 0;
    if (ctx->has_planes) {
        if (in->seq2_bytes < in->qual_bytes / 4 || (in->qual_bits != 0 && in->qual_bits != 2 && in->qual_bits != 4) || (in->qual_bytes & 7) ||
            (in->qual_bits && (!in->qualp || in->qualp_bytes < in->qual_bytes * in->qual_bits / 8)) || in->n_seq_exc < 0 || (in->n_seq_exc && !in->seq_exc)) {
            snprintf(ctx->err, sizeof ctx->err, "compact planes do not cover the quality buffer"); return CG_ERR_BAD_ARG;
        }
        if ((e = ensure(ctx, &ctx->b_seq2, (size_t)in->qual_bytes / 4 + 64)) || (e = ensure(ctx, &ctx->b_exc, ((size_t)in->n_seq_exc + 1) * 8)) ||
            (in->qual_bits && (e = ensure(ctx, &ctx->b_qualp, (size_t)in->qual_bytes * in->qual_bits / 8 + 64)))) return e;
        memcpy(ctx->dict.w, in->qual_dict, 16);
    }
    ctx->has_meta = n > 0 && in->packed == 1 && in->meta_planes == 1 && in->tid_runs && in->pos_d8 && in->pos_abs && in->lq8 && in->nc8 &&
                    in->n_tid_runs > 0 && in->n_pos_abs > 0 && in->n_cigar_x >= 0 && (in->n_cigar_x == 0 || in->cigar_x) && in->n_cigar_x <= in->n_cigar_total;
    if (ctx->has_meta) {
        if ((e = ensure(ctx, &ctx->b_truns, (size_t)in->n_tid_runs * 8)) || (e = ensure(ctx, &ctx->b_pabs, (size_t)in->n_pos_abs * 8)) ||
            (e = ensure(ctx, &ctx->b_absS, (size_t)in->n_pos_abs * 4)) || (e = ensure(ctx, &ctx->b_pd8, n1)) || (e = ensure(ctx, &ctx->b_lq8, n1)) ||
            (e = ensure(ctx, &ctx->b_nc8, n1)) || (e = ensure(ctx, &ctx->b_cigx, ((size_t)in->n_cigar_x + 1) * 4)) || (e = ensure(ctx, &ctx->b_lqd, 1024)) ||
            (e = ensure(ctx, &ctx->b_xoff, n1 * 4))) return e;
        ctx->n_truns = in->n_tid_runs; ctx->n_pabs = in->n_pos_abs; ctx->n_cigx = in->n_cigar_x;
    }
    ctx->qual_bytes = in->qual_bytes; ctx->cigar_total = in->n_cigar_total;
    ctx->packed = in->packed == 1; ctx->offsets_ready = 0;
    ctx->h2d_bytes = 0;
    return 0;
}

/* the small per-record arrays and the CIGARs: everything the read/tile preparation needs */
static int upload_meta(cg_ctx *ctx, const cg_batch *in, cudaStream_t st) {
    const int64_t n = in->n_reads;
    if (!n) return 0;
    if (ctx->has_meta) {                                       /* about 6 bytes per record instead of 21; run_prep expands them */
        CG_CHECK(cudaMemcpyAsync(ctx->b_truns.p, in->tid_runs, (size_t)in->n_tid_runs * 8, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_pabs.p, in->pos_abs, (size_t)in->n_pos_abs * 8, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_lqd.p, in->lq_dict, 1024, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_pd8.p, in->pos_d8, (size_t)n, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_lq8.p, in->lq8, (size_t)n, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_nc8.p, in->nc8, (size_t)n, cudaMemcpyHostToDevice, st));
        if (in->n_cigar_x) CG_CHECK(cudaMemcpyAsync(ctx->b_cigx.p, in->cigar_x, (size_t)in->n_cigar_x * 4, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_flag.p, in->flag, (size_t)n * 2, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_mapq.p, in->mapq, (size_t)n, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += n * (1 + 1 + 1 + 2 + 1) + (in->n_tid_runs + in->n_pos_abs) * 8 + 1024 + in->n_cigar_x * 4;
        if (ctx->has_planes && in->n_seq_exc) {
            CG_CHECK(cudaMemcpyAsync(ctx->b_exc.p, in->seq_exc, (size_t)in->n_seq_exc * 8, cudaMemcpyHostToDevice, st));
            ctx->h2d_bytes += in->n_seq_exc * 8;
        }
        return 0;
    }
    CG_CHECK(cudaMemcpyAsync(ctx->b_tid.p, in->tid, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CG_CHECK(cudaMemcpyAsync(ctx->b_pos.p, in->pos, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CG_CHECK(cudaMemcpyAsync(ctx->b_flag.p, in->flag, (size_t)n * 2, cudaMemcpyHostToDevice, st));
    CG_CHECK(cudaMemcpyAsync(ctx->b_mapq.p, in->mapq, (size_t)n, cudaMemcpyHostToDevice, st));
    CG_CHECK(cudaMemcpyAsync(ctx->b_lq.p, in->l_qseq, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CG_CHECK(cudaMemcpyAsync(ctx->b_nc.p, in->n_cigar, (size_t)n * 2, cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += n * (4 + 4 + 2 + 1 + 4 + 2) + in->n_cigar_total * 4;
    if (!ctx->packed) {                                        /* a packed batch gets its two offset arrays from scans (run_prep) */
        CG_CHECK(cudaMemcpyAsync(ctx->b_off.p, in->off, (size_t)n * 8, cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ctx->b_coff.p, in->cigar_off, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += n * 12;
    }
    if (in->n_cigar_total) CG_CHECK(cudaMemcpyAsync(ctx->b_cigar.p, in->cigar, (size_t)in->n_cigar_total * 4, cudaMemcpyHostToDevice, st));
    if (ctx->has_planes && in->n_seq_exc) {
        CG_CHECK(cudaMemcpyAsync(ctx->b_exc.p, in->seq_exc, (size_t)in->n_seq_exc * 8, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += in->n_seq_exc * 8;
    }
    return 0;
}

/* bytes [b0, b1) of the quality buffer and the matching half of the packed sequences */
static int upload_bases(cg_ctx *ctx, const cg_batch *in, int64_t b0, int64_t b1, cudaStream_t st) {
    if (b1 <= b0) return 0;
    if (ctx->has_planes) {                                     /* chunk bounds are record offsets: multiples of 8 positions */
        CG_CHECK(cudaMemcpyAsync((char *)ctx->b_seq2.p + b0 / 4, in->seq2 + b0 / 4, (size_t)(b1 - b0) / 4, cudaMemcpyHostToDevice, st));
        ctx->h2d_bytes += (b1 - b0) / 4;
        if (ctx->qual_bits) {
            const int64_t q0 = b0 * ctx->qual_bits / 8, q1 = b1 * ctx->qual_bits / 8;
            CG_CHECK(cudaMemcpyAsync((char *)ctx->b_qualp.p + q0, in->qualp + q0, (size_t)(q1 - q0), cudaMemcpyHostToDevice, st));
            ctx->h2d_bytes += q1 - q0;
        } else {
            CG_CHECK(cudaMemcpyAsync((char *)ctx->b_qual.p + CG_FRONT_PAD + b0, in->qual + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, st));
            ctx->h2d_bytes += b1 - b0;
        }
        return 0;
    }
    CG_CHECK(cudaMemcpyAsync((char *)ctx->b_qual.p + CG_FRONT_PAD + b0, in->qual + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, st));
    int64_t s0 = b0 >> 1, s1 = (b1 + 1) >> 1;
    if (s1 > in->seq_bytes) s1 = in->seq_bytes;
    if (s1 > s0) CG_CHECK(cudaMemcpyAsync((char *)ctx->b_seq.p + CG_FRONT_PAD + s0, in->seq + s0, (size_t)(s1 - s0), cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += (b1 - b0) + (s1 > s0 ? s1 - s0 : 0);
    return 0;
}

/* positions [b0, b1) have landed as compact planes: expand them into the working arrays (on the compute stream) */
static int expand_bases(cg_ctx *ctx, const cg_batch *in, int64_t b0, int64_t b1, cudaStream_t st) {
    if (!ctx->has_planes || b1 <= b0) return 0;
    const int64_t g0 = b0 >> 3, g1 = b1 >> 3;
    k_unpack<<<(unsigned)((g1 - g0 + 255) / 256), 256, 0, st>>>((const uint8_t *)ctx->b_seq2.p, (const uint8_t *)ctx->b_qualp.p, (uint8_t *)ctx->b_seq.p + CG_FRONT_PAD,
                                                                 (uint8_t *)ctx->b_qual.p + CG_FRONT_PAD, g0, g1, ctx->qual_bits, ctx->dict);
    ctx->launches++;
    if (in->n_seq_exc) {                                       /* the exceptions inside [b0, b1): the list is ascending */
        int64_t lo = 0, hi = in->n_seq_exc, e0, e1;
        while (lo < hi) { const int64_t m = (lo + hi) >> 1; if ((int64_t)(in->seq_exc[m] >> 4) < b0) lo = m + 1; else hi = m; }
        e0 = lo; hi = in->n_seq_exc;
        while (lo < hi) { const int64_t m = (lo + hi) >> 1; if ((int64_t)(in->seq_exc[m] >> 4) < b1) lo = m + 1; else hi = m; }
        e1 = lo;
        if (e1 > e0) { k_unpack_exc<<<(unsigned)((e1 - e0 + 255) / 256), 256, 0, st>>>((const uint64_t *)ctx->b_exc.p, e0, e1, (uint8_t *)ctx->b_seq.p + CG_FRONT_PAD); ctx->launches++; }
    }
    CG_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int cg_upload(cg_ctx *ctx, const cg_batch *in) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    CG_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ctx->resident = 0; ctx->win_on = 0;
    int e;
    if ((e = alloc_inputs(ctx, in))) return e;
    T0(CG_T_H2D);
    if ((e = upload_meta(ctx, in, st)) || (e = upload_bases(ctx, in, 0, in->qual_bytes, st)) || (e = expand_bases(ctx, in, 0, in->qual_bytes, st))) return e;
    T1(CG_T_H2D);
    ctx->resident = 1;
    return 0;
}

template <class T, class Op, class Load, class Store>
static int run_scan(cg_ctx *ctx, Load ld, Store st_, int64_t n, T ident, T *total_dev) {
    cudaStream_t st = ctx->stream;
    int nb = (int)((n + SCAN_CHUNK - 1) / SCAN_CHUNK);
    if (nb < 1) nb = 1;
    int e = ensure(ctx, &ctx->b_aggr, (size_t)nb * sizeof(T) + 64);
    if (e) return e;
    T *aggr = (T *)ctx->b_aggr.p;
    k_scan_reduce<T, Op, Load><<<nb, SCAN_THREADS, 0, st>>>(ld, n, ident, aggr);
    k_scan_aggr<T, Op><<<1, SCAN_THREADS, 0, st>>>(aggr, nb, ident, total_dev);
    k_scan_apply<T, Op, Load, Store><<<nb, SCAN_THREADS, 0, st>>>(ld, st_, n, ident, aggr);
    ctx->launches += 3;
    CG_CHECK(cudaGetLastError());
    return 0;
}

static inline int nblk(int64_t n, int t) { int64_t b = (n + t - 1) / t; return (int)(b < 1 ? 1 : b); }

/* ---- slices ------------------------------------------------------------------------------
 * The chain runs over SLICES of the batch in position order: columns of tiles [t0,t1), then the sparse passes of
 * those columns with the cross-column state (keep-window chain, depth average) carried from slice to slice on the
 * device, then the rewrite of every record whose last column lies below the slice end.  A resident batch is one
 * slice; cg_process cuts the batch so that slice i starts as soon as upload chunk i has landed and its qualities
 * travel back while later chunks are still arriving (H2D, kernels and D2H overlap, PCIe is full duplex). */
/* upload chunk i ends before record rb[i]; out[3i] = tiles complete once it has landed, out[3i+1] = records final then,
 * out[3i+2] = pileup reads whose bases are on the device then (their cell rows can be built) */
__global__ void k_bounds(const __grid_constant__ CgDev D, const __grid_constant__ CgBounds B, int64_t *out) {
    const int i = threadIdx.x;
    if (i >= B.n) return;
    const int64_t r = B.rb[i];
    const int j = r < D.n_reads ? D.jmap[r] : D.n_pile;            /* first pileup read at/after record r */
    int64_t T = D.n_tiles, rec = D.n_reads;
    if (j < D.n_pile) {
        T = D.rd[j].col0 >> 5;                                      /* columns < 32T only see reads before j */
        const int R = D.tile_lo[T];                                 /* reads before R end at or below column 32T */
        rec = R < D.n_pile ? (int64_t)D.orig[R] : D.n_reads;
        if (rec > r) rec = r;
    }
    out[3 * i] = T; out[3 * i + 1] = rec; out[3 * i + 2] = j;
}
__global__ void k_window_max(const __grid_constant__ CgDev D, int32_t *out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int v = t < D.n_tiles ? D.tile_start[t + 1] - D.tile_lo[t] : 0;
    v = __reduce_max_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v > 0) atomicMax(out, v);
}
struct LdEvFlagOff { const uint16_t *ev; uint16_t mask; __device__ int32_t operator()(int64_t c) const { return (ev[c] & mask) != 0; } };
struct StCompactOff { int32_t *out; const uint16_t *ev; uint16_t mask; int32_t c0; __device__ void operator()(int64_t c, int32_t, int32_t ex) const { if (ev[c] & mask) out[ex] = (int32_t)c + c0; } };
struct StI64Carry { int64_t *p; const CgEpochCarry *cy; __device__ void operator()(int64_t i, int64_t inc, int64_t) const { p[i] = inc + cy->dsum_last; } };
struct StI32Carry { int32_t *p; const CgEpochCarry *cy; __device__ void operator()(int64_t i, int32_t inc, int32_t) const { p[i] = inc + cy->csum_last; } };

static int run_prep(cg_ctx *ctx, const CgBounds *bounds, int64_t *h_bounds) {
    cudaStream_t st = ctx->stream;
    CgDev *D = &ctx->D;
    const int64_t n = D->n_reads;
    const size_t n1 = (size_t)n + 1;
    int e, check_packed = 0;
    ctx->launches = 0;
    for (int i = 0; i < CG_N_TIMERS; i++) if (i != CG_T_H2D && i != CG_T_D2H) ctx->ms[i] = 0;
    D->T = ctx->dT; cg_devparams_from(&D->P, &ctx->params);
    if (ctx->win_on) {
        const cg_window *w = &ctx->win;
        D->P.win_on = 1; D->P.win_lo_tid = w->first == 1 ? -1 : w->lo_tid; D->P.win_lo_pos = w->lo_pos; D->P.win_cnt_pos = w->cnt_pos;
        D->P.win_hi_tid = w->hi_tid; D->P.win_hi_pos = w->hi_pos;
    }
    D->bed = (const cg_bed_reg *)ctx->b_bed.p; D->bed_pm = (const int64_t *)ctx->b_bedpm.p;
    if ((e = ensure(ctx, &ctx->b_scal, sizeof(CgScalars)))) return e;
    CgScalars *scal = (CgScalars *)ctx->b_scal.p;
    D->counters = scal->counters;
    D->maxdepth = &scal->h.maxdepth; D->err = &scal->h.err; D->beyond = &scal->h.beyond;
    if ((e = ensure(ctx, &ctx->b_jmap, n1 * 4)) || (e = ensure(ctx, &ctx->b_rspan, n1 * 4)) || (e = ensure(ctx, &ctx->b_rd, n1 * sizeof(CgRead))) ||
        (e = ensure(ctx, &ctx->b_ks, n1 * 8)) || (e = ensure(ctx, &ctx->b_ke, n1 * 8)) || (e = ensure(ctx, &ctx->b_gap, n1 * 8)) ||
        (e = ensure(ctx, &ctx->b_gapraw, n1 * 8)) || (e = ensure(ctx, &ctx->b_pmax, n1 * 4)) || (e = ensure(ctx, &ctx->b_orig, n1 * 4)) ||
        (e = ensure(ctx, &ctx->b_rbf, n1)) || (e = ensure(ctx, &ctx->b_isl, n1 * sizeof(CgIsland))) || (e = ensure(ctx, &ctx->b_glist, n1 * 4))) return e;
    D->jmap = (int32_t *)ctx->b_jmap.p; D->rspan = (int32_t *)ctx->b_rspan.p; D->rd = (CgRead *)ctx->b_rd.p;
    D->ks = (int64_t *)ctx->b_ks.p; D->ke = (int64_t *)ctx->b_ke.p; D->gap = (int64_t *)ctx->b_gap.p;
    D->pmaxcol = (int32_t *)ctx->b_pmax.p; D->orig = (int32_t *)ctx->b_orig.p; D->r_bf = (uint8_t *)ctx->b_rbf.p;
    D->isl = (CgIsland *)ctx->b_isl.p;
    D->glist = ctx->generic ? NULL : (int32_t *)ctx->b_glist.p; D->n_glist = &scal->n_glist;
    int64_t *gapraw = (int64_t *)ctx->b_gapraw.p;

    T0(CG_T_TILES);
    CG_CHECK(cudaMemsetAsync(scal, 0, sizeof(CgScalars), st));
    {
        CgChainCarry cc; memset(&cc, 0, sizeof cc); cc.bkey = INT64_MIN; cc.ukey = INT64_MIN; cg_win_reset(&cc.w);
        memcpy(ctx->h_carry_init, &cc, sizeof cc);
        CG_CHECK(cudaMemcpyAsync(&scal->chain, ctx->h_carry_init, sizeof cc, cudaMemcpyHostToDevice, st));
        if (ctx->win_on && !ctx->win.first && ctx->have_saved) {       /* continue where the previous call of the chain stopped */
            const CgSavedCarry *sv = (const CgSavedCarry *)ctx->b_saved.p;
            CG_CHECK(cudaMemcpyAsync(&scal->chain, &sv->cc, sizeof(CgChainCarry), cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync(&scal->epoch, &sv->ec, sizeof(CgEpochCarry), cudaMemcpyDeviceToDevice, st));
        }
    }
    if (n > 0 && ctx->packed && !ctx->offsets_ready) {         /* once per uploaded batch: off = running sum of the padded lengths, cigar_off = running sum of n_cigar */
        if (ctx->has_meta) {                                   /* the per-record arrays from their compact planes first */
            LdD8 ld8 = { (const uint8_t *)ctx->b_pd8.p }; StInclU32 ss = { (uint32_t *)ctx->b_pos.p };
            if ((e = run_scan<uint32_t, OpSum>(ctx, ld8, ss, n, 0u, (uint32_t *)NULL))) return e;
            k_meta_gather<<<nblk(ctx->n_pabs, 256), 256, 0, st>>>((const uint64_t *)ctx->b_pabs.p, ctx->n_pabs, (const uint32_t *)ctx->b_pos.p, (uint32_t *)ctx->b_absS.p);
            k_meta_expand<<<nblk(n, 256), 256, 0, st>>>(n, (const uint64_t *)ctx->b_truns.p, ctx->n_truns, (const uint64_t *)ctx->b_pabs.p, ctx->n_pabs,
                (const uint32_t *)ctx->b_absS.p, (const uint8_t *)ctx->b_lq8.p, (const int32_t *)ctx->b_lqd.p, (const uint8_t *)ctx->b_nc8.p,
                (int32_t *)ctx->b_tid.p, (int32_t *)ctx->b_pos.p, (int32_t *)ctx->b_lq.p, (uint16_t *)ctx->b_nc.p);
            ctx->launches += 2;
        }
        LdPad8 lp = { D->l_qseq }; StExcl64 so = { (int64_t *)ctx->b_off.p };
        if ((e = run_scan<int64_t, OpSum>(ctx, lp, so, n, (int64_t)0, &scal->h.qual_total))) return e;
        LdNCig ln = { D->n_cigar }; StExcl32 sc = { (int32_t *)ctx->b_coff.p };
        if ((e = run_scan<int32_t, OpSum>(ctx, ln, sc, n, 0, &scal->h.cigar_total))) return e;
        if (ctx->has_meta) {
            LdNcx lx = { (const uint8_t *)ctx->b_nc8.p }; StExcl32 sx = { (int32_t *)ctx->b_xoff.p };
            if ((e = run_scan<int32_t, OpSum>(ctx, lx, sx, n, 0, (int32_t *)NULL))) return e;
            k_meta_cigar<<<nblk(n, 256), 256, 0, st>>>(n, (const uint8_t *)ctx->b_nc8.p, D->l_qseq, (const int32_t *)ctx->b_coff.p, (const int32_t *)ctx->b_xoff.p,
                (const uint32_t *)ctx->b_cigx.p, (uint32_t *)ctx->b_cigar.p, ctx->cigar_total, ctx->n_cigx);
            ctx->launches++;
        }
        ctx->offsets_ready = 1; check_packed = 1;
    }
    if (n > 0) {
        k_prep_read<<<nblk(n, 256), 256, 0, st>>>(*D); ctx->launches++;
        LdPileFlag lpf = { D->rspan }; StJmap sj = { D->jmap };
        if ((e = run_scan<int32_t, OpSum>(ctx, lpf, sj, n, 0, &scal->h.n_pile))) return e;
        k_prep_keys<<<nblk(n, 256), 256, 0, st>>>(*D); ctx->launches++;
        /* ke := inclusive prefix max (only the first n_pile entries are meaningful; the tail is never read) */
        CG_CHECK(cudaMemcpyAsync(ctx->h_dims, &scal->h, sizeof(CgScalHead), cudaMemcpyDeviceToHost, st));
        CG_CHECK(cudaStreamSynchronize(st));
        if (check_packed) {                                        /* packed = 1 is a promise about the layout: the running sums must end where the buffers do */
            const int64_t qtot = ctx->h_dims->qual_total;
            if (qtot > ctx->qual_bytes || (int64_t)ctx->h_dims->cigar_total > ctx->cigar_total) {
                snprintf(ctx->err, sizeof ctx->err, "packed batch: the padded lengths sum to %lld quality bytes (buffer holds %lld), the CIGARs to %d operations (buffer holds %lld)",
                         (long long)qtot, (long long)ctx->qual_bytes, ctx->h_dims->cigar_total, (long long)ctx->cigar_total);
                return CG_ERR_BAD_ARG;
            }
        }
        D->n_pile = ctx->h_dims->n_pile;
    } else D->n_pile = 0;
    const int np = D->n_pile;
    if (np > 0) {
        LdI64 lke = { D->ke }; StI64Incl ske = { D->ke };
        if ((e = run_scan<int64_t, OpMax>(ctx, lke, ske, np, (int64_t)INT64_MIN, (int64_t *)NULL))) return e;
        k_gap<<<nblk(np, 256), 256, 0, st>>>(*D, &scal->h.n_pile, gapraw); ctx->launches++;
        LdI64 lg = { gapraw }; StI64Incl sg = { D->gap };
        if ((e = run_scan<int64_t, OpSum>(ctx, lg, sg, np, (int64_t)0, (int64_t *)NULL))) return e;
        LdIslandFlag lif = { gapraw }; StIsland sis = { D->isl, D->ks, D->gap, gapraw };
        if ((e = run_scan<int32_t, OpSum>(ctx, lif, sis, np, 0, &scal->h.n_islands))) return e;
        k_finish_read<<<nblk(np, 256), 256, 0, st>>>(*D, &scal->h.n_pile, &scal->h.n_cols); ctx->launches++;
        if (!ctx->generic) {                                       /* cell matrix: first group of every row, total in cell_groups */
            if ((e = ensure(ctx, &ctx->b_crec, ((size_t)np + 1) * sizeof(CgCellRec)))) return e;
            D->crec = (CgCellRec *)ctx->b_crec.p;
            LdNgrp lg2 = { D->rd }; StCellRec sc2 = { D->crec, D->rd };
            if ((e = run_scan<int64_t, OpSum>(ctx, lg2, sc2, np, (int64_t)0, &scal->h.cell_groups))) return e;
        }
    }
    CG_CHECK(cudaMemcpyAsync(ctx->h_dims, &scal->h, sizeof(CgScalHead), cudaMemcpyDeviceToHost, st));
    CG_CHECK(cudaStreamSynchronize(st));
    if (ctx->h_dims->err) { snprintf(ctx->err, sizeof ctx->err, "device reported error %d while building read records", ctx->h_dims->err); return ctx->h_dims->err; }
    D->n_cols = np > 0 ? ctx->h_dims->n_cols : 0; D->n_islands = np > 0 ? ctx->h_dims->n_islands : 0;
    D->n_tiles = (D->n_cols + 31) / 32;
    D->n_flagged = 0;
    if (np > 0 && !ctx->generic) {
        const int64_t ng = ctx->h_dims->cell_groups;
        if (ng >= (1LL << 32)) { snprintf(ctx->err, sizeof ctx->err, "batch too large: split it"); return CG_ERR_BAD_ARG; }
        if ((e = ensure(ctx, &ctx->b_cells, (size_t)ng * 16 + 64))) return e;
        D->cells = (uint16_t *)ctx->b_cells.p;
    }
    const int nc = D->n_cols;
    const size_t nc1 = (size_t)nc + 64;
    D->want_dump = 0;
    if ((e = ensure(ctx, &ctx->b_tlo, ((size_t)D->n_tiles + 2) * 4)) || (e = ensure(ctx, &ctx->b_tstart, ((size_t)D->n_tiles + 2) * 4)) ||
        (e = ensure(ctx, &ctx->b_cb, nc1)) || (e = ensure(ctx, &ctx->b_ev, nc1 * 2)) || (e = ensure(ctx, &ctx->b_depth, nc1 * 4)) ||
        (e = ensure(ctx, &ctx->b_fcol, nc1 * 4))) return e;
    D->tile_lo = (int32_t *)ctx->b_tlo.p; D->tile_start = (int32_t *)ctx->b_tstart.p;
    D->cb = (uint8_t *)ctx->b_cb.p; D->ev = (uint16_t *)ctx->b_ev.p; D->depth = (uint32_t *)ctx->b_depth.p; D->fcol = (int32_t *)ctx->b_fcol.p;
    if (ctx->dump_columns || getenv("CG_COLUMN_DUMP")) {
        if ((e = ensure(ctx, &ctx->b_dump, nc1 * sizeof(cg_column)))) return e;
        D->coldump = (cg_column *)ctx->b_dump.p; D->want_dump = 1;
    }
    ctx->need_depth = 0;
    for (int i = 0; i < 3 * CG_MAX_CHUNKS; i++) h_bounds[i] = 0;
    if (np > 0 && nc > 0) {
        CG_CHECK(cudaMemsetAsync(D->cb, 0, nc1, st));              /* k_paint may mark columns of a later slice before k_column fills them */
        k_fill_i32<<<nblk(D->n_tiles + 2, 256), 256, 0, st>>>(D->tile_lo, D->n_tiles + 2, np);
        k_fill_i32<<<nblk(D->n_tiles + 2, 256), 256, 0, st>>>(D->tile_start, D->n_tiles + 2, np);
        k_tile_index<<<nblk(np, 256), 256, 0, st>>>(*D);
        k_window_max<<<nblk(D->n_tiles, 256), 256, 0, st>>>(*D, &scal->h.window_max);
        k_bounds<<<1, CG_MAX_CHUNKS, 0, st>>>(*D, *bounds, scal->bounds); ctx->launches += 5;
        CG_CHECK(cudaMemcpyAsync(ctx->h_dims, &scal->h, sizeof(CgScalHead), cudaMemcpyDeviceToHost, st));
        CG_CHECK(cudaMemcpyAsync(h_bounds, scal->bounds, sizeof scal->bounds, cudaMemcpyDeviceToHost, st));
        CG_CHECK(cudaStreamSynchronize(st));
        /* over-depth (snp_score.c:1673) needs n_plp > -P * mean depth >= -P: impossible when no tile has more than -P candidates */
        ctx->need_depth = ctx->params.over_depth < 1.0 || (double)ctx->h_dims->window_max > ctx->params.over_depth;
        ctx->depth_matters = ctx->need_depth;
        if (ctx->win_on) ctx->need_depth = 1;                       /* a later call of the chain may need the running average */
        if (ctx->need_depth) {
            if ((e = ensure(ctx, &ctx->b_dsum, nc1 * 8)) || (e = ensure(ctx, &ctx->b_csum, nc1 * 4))) return e;
            D->dsum = (int64_t *)ctx->b_dsum.p; D->csum = (int32_t *)ctx->b_csum.p;
            ctx->epoch_cap = D->n_islands + nc / 262144 + 16 + 2 * CG_MAX_CHUNKS;
            if ((e = ensure(ctx, &ctx->b_epoch, (size_t)ctx->epoch_cap * sizeof(CgEpoch)))) return e;
        }
    }
    T1(CG_T_TILES);
    ctx->nf_total = 0;
    return 0;
}

/* One slice: tiles [t0,t1) -> their columns -> sparse passes over columns [c0,c1) -> records [r0,r1).  The work falls in three parts:
 *   A   (no carried state)  cell rows, column stage, flagged columns + their STR searches;
 *   B1  (the carry)         depth prefix sums + epochs, keep-window chain: small, and all the NEXT slice / call / region shard needs;
 *   B2  (the rest)          over-depth test, window painting, per-read rewrite.
 * A single context runs A, B1, B2 slice after slice.  Region shards on several devices (cg_shard_*) run A for all their slices at
 * once, pass the carry from shard to shard through B1 alone, and run B2 concurrently again. */

static int slice_A(cg_ctx *ctx, CgSlice *s, int timed) {
    cudaStream_t st = ctx->stream;
    CgDev *D = &ctx->D;
    CgScalars *scal = (CgScalars *)ctx->b_scal.p;
    int e;
    const int ncs = s->c1 > s->c0 ? s->c1 - s->c0 : 0;          /* columns of the sparse passes: the tiles' own, except in chained calls */
    int nfs = 0;
    const int kb = ctx->nf_total;
    if (timed) T0(CG_T_CELLS);
    if (s->je > s->jb && !ctx->generic) {                       /* cell rows of the pileup reads whose bases have landed */
        k_cells<<<nblk((int64_t)(s->je - s->jb) * 4, 256), 256, 0, st>>>(*D, s->jb, s->je);
        k_cells_general<<<148 * 4, 256, 0, st>>>(*D, s->jb, s->je);
        ctx->launches += 2;
    }
    if (timed) { T1(CG_T_CELLS); T0(CG_T_COLUMNS); }
    D->item_bound = &scal->h.slice.item_bound;
    if (s->t1 > s->t0) {
        CG_CHECK(cudaMemsetAsync(&scal->h.slice, 0, sizeof scal->h.slice, st));
        if (ctx->generic) k_column_generic<<<nblk((int64_t)(s->t1 - s->t0) * 32, 128), 128, 0, st>>>(*D, s->t0, s->t1);
        else {
            /* persistent warps claim tiles from a counter: one warp slot per resident warp, never more warps than tiles */
            int blocks = nblk(s->t1 - s->t0, COL_WARPS);
            if (blocks > 148 * COL_MINB) blocks = 148 * COL_MINB;
            k_column<<<blocks, COL_WARPS * 32, 0, st>>>(*D, s->t0, s->t1, &scal->h.slice.tile_counter);
        }
        ctx->launches++;
    }
    if (timed) { T1(CG_T_COLUMNS); T0(CG_T_FLAGGED); }
    if (ncs > 0) {
        LdEvFlagOff lf = { D->ev + s->c0, CG_EV_FLAGGED }; StCompactOff sc = { D->fcol + kb, D->ev + s->c0, CG_EV_FLAGGED, s->c0 };
        if ((e = run_scan<int32_t, OpSum>(ctx, lf, sc, ncs, 0, &scal->h.n_flagged))) return e;
        k_publish<<<1, 32, 0, st>>>((const int32_t *)&scal->h, (int32_t *)ctx->d_hdims, (int)(sizeof(CgScalHead) / 4)); ctx->launches++;
        CG_CHECK(cudaStreamSynchronize(st));
        nfs = ctx->h_dims->n_flagged;
    }
    const int ke = kb + nfs;
    if ((e = ensure_keep(ctx, &ctx->b_trig, ((size_t)ke + 1) * sizeof(CgTrig))) || (e = ensure_keep(ctx, &ctx->b_twin, ((size_t)ke + 1) * sizeof(CgWin)))) return e;
    D->trig = (CgTrig *)ctx->b_trig.p; D->twin = (CgWin *)ctx->b_twin.p;
    D->n_flagged = ke;
    if (nfs > 0) {
        int threads = FL_WARPS * 32, blocks = nblk(nfs, FL_WARPS);
        if (blocks > 148 * 8) blocks = 148 * 8;
        /* the item list holds at most what the slice's columns announced (their bound came over with n_flagged) */
        const int64_t ub = (int64_t)ctx->h_dims->slice.item_bound;
        if (ub > 0x7fffff00LL) { snprintf(ctx->err, sizeof ctx->err, "too many STR searches in one slice"); return CG_ERR_OVERFLOW; }
        if ((e = ensure(ctx, &ctx->b_items, ((size_t)ub + 1) * sizeof(CgStrItem)))) return e;
        D->sitem = (CgStrItem *)ctx->b_items.p; D->sitem_cap = ub; D->n_sitem = &scal->h.n_sitem;
        CG_CHECK(cudaMemsetAsync(&scal->h.n_sitem, 0, sizeof scal->h.n_sitem, st));
        k_flagged<<<blocks, threads, 0, st>>>(*D, kb, ke); ctx->launches++;
        if (ub > 0) {
            int sblocks = nblk(ub, STR_THREADS);
            if (sblocks > 148 * 8) sblocks = 148 * 8;
            k_str_items<<<sblocks, STR_THREADS, 0, st>>>(*D); ctx->launches++;
        }
    }
    if (timed) T1(CG_T_FLAGGED);
    s->kb = kb; s->ke = ke;
    ctx->nf_total = ke;
    CG_CHECK(cudaGetLastError());
    return 0;
}

/* what: 1 = B1, 2 = B2, 3 = both */
static int slice_B(cg_ctx *ctx, const CgSlice *s, int what, int timed) {
    cudaStream_t st = ctx->stream;
    CgDev *D = &ctx->D;
    CgChainCarry *ccarry = &((CgScalars *)ctx->b_scal.p)->chain;
    CgEpochCarry *ecarry = &((CgScalars *)ctx->b_scal.p)->epoch;
    int e;
    const int c0 = s->c0, c1 = s->c1, kb = s->kb, ke = s->ke, nfs = ke - kb;
    const int ncs = c1 > c0 ? c1 - c0 : 0;
    D->trig = (CgTrig *)ctx->b_trig.p; D->twin = (CgWin *)ctx->b_twin.p;
    if (D->n_flagged < ke) D->n_flagged = ke;
    if (timed) T0(CG_T_DEPTH);
    if (ctx->need_depth && ncs > 0) {
        if (what & 1) {
            LdDepthCounted ld = { D->depth + c0, D->ev + c0 }; StI64Carry sd = { D->dsum + c0, ecarry };
            if ((e = run_scan<int64_t, OpSum>(ctx, ld, sd, ncs, (int64_t)0, (int64_t *)NULL))) return e;
            LdCounted lc = { D->ev + c0 }; StI32Carry sc2 = { D->csum + c0, ecarry };
            if ((e = run_scan<int32_t, OpSum>(ctx, lc, sc2, ncs, 0, (int32_t *)NULL))) return e;
            k_epochs<<<1, 32, 0, st>>>(*D, (CgEpoch *)ctx->b_epoch.p, ecarry, ctx->epoch_cap, c0, c1); ctx->launches++;
        }
        if (what & 2) { k_deep<<<nblk(ncs, 256), 256, 0, st>>>(*D, (const CgEpoch *)ctx->b_epoch.p, ecarry, c0, c1); ctx->launches++; }
    }
    if (timed) { T1(CG_T_DEPTH); T0(CG_T_CHAIN); }
    if (nfs > 0) {
        if (what & 1) {
            /* b_chain holds bmax (first half) and umax (second half) per flagged entry, indexed by slice-local position */
            if ((e = ensure(ctx, &ctx->b_chain, ((size_t)nfs + 1) * 16))) return e;
            int64_t *bmax = (int64_t *)ctx->b_chain.p, *umax = bmax + nfs;
            double mul = ctx->params.iSTR_mul > ctx->params.sSTR_mul ? ctx->params.iSTR_mul : ctx->params.sSTR_mul;
            double add = ctx->params.iSTR_add > ctx->params.sSTR_add ? ctx->params.iSTR_add : ctx->params.sSTR_add;
            if (mul < 0) mul = 0;
            LdTrigB lb = { D->trig + kb, ccarry }; StI64Incl sb = { bmax };
            if ((e = run_scan<int64_t, OpMax>(ctx, lb, sb, nfs, (int64_t)INT64_MIN, (int64_t *)NULL))) return e;
            LdTrigU lu = { D->trig + kb, bmax, ccarry, mul, add }; StI64Incl su = { umax };
            if ((e = run_scan<int64_t, OpMax>(ctx, lu, su, nfs, (int64_t)INT64_MIN, (int64_t *)NULL))) return e;
            k_chain<<<nblk(nfs, 128), 128, 0, st>>>(*D, umax - kb, ccarry, kb, ke);
            k_chain_carry<<<1, 32, 0, st>>>(*D, bmax - kb, umax - kb, ccarry, kb, ke); ctx->launches += 2;
        }
        if (what & 2) { k_paint<<<nblk(nfs, 128), 128, 0, st>>>(*D, kb, ke); ctx->launches++; }
    }
    if (timed) { T1(CG_T_CHAIN); T0(CG_T_REWRITE); }
    if ((what & 2) && s->r1 > s->r0) {
        if (ctx->generic) k_rewrite_generic<<<nblk(s->r1 - s->r0, 128), 128, 0, st>>>(*D, s->r0, s->r1);
        else k_rewrite<<<nblk(s->r1 - s->r0, RW_READS), RW_THREADS, 0, st>>>(*D, s->r0, s->r1);
        ctx->launches++;
    }
    if (timed) T1(CG_T_REWRITE);
    CG_CHECK(cudaGetLastError());
    return 0;
}

static void read_timer(cg_ctx *ctx, int i) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev[i][0], ctx->ev[i][1]) == cudaSuccess) ctx->ms[i] = ms; else cudaGetLastError();
}
/* the spans of the last call's uploads and downloads */
static void read_copy_timers(cg_ctx *ctx) { read_timer(ctx, CG_T_H2D); read_timer(ctx, CG_T_D2H); }

/* ordered BED event list, counters, dump flags; leaves everything small on the host side of the context */
static int run_finish(cg_ctx *ctx, int timed) {
    cudaStream_t st = ctx->stream;
    CgDev *D = &ctx->D;
    CgScalars *scal = (CgScalars *)ctx->b_scal.p;
    const int nc = D->n_cols;
    int e;
    if (timed) T0(CG_T_EVENTS);
    if (nc > 0) {
        /* BED events: ordered compaction; capacity grows on demand */
        if (!ctx->b_events.p) { if ((e = ensure(ctx, &ctx->b_events, sizeof(cg_bed_event) * 65536))) return e; }
        ctx->events_cap_dev = (int64_t)(ctx->b_events.cap / sizeof(cg_bed_event));
        LdEvCount le = { D->ev }; StEvents se = { (cg_bed_event *)ctx->b_events.p, D->ev, *D, ctx->events_cap_dev };
        if ((e = run_scan<int32_t, OpSum>(ctx, le, se, nc, 0, &scal->h.n_events))) return e;
        if (D->want_dump) { k_dump_flags<<<nblk(nc, 256), 256, 0, st>>>(*D); ctx->launches++; }
    }
    if (timed) T1(CG_T_EVENTS);
    T1(CG_T_TOTAL);
    CG_CHECK(cudaMemcpyAsync(ctx->h_dims, &scal->h, sizeof(CgScalHead), cudaMemcpyDeviceToHost, st));
    CG_CHECK(cudaMemcpyAsync(ctx->h_counters, D->counters, sizeof(unsigned long long) * CG_N_COUNTERS, cudaMemcpyDeviceToHost, st));
    CG_CHECK(cudaStreamSynchronize(st));
    CG_CHECK(cudaGetLastError());
    for (int i = 0; i < CG_N_TIMERS; i++) {
        if (i == CG_T_H2D || i == CG_T_D2H) continue;
        if (!timed && i != CG_T_TOTAL && i != CG_T_TILES) continue;
        read_timer(ctx, i);
    }
    if (ctx->h_dims->err) { snprintf(ctx->err, sizeof ctx->err, "device reported error %d", ctx->h_dims->err); return ctx->h_dims->err; }
    if (ctx->h_dims->n_events > ctx->events_cap_dev) {
        /* more BED events than the device list holds: grow and redo the (cheap) ordered scatter */
        if ((e = ensure(ctx, &ctx->b_events, sizeof(cg_bed_event) * ((size_t)ctx->h_dims->n_events + 1024)))) return e;
        ctx->events_cap_dev = (int64_t)(ctx->b_events.cap / sizeof(cg_bed_event));
        LdEvCount le = { D->ev }; StEvents se = { (cg_bed_event *)ctx->b_events.p, D->ev, *D, ctx->events_cap_dev };
        if ((e = run_scan<int32_t, OpSum>(ctx, le, se, nc, 0, &scal->h.n_events))) return e;
        CG_CHECK(cudaStreamSynchronize(st));
    }
    ctx->resident = 2;
    return 0;
}

extern "C" int cg_run(cg_ctx *ctx) {
    if (!ctx->resident || stream_busy(ctx)) return CG_ERR_STATE;
    CG_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    CgBounds B; memset(&B, 0, sizeof B); B.n = 1; B.rb[0] = ctx->D.n_reads;
    int64_t hb[3 * CG_MAX_CHUNKS];
    int e;
    T0(CG_T_TOTAL);
    if ((e = run_prep(ctx, &B, hb))) return e;
    CgSlice sl; memset(&sl, 0, sizeof sl);
    sl.t1 = ctx->D.n_tiles; sl.c1 = ctx->D.n_cols; sl.r1 = ctx->D.n_reads; sl.je = ctx->D.n_pile;
    if ((e = slice_A(ctx, &sl, 1)) || (e = slice_B(ctx, &sl, 3, 1))) return e;
    return run_finish(ctx, 1);
}

/* events, counters, column dump (small); the qualities only when q_too */
static int download_results(cg_ctx *ctx, cg_result *out, int q_too) {
    cudaStream_t st = ctx->stream;
    if (q_too) T0(CG_T_D2H);
    if (q_too && out->qual_out && ctx->qual_bytes) CG_CHECK(cudaMemcpyAsync(out->qual_out, ctx->b_qout.p, (size_t)ctx->qual_bytes, cudaMemcpyDeviceToHost, st));
    out->n_events = ctx->h_dims->n_events;
    if (out->events && out->n_events) {
        int64_t k = out->n_events < out->events_cap ? out->n_events : out->events_cap;
        if (k) CG_CHECK(cudaMemcpyAsync(out->events, ctx->b_events.p, sizeof(cg_bed_event) * (size_t)k, cudaMemcpyDeviceToHost, st));
    }
    out->n_columns = 0;
    cg_column *tmp = NULL;
    if (out->columns && ctx->D.want_dump && ctx->D.n_cols) {
        tmp = (cg_column *)malloc(sizeof(cg_column) * (size_t)ctx->D.n_cols);
        if (!tmp) return CG_ERR_NOMEM;
        CG_CHECK(cudaMemcpyAsync(tmp, ctx->b_dump.p, sizeof(cg_column) * (size_t)ctx->D.n_cols, cudaMemcpyDeviceToHost, st));
    }
    if (q_too) T1(CG_T_D2H);
    CG_CHECK(cudaStreamSynchronize(st));
    for (int i = 0; i < CG_N_COUNTERS; i++) out->counters[i] = (int64_t)ctx->h_counters[i];
    if (ctx->h_dims->beyond) out->counters[CG_CNT_COLUMNS]++;   /* snp_score.c:1476 runs before the region break at 1516-1517 */
    if (tmp) {
        for (int c = 0; c < ctx->D.n_cols; c++) {
            if (tmp[c].tid < 0) continue;
            if (out->n_columns < out->columns_cap) out->columns[out->n_columns] = tmp[c];
            out->n_columns++;
        }
        free(tmp);
    }
    return 0;
}

extern "C" int cg_download(cg_ctx *ctx, cg_result *out) {
    if (ctx->resident != 2) return CG_ERR_STATE;
    CG_CHECK(cudaSetDevice(ctx->device));
    int e = download_results(ctx, out, 1);
    if (e) return e;
    read_copy_timers(ctx);
    return 0;
}

/* ---- records already in GPU memory (cg_process_device) ---------------------------------------------------------------------------
 * The per-record arrays and the CIGARs are copied device to device into the working buffers (so the caller's buffers are free once
 * the stream has passed the call) and the batch is treated as packed: the scans cg_run would run rebuild off[] and cigar_off[] here,
 * two more give where every record starts in the caller's arrays, and all sums are checked at one host synchronisation before any
 * kernel uses an offset.  k_ingest repacks qualities and sequences into the padded working layout, the resident chain runs as in
 * cg_run, and k_emit gathers the rewritten qualities into the caller's concatenated layout.  One warp per record; the per-item
 * bodies (cg_pipeline.h) are the emulation's. */
#define IO_THREADS 256
__global__ void __launch_bounds__(IO_THREADS) k_ingest(const __grid_constant__ CgIngest I, int64_t n) {
    const int64_t r = ((int64_t)blockIdx.x * IO_THREADS + threadIdx.x) >> 5;
    if (r >= n) return;
    const int ng = (I.l_qseq[r] + 7) >> 3;
    for (int k = threadIdx.x & 31; k < ng; k += 32) cg_ingest_group(&I, r, k);
}
__global__ void __launch_bounds__(IO_THREADS) k_emit(const __grid_constant__ CgEmit E, int64_t n) {
    const int64_t r = ((int64_t)blockIdx.x * IO_THREADS + threadIdx.x) >> 5;
    if (r >= n) return;
    const int nw = cg_emit_words(&E, r);
    for (int j = threadIdx.x & 31; j < nw; j += 32) cg_emit_word(&E, r, j);
}
struct LdLen { const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return (int64_t)lq[i]; } };
struct LdHalf { const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return ((int64_t)lq[i] + 1) >> 1; } };
struct LdNeg { const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return lq[i] < 0 ? 1 : 0; } };
struct LdNCig64 { const uint16_t *nc; __device__ int64_t operator()(int64_t i) const { return (int64_t)nc[i]; } };
struct StExcl32of64 { int32_t *p; __device__ void operator()(int64_t i, int64_t, int64_t ex) const { p[i] = (int32_t)ex; } };
struct StNone { __device__ void operator()(int64_t, int64_t, int64_t) const {} };

static int dev_ptr_check(cg_ctx *ctx, const void *p, int64_t count, const char *name) {
    if (count == 0) return 0;
    cudaPointerAttributes a;
    if (p && cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeDevice && a.device == ctx->device) return 0;
    cudaGetLastError();
    snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: %s is not device memory of device %d", name, ctx->device);
    return CG_ERR_BAD_ARG;
}

/* what cg_process_device and cg_stream_device reject before anything is enqueued; n_total / cig_total / q_total: the working batch */
static int dev_check(cg_ctx *ctx, const cg_dev_batch *in, const uint8_t *qual_out, int64_t qual_cnt, const cg_result *out, int64_t n_total, int64_t cig_total, int64_t q_total) {
    const int64_t n = in->n_reads;
    if (n < 0 || in->n_cigar_total < 0 || in->seq_len < 0 || in->qual_len < 0) {
        snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: negative count (n_reads %lld, n_cigar_total %lld, seq_len %lld, qual_len %lld)",
                 (long long)n, (long long)in->n_cigar_total, (long long)in->seq_len, (long long)in->qual_len);
        return CG_ERR_BAD_ARG;
    }
    if (out->qual_out || out->qual_head) { snprintf(ctx->err, sizeof ctx->err, "the qualities go to qual_out; out->qual_out and out->qual_head must be NULL"); return CG_ERR_BAD_ARG; }
    if (n_total > 0x7fffff00LL || cig_total > 0x7fffff00LL || q_total + 8 * n_total >= (1LL << 35)) { snprintf(ctx->err, sizeof ctx->err, "batch too large: split it"); return CG_ERR_BAD_ARG; }
    int e;
    if ((e = dev_ptr_check(ctx, in->tid, n, "tid")) || (e = dev_ptr_check(ctx, in->pos, n, "pos")) || (e = dev_ptr_check(ctx, in->flag, n, "flag")) ||
        (e = dev_ptr_check(ctx, in->mapq, n, "mapq")) || (e = dev_ptr_check(ctx, in->l_qseq, n, "l_qseq")) || (e = dev_ptr_check(ctx, in->n_cigar, n, "n_cigar")) ||
        (e = dev_ptr_check(ctx, in->cigar, in->n_cigar_total, "cigar")) || (e = dev_ptr_check(ctx, in->seq, in->seq_len, "seq")) ||
        (e = dev_ptr_check(ctx, in->qual, in->qual_len, "qual")) || (e = dev_ptr_check(ctx, qual_out, qual_cnt, "qual_out"))) return e;
    return 0;
}

/* The records held for a stream (none for cg_process_device) followed by `in`, as one packed working batch: per-record arrays and CIGARs
 * copied device to device, the running sums of the padded lengths, n_cigar, l_qseq, (l_qseq + 1) / 2 and the count of negative lengths.
 * before_sync() enqueues whatever else must come back at the one synchronisation; then the sums are checked.  The held records' bytes are
 * already in the padded layout and go to the front of the working arrays; `in`'s go through k_ingest (dev_ingest) afterwards. */
template <class F>
static int dev_stage(cg_ctx *ctx, const cg_dev_batch *in, F before_sync) {
    cudaStream_t st = ctx->stream;
    const int64_t nh = ctx->st_n, ni = in->n_reads, n = nh + ni;
    int e;
    cg_batch hb; memset(&hb, 0, sizeof hb);                     /* the padded lengths of `in` sum to at most qual_len + 7 per record */
    hb.n_reads = n; hb.n_cigar_total = ctx->st_cig + in->n_cigar_total; hb.qual_bytes = ctx->st_padded + in->qual_len + 7 * ni;
    hb.seq_bytes = (hb.qual_bytes + 1) / 2; hb.packed = 1;
    if ((e = alloc_inputs(ctx, &hb))) return e;
    if ((e = ensure(ctx, &ctx->b_qsrc, ((size_t)n + 1) * 8)) || (e = ensure(ctx, &ctx->b_ssrc, ((size_t)n + 1) * 8)) || (e = ensure(ctx, &ctx->b_dvsum, 64)) ||
        (e = ensure(ctx, &ctx->b_scal, sizeof(CgScalars))) || (e = ensure(ctx, &ctx->b_rspan, ((size_t)n + 1) * 4))) return e;
    CgDev *D = &ctx->D;
    D->rspan = (int32_t *)ctx->b_rspan.p; D->err = &((CgScalars *)ctx->b_scal.p)->h.err;
    int64_t h[5] = { 0, 0, 0, 0, 0 };                            /* [0] padded lengths [1] n_cigar [2] l_qseq [3] (l_qseq + 1) / 2 [4] negative l_qseq */
    if (n > 0) {
        if (nh > 0) {
            CG_CHECK(cudaMemcpyAsync(ctx->b_tid.p, ctx->b_htid.p, (size_t)nh * 4, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync(ctx->b_pos.p, ctx->b_hpos.p, (size_t)nh * 4, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync(ctx->b_flag.p, ctx->b_hflag.p, (size_t)nh * 2, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync(ctx->b_mapq.p, ctx->b_hmapq.p, (size_t)nh, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync(ctx->b_lq.p, ctx->b_hlq.p, (size_t)nh * 4, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync(ctx->b_nc.p, ctx->b_hnc.p, (size_t)nh * 2, cudaMemcpyDeviceToDevice, st));
            if (ctx->st_cig) CG_CHECK(cudaMemcpyAsync(ctx->b_cigar.p, ctx->b_hcig.p, (size_t)ctx->st_cig * 4, cudaMemcpyDeviceToDevice, st));
            if (ctx->st_padded) {
                CG_CHECK(cudaMemcpyAsync((char *)ctx->b_qual.p + CG_FRONT_PAD, ctx->b_hqual.p, (size_t)ctx->st_padded, cudaMemcpyDeviceToDevice, st));
                CG_CHECK(cudaMemcpyAsync((char *)ctx->b_seq.p + CG_FRONT_PAD, ctx->b_hseq.p, (size_t)ctx->st_padded / 2, cudaMemcpyDeviceToDevice, st));
            }
        }
        if (ni > 0) {
            CG_CHECK(cudaMemcpyAsync((int32_t *)ctx->b_tid.p + nh, in->tid, (size_t)ni * 4, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync((int32_t *)ctx->b_pos.p + nh, in->pos, (size_t)ni * 4, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync((uint16_t *)ctx->b_flag.p + nh, in->flag, (size_t)ni * 2, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync((uint8_t *)ctx->b_mapq.p + nh, in->mapq, (size_t)ni, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync((int32_t *)ctx->b_lq.p + nh, in->l_qseq, (size_t)ni * 4, cudaMemcpyDeviceToDevice, st));
            CG_CHECK(cudaMemcpyAsync((uint16_t *)ctx->b_nc.p + nh, in->n_cigar, (size_t)ni * 2, cudaMemcpyDeviceToDevice, st));
            if (in->n_cigar_total) CG_CHECK(cudaMemcpyAsync((uint32_t *)ctx->b_cigar.p + ctx->st_cig, in->cigar, (size_t)in->n_cigar_total * 4, cudaMemcpyDeviceToDevice, st));
        }
        int64_t *sums = (int64_t *)ctx->b_dvsum.p;
        LdPad8 lp = { D->l_qseq }; StExcl64 so = { (int64_t *)ctx->b_off.p };
        LdNCig64 ln = { D->n_cigar }; StExcl32of64 sc = { (int32_t *)ctx->b_coff.p };
        LdLen ll = { D->l_qseq }; StExcl64 sq = { (int64_t *)ctx->b_qsrc.p };
        LdHalf lh = { D->l_qseq }; StExcl64 ss = { (int64_t *)ctx->b_ssrc.p };
        LdNeg lneg = { D->l_qseq }; StNone none;
        if ((e = run_scan<int64_t, OpSum>(ctx, lp, so, n, (int64_t)0, sums + 0)) || (e = run_scan<int64_t, OpSum>(ctx, ln, sc, n, (int64_t)0, sums + 1)) ||
            (e = run_scan<int64_t, OpSum>(ctx, ll, sq, n, (int64_t)0, sums + 2)) || (e = run_scan<int64_t, OpSum>(ctx, lh, ss, n, (int64_t)0, sums + 3)) ||
            (e = run_scan<int64_t, OpSum>(ctx, lneg, none, n, (int64_t)0, sums + 4))) return e;
        if ((e = before_sync(sums))) return e;
        CG_CHECK(cudaMemcpyAsync(h, sums, sizeof h, cudaMemcpyDeviceToHost, st));
        CG_CHECK(cudaStreamSynchronize(st));
        if (h[4]) { snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: %lld records have a negative l_qseq", (long long)h[4]); return CG_ERR_BAD_ARG; }
        if (h[2] != ctx->st_qual + in->qual_len || h[3] != ctx->st_seq + in->seq_len || h[1] != ctx->st_cig + in->n_cigar_total) {
            snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: the records hold %lld quality bytes (qual_len %lld), %lld sequence bytes (seq_len %lld), %lld CIGAR operations (n_cigar_total %lld)",
                     (long long)(h[2] - ctx->st_qual), (long long)in->qual_len, (long long)(h[3] - ctx->st_seq), (long long)in->seq_len,
                     (long long)(h[1] - ctx->st_cig), (long long)in->n_cigar_total);
            return CG_ERR_BAD_ARG;
        }
    }
    ctx->qual_bytes = h[0]; ctx->offsets_ready = 1;
    return 0;
}

/* `in`'s qualities and sequences into the padded working layout, behind the held records */
static int dev_ingest(cg_ctx *ctx, const cg_dev_batch *in) {
    const int64_t nh = ctx->st_n, ni = in->n_reads;
    if (ni <= 0) return 0;
    const CgDev *D = &ctx->D;
    const CgIngest I = { D->l_qseq + nh, D->off + nh, (const int64_t *)ctx->b_qsrc.p + nh, (const int64_t *)ctx->b_ssrc.p + nh, in->qual, in->seq,
                         (uint8_t *)ctx->b_qual.p + CG_FRONT_PAD, (uint8_t *)ctx->b_seq.p + CG_FRONT_PAD, ctx->st_qual, ctx->st_seq };
    k_ingest<<<(unsigned)nblk(ni * 32, IO_THREADS), IO_THREADS, 0, ctx->stream>>>(I, ni);
    CG_CHECK(cudaGetLastError());
    return 0;
}

/* the rewritten qualities of working records [r0, r1) to qual_out, which starts at record r0 */
static int dev_emit(cg_ctx *ctx, int64_t r0, int64_t r1, int64_t qbase, uint8_t *qual_out) {
    if (r1 <= r0) return 0;
    const CgDev *D = &ctx->D;
    const CgEmit E = { D->l_qseq + r0, D->off + r0, (const int64_t *)ctx->b_qsrc.p + r0, (const uint8_t *)ctx->b_qout.p, qual_out, qbase };
    k_emit<<<(unsigned)nblk((r1 - r0) * 32, IO_THREADS), IO_THREADS, 0, ctx->stream>>>(E, r1 - r0);
    ctx->launches++;
    CG_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int cg_process_device(cg_ctx *ctx, const cg_dev_batch *in, uint8_t *qual_out, cg_result *out) {
    if (!ctx) return CG_ERR_BAD_ARG;
    if (stream_busy(ctx)) return CG_ERR_STATE;
    if (!in || !out) { snprintf(ctx->err, sizeof ctx->err, "cg_process_device: no batch or no result"); return CG_ERR_BAD_ARG; }
    CG_CHECK(cudaSetDevice(ctx->device));
    int e;
    if ((e = dev_check(ctx, in, qual_out, in->qual_len, out, in->n_reads, in->n_cigar_total, in->qual_len))) return e;
    ctx->resident = 0; ctx->win_on = 0;
    ctx->dump_columns = out->columns != NULL;
    if ((e = dev_stage(ctx, in, [](int64_t *) { return 0; }))) return e;
    const int64_t n = in->n_reads;
    cudaStream_t st = ctx->stream;
    T0(CG_T_H2D);
    if ((e = dev_ingest(ctx, in))) return e;
    T1(CG_T_H2D);
    ctx->resident = 1;
    if ((e = cg_run(ctx))) return e;
    T0(CG_T_D2H);
    if (in->qual_len > 0 && (e = dev_emit(ctx, 0, n, 0, qual_out))) return e;
    T1(CG_T_D2H);
    if ((e = download_results(ctx, out, 0))) return e;          /* events, counters, column dump; synchronises the stream */
    read_copy_timers(ctx);
    ctx->h2d_bytes = 0;
    return 0;
}

/* ---- streams (cg_stream_device) ----------------------------------------------------------------------------------------------------
 * k_stream_plan reduces the cut quantities of the working batch (one thread per record, warp reductions, one atomic per warp and field),
 * k_stream_cut turns them into the cut, k_stream_keep flags the records held for later calls, and three scans over the flag give where
 * k_retain puts each of them in the held store.  All of it before the call's one synchronisation. */
__global__ void k_stream_init(CgStreamRed *red) { cg_stream_red_init(red); }
__global__ void __launch_bounds__(256) k_stream_plan(const __grid_constant__ CgDev D, int64_t n, int64_t n_held, int64_t e0, CgStreamRed *red) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    CgStreamRed c;
    if (r < n) c = cg_stream_plan_item(&D, r, n, n_held, e0); else cg_stream_red_init(&c);
    const unsigned all = 0xffffffffu;
    c.mmax = __reduce_max_sync(all, c.mmax); c.mtid = __reduce_max_sync(all, c.mtid);
    c.smin = __reduce_min_sync(all, c.smin); c.fmin = __reduce_min_sync(all, c.fmin);
    c.unplaced = __reduce_or_sync(all, (unsigned)c.unplaced);
    for (int o = 16; o > 0; o >>= 1) {
        const uint64_t a = __shfl_xor_sync(all, c.kmin, o), b = __shfl_xor_sync(all, c.kmax, o);
        if (a < c.kmin) c.kmin = a;
        if (b > c.kmax) c.kmax = b;
    }
    if ((threadIdx.x & 31) == 0) {
        if (c.mmax >= 0) atomicMax(&red->mmax, c.mmax);
        if (c.mtid >= 0) atomicMax(&red->mtid, c.mtid);
        if (c.smin != 0x7fffffff) atomicMin(&red->smin, c.smin);
        if (c.fmin != 0x7fffffff) atomicMin(&red->fmin, c.fmin);
        if (c.kmin <= c.kmax) { atomicMin((unsigned long long *)&red->kmin, (unsigned long long)c.kmin); atomicMax((unsigned long long *)&red->kmax, (unsigned long long)c.kmax); }
        if (c.unplaced) atomicOr(&red->unplaced, 1);
    }
}
__global__ void k_stream_cut(const __grid_constant__ CgDev D, const CgStreamRed *red, CgStreamCut *cut, int64_t n, int64_t e0, int last, const int64_t *qsrc, const int64_t *q_total) {
    *cut = cg_stream_cut(&D, red, n, e0, last, qsrc, *q_total);
}
__global__ void __launch_bounds__(256) k_stream_keep(const __grid_constant__ CgDev D, const CgStreamCut *cut, uint8_t *keep, int64_t n) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) keep[r] = (uint8_t)cg_stream_keep(&D, r, cut);
}
__global__ void __launch_bounds__(IO_THREADS) k_retain(const __grid_constant__ CgRetain K, const uint8_t *__restrict__ keep, int64_t n) {
    const int64_t r = ((int64_t)blockIdx.x * IO_THREADS + threadIdx.x) >> 5;
    if (r >= n || !keep[r]) return;
    const int ni = cg_retain_items(&K, r);
    for (int j = threadIdx.x & 31; j < ni; j += 32) cg_retain_item(&K, r, j);
}
struct LdKeep { const uint8_t *keep; __device__ int64_t operator()(int64_t i) const { return keep[i]; } };
struct LdKeepPad { const uint8_t *keep; const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return keep[i] ? (((int64_t)lq[i] + 7) & ~(int64_t)7) : 0; } };
struct LdKeepCig { const uint8_t *keep; const uint16_t *nc; __device__ int64_t operator()(int64_t i) const { return keep[i] ? (int64_t)nc[i] : 0; } };
struct LdKeepLen { const uint8_t *keep; const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return keep[i] ? (int64_t)lq[i] : 0; } };
struct LdKeepHalf { const uint8_t *keep; const int32_t *lq; __device__ int64_t operator()(int64_t i) const { return keep[i] ? ((int64_t)lq[i] + 1) >> 1 : 0; } };

/* the qualities of records [r0, r1) go home on the download stream once everything queued on the compute stream so far is done;
 * bytes below out->head_bytes (a region shard's read halo) go to out->qual_head instead of out->qual_out */
static int enqueue_d2h(cg_ctx *ctx, const cg_batch *in, cg_result *out, int64_t r0, int64_t r1, int chunk) {
    const int64_t n = in->n_reads;
    if (r1 <= r0 || (!out->qual_out && !out->qual_head)) return 0;
    int64_t b0 = in->off[r0], b1 = r1 < n ? in->off[r1] : in->qual_bytes;
    CG_CHECK(cudaEventRecord(ctx->ev_done[chunk], ctx->stream));
    CG_CHECK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_done[chunk], 0));
    const int64_t hb = out->qual_head ? out->head_bytes : 0;
    if (b0 < hb) {
        const int64_t e1 = b1 < hb ? b1 : hb;
        CG_CHECK(cudaMemcpyAsync(out->qual_head + b0, (char *)ctx->b_qout.p + b0, (size_t)(e1 - b0), cudaMemcpyDeviceToHost, ctx->s_d2h));
        b0 = e1;
    }
    if (b1 > b0 && out->qual_out) CG_CHECK(cudaMemcpyAsync(out->qual_out + b0, (char *)ctx->b_qout.p + b0, (size_t)(b1 - b0), cudaMemcpyDeviceToHost, ctx->s_d2h));
    return 0;
}

/* CG_TRACE: the host-side timeline of a streamed call on stderr (t0 = NULL: off) */
static void trace_at(const struct timespec *t0, const char *what, int i) {
    if (!t0) return;
    struct timespec t1; clock_gettime(CLOCK_MONOTONIC, &t1);
    fprintf(stderr, "[cg_process] %8.3f ms  %s %d\n", (t1.tv_sec - t0->tv_sec) * 1e3 + (t1.tv_nsec - t0->tv_nsec) * 1e-6, what, i);
}

/* the end of a streamed call (process_streamed, cg_shard_end), once every slice's downloads are queued: events, counters and dumps,
 * then both copy streams drained */
static int finish_streamed(cg_ctx *ctx, cg_result *out, const cg_window *win, int timed, const struct timespec *trace) {
    cudaEventRecord(ctx->ev[CG_T_D2H][1], ctx->s_d2h);
    /* a call without any pileup column (placed-unmapped reads in a coverage gap) leaves the state it resumed from untouched */
    if (win) ctx->have_saved = win->hi_tid >= 0 && (ctx->D.n_cols > 0 || (!win->first && ctx->have_saved));
    int e = run_finish(ctx, timed);
    ctx->win_on = 0;
    if (e) return e;
    trace_at(trace, "finish done", 0);
    if ((e = download_results(ctx, out, 0))) return e;
    CG_CHECK(cudaStreamSynchronize(ctx->s_d2h));
    trace_at(trace, "d2h drained", 0);
    CG_CHECK(cudaStreamSynchronize(ctx->s_h2d));
    read_copy_timers(ctx);
    return 0;
}

/* End to end, streamed: the base data goes up in chunks on a copy stream; slice i of the chain starts when chunk i has
 * landed; the qualities of the records it finalises go down on a second copy stream while later chunks still arrive.
 * phase 0: everything (cg_process / cg_process_window).  phase 1: a region shard's part A only (cg_shard_begin): its slices are
 * recorded in the context for cg_shard_carry (B1) and cg_shard_end (B2 + downloads). */
static int process_streamed(cg_ctx *ctx, const cg_batch *in, cg_result *out, const cg_window *win, int phase) {
    CG_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    int e;
    /* a resident batch: a region shard on the batch cg_upload left on the device (timing the chain alone, phase 1), or one call of a
     * stream on the batch cg_stream_device ingested (phase 0 with a window; its qualities stay on the device) */
    const int res_mode = in == NULL;
    if (res_mode && !ctx->resident) return CG_ERR_STATE;
    ctx->win_on = 0; ctx->n_sl = 0; ctx->shard_state = 0;
    ctx->dump_columns = out->columns != NULL;
    if (!res_mode) { ctx->resident = 0; if ((e = alloc_inputs(ctx, in))) return e; }
    if (win) {                                                 /* one call of a chain (cg_process_window) */
        if ((e = ensure(ctx, &ctx->b_saved, sizeof(CgSavedCarry)))) return e;
        ctx->win = *win; ctx->win_on = 1; ctx->depth_matters = 0;
    }
    if (!ctx->s_h2d) {
        CG_CHECK(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking));
        CG_CHECK(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < CG_MAX_CHUNKS; i++) {
            CG_CHECK(cudaEventCreateWithFlags(&ctx->ev_up[i], cudaEventDisableTiming));
            CG_CHECK(cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming));
        }
        CG_CHECK(cudaEventCreateWithFlags(&ctx->ev_misc, cudaEventDisableTiming));
    }
    /* chunk the records by quality bytes (about 96 MB per chunk, at most CG_MAX_CHUNKS) */
    const int64_t n = res_mode ? ctx->D.n_reads : in->n_reads;
    const int64_t qbytes = res_mode ? ctx->qual_bytes : in->qual_bytes;
    int nch = res_mode ? 1 : (int)(qbytes / (ctx->chunk_bytes > 0 ? ctx->chunk_bytes : (96LL << 20))) + 1;
    if (nch > CG_MAX_CHUNKS) nch = CG_MAX_CHUNKS;
    if (n < nch) nch = n > 0 ? (int)n : 1;
    CgBounds B; memset(&B, 0, sizeof B); B.n = nch;
    int64_t boff[CG_MAX_CHUNKS + 1]; boff[0] = 0;
    for (int i = 0; i < nch; i++) {
        int64_t r = n;
        if (i + 1 < nch) {
            /* equal chunks, except that the last two are 1/2 and 1/4 of a chunk: what remains to be done after the last
             * byte has landed (last slice + its download) shrinks with the last chunk */
            const double wtot = nch >= 4 ? (nch - 2) + 0.75 : (double)nch;
            const double wacc = nch >= 4 ? (i + 1 <= nch - 2 ? (double)(i + 1) : (nch - 2) + 0.5) : (double)(i + 1);
            const int64_t target = (int64_t)((double)qbytes * (wacc / wtot));
            int64_t lo = i ? B.rb[i - 1] : 0, hi = n;
            while (lo < hi) { int64_t mid = (lo + hi) >> 1; if (in->off[mid] < target) lo = mid + 1; else hi = mid; }
            r = lo;
        }
        B.rb[i] = r;
        boff[i + 1] = r < n ? in->off[r] : qbytes;
    }
    T0(CG_T_TOTAL);
    cudaEventRecord(ctx->ev[CG_T_H2D][0], st);
    if (!res_mode && (e = upload_meta(ctx, in, st))) return e;
    /* the copy stream must not run ahead of buffer (re)allocation or of earlier users of the buffers: order it after st */
    CG_CHECK(cudaEventRecord(ctx->ev_misc, st));
    CG_CHECK(cudaStreamWaitEvent(ctx->s_h2d, ctx->ev_misc, 0));
    CG_CHECK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_misc, 0));
    for (int i = 0; i < nch; i++) {
        if (!res_mode && (e = upload_bases(ctx, in, boff[i], boff[i + 1], ctx->s_h2d))) return e;
        CG_CHECK(cudaEventRecord(ctx->ev_up[i], ctx->s_h2d));
    }
    cudaEventRecord(ctx->ev[CG_T_H2D][1], ctx->s_h2d);
    int64_t hb[3 * CG_MAX_CHUNKS];
    struct timespec ts0; clock_gettime(CLOCK_MONOTONIC, &ts0);
    const struct timespec *trace = getenv("CG_TRACE") ? &ts0 : NULL;
    if ((e = run_prep(ctx, &B, hb))) { ctx->win_on = 0; return e; }
    trace_at(trace, "prep done, chunks", nch);
    /* chained call: re-open the window the previous call left active, find the column where the state is saved for the next one */
    CgChainCarry *ccarry = &((CgScalars *)ctx->b_scal.p)->chain;
    CgEpochCarry *ecarry = &((CgScalars *)ctx->b_scal.p)->epoch;
    int cS = -1;                                               /* -1: nothing to save */
    if (win && ctx->D.n_cols > 0) {
        if (phase == 0 && !win->first && ctx->have_saved) { k_paint_carry<<<1, 32, 0, st>>>(ctx->D, ccarry, win->lo_tid, win->lo_pos); ctx->launches++; }
        if (win->hi_tid >= 0) {
            k_find_col<<<1, 32, 0, st>>>(ctx->D, win->hi_tid, win->next_lo_pos, &ctx->d_hdims->next_col); ctx->launches++;
            CG_CHECK(cudaStreamSynchronize(st));
            cS = ctx->h_dims->next_col;
        }
    }
    int tprev = 0, jprev = 0; int64_t rprev = 0;
    if (phase == 0) cudaEventRecord(ctx->ev[CG_T_D2H][0], ctx->s_d2h);
    for (int i = 0; i < nch; i++) {
        int t1 = (i + 1 == nch) ? ctx->D.n_tiles : (int)hb[3 * i];
        int64_t r1 = (i + 1 == nch) ? n : hb[3 * i + 1];
        int j1 = (i + 1 == nch) ? ctx->D.n_pile : (int)hb[3 * i + 2];
        if (t1 < tprev) t1 = tprev;
        if (r1 < rprev) r1 = rprev;
        if (j1 < jprev) j1 = jprev;
        CG_CHECK(cudaStreamWaitEvent(st, ctx->ev_up[i], 0));
        if (!res_mode && (e = expand_bases(ctx, in, boff[i], boff[i + 1], st))) { ctx->win_on = 0; return e; }
        const int c0 = tprev * 32 < ctx->D.n_cols ? tprev * 32 : ctx->D.n_cols, c1 = t1 * 32 < ctx->D.n_cols ? t1 * 32 : ctx->D.n_cols;
        /* the slice(s) of this chunk: when the next call's first column cS lies inside, the sparse passes stop there, both carries are
         * saved, and a second slice (no tiles of its own) finishes the columns from cS on */
        CgSlice sl[2]; int ns = 1;
        memset(sl, 0, sizeof sl);
        sl[0].t0 = tprev; sl[0].t1 = t1; sl[0].c0 = c0; sl[0].c1 = c1; sl[0].jb = jprev; sl[0].je = j1; sl[0].r0 = rprev; sl[0].r1 = r1; sl[0].chunk = i;
        if (cS >= 0 && cS < c1) {
            sl[1] = sl[0];
            sl[0].c1 = cS; sl[0].r0 = sl[0].r1 = 0; sl[0].save_after = 1;
            sl[1].t0 = sl[1].t1 = t1; sl[1].c0 = cS; sl[1].jb = sl[1].je = j1;
            ns = 2; cS = -2;                                   /* saved (or about to be) */
        }
        for (int k = 0; k < ns; k++) {
            if ((e = slice_A(ctx, &sl[k], res_mode && k == 0))) { ctx->win_on = 0; return e; }   /* stage timers on a resident batch: the slice that owns the tiles */
            if (phase == 0) {
                if ((e = slice_B(ctx, &sl[k], 3, 0))) { ctx->win_on = 0; return e; }
                if (sl[k].save_after) { k_carry_save<<<1, 32, 0, st>>>(ccarry, ecarry, (CgSavedCarry *)ctx->b_saved.p); ctx->launches++; }
            } else ctx->sl[ctx->n_sl++] = sl[k];
        }
        if (phase == 0 && !res_mode && (e = enqueue_d2h(ctx, in, out, rprev, r1, i))) { ctx->win_on = 0; return e; }
        tprev = t1; rprev = r1; jprev = j1;
        trace_at(trace, "slice enqueued (host passed its column sync)", i);
    }
    if (phase != 0) {                                          /* a region shard: the rest follows in cg_shard_carry / cg_shard_end */
        ctx->shard_in = in; ctx->shard_save_end = cS >= 0; ctx->shard_state = 1; ctx->shard_timed = res_mode;
        return 0;
    }
    if (cS >= 0) { k_carry_save<<<1, 32, 0, st>>>(ccarry, ecarry, (CgSavedCarry *)ctx->b_saved.p); ctx->launches++; }   /* next call starts beyond this batch's columns */
    return finish_streamed(ctx, out, win, 0, trace);
}

/* ---- region shards of one contig on several devices at once (include/crumble_gpu.h) -------------------------------------------
 * cg_shard_begin   upload + part A of every slice (no carried state): all shards run this concurrently;
 * cg_shard_carry   the true incoming state (from the shard on the left, or none at a contig start) -> part B1 of the slices below the
 *                  right neighbour's first column -> the outgoing state.  Small (prefix sums, epochs, window chain), and the only
 *                  thing that runs shard after shard;
 * cg_shard_end     part B1 of the remaining slices, part B2 (over-depth test, painting, rewrite), downloads: concurrent again. */
extern "C" int cg_shard_begin(cg_ctx *ctx, const cg_batch *in, const cg_window *win, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    if (!win) return CG_ERR_BAD_ARG;
    if (ctx->params.region_tid >= 0) { snprintf(ctx->err, sizeof ctx->err, "region shards and a -r region do not combine"); return CG_ERR_BAD_ARG; }
    cg_window w = *win;
    if (w.first == 2) w.first = 0;                             /* there is no speculative start here: the true state arrives in cg_shard_carry */
    return process_streamed(ctx, in, out, &w, 1);
}

extern "C" int cg_shard_carry(cg_ctx *ctx, const void *carry_in, void *carry_out) {
    if (ctx->shard_state != 1 || stream_busy(ctx)) return CG_ERR_STATE;
    CG_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    CgChainCarry *ccarry = &((CgScalars *)ctx->b_scal.p)->chain;
    CgEpochCarry *ecarry = &((CgScalars *)ctx->b_scal.p)->epoch;
    int e;
    if (!ctx->win.first) {
        if (!carry_in) { snprintf(ctx->err, sizeof ctx->err, "this shard continues a contig: it needs the state of the shard on its left"); return CG_ERR_BAD_ARG; }
        CgSavedCarry sv; memcpy(&sv, carry_in, sizeof sv);
        memcpy(ctx->h_carry_io, &sv, sizeof sv);
        CG_CHECK(cudaMemcpyAsync(ccarry, &((CgSavedCarry *)ctx->h_carry_io)->cc, sizeof(CgChainCarry), cudaMemcpyHostToDevice, st));
        CG_CHECK(cudaMemcpyAsync(ecarry, &((CgSavedCarry *)ctx->h_carry_io)->ec, sizeof(CgEpochCarry), cudaMemcpyHostToDevice, st));
        ctx->have_saved = 1;
    }
    int k = 0;
    for (; k < ctx->n_sl; k++) {
        if ((e = slice_B(ctx, &ctx->sl[k], 1, 0))) return e;
        if (ctx->sl[k].save_after) { k++; break; }
    }
    ctx->shard_next = k;
    const int saves = (k > 0 && ctx->sl[k - 1].save_after) || ctx->shard_save_end;
    if (saves) {
        if (ctx->shard_save_end) for (; k < ctx->n_sl; k++) if ((e = slice_B(ctx, &ctx->sl[k], 1, 0))) return e;    /* the next shard starts beyond these columns */
        ctx->shard_next = k;
        k_carry_save<<<1, 32, 0, st>>>(ccarry, ecarry, (CgSavedCarry *)ctx->b_saved.p); ctx->launches++;
        if (carry_out) {
            CG_CHECK(cudaMemcpyAsync(ctx->h_carry_io + CG_CARRY_BYTES, ctx->b_saved.p, sizeof(CgSavedCarry), cudaMemcpyDeviceToHost, st));
            CG_CHECK(cudaStreamSynchronize(st));
            memset(carry_out, 0, CG_CARRY_BYTES);
            memcpy(carry_out, ctx->h_carry_io + CG_CARRY_BYTES, sizeof(CgSavedCarry));
        }
    } else if (carry_out) memset(carry_out, 0, CG_CARRY_BYTES);
    ctx->shard_state = 2;
    return 0;
}

extern "C" int cg_shard_end(cg_ctx *ctx, cg_result *out) {
    if (ctx->shard_state != 2 || stream_busy(ctx)) return CG_ERR_STATE;
    CG_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const cg_batch *in = ctx->shard_in;
    CgChainCarry *imported = &((CgScalars *)ctx->b_scal.p)->chain_import;
    int e;
    ctx->shard_state = 0;
    for (int k = ctx->shard_next; k < ctx->n_sl; k++) if ((e = slice_B(ctx, &ctx->sl[k], 1, 0))) { ctx->win_on = 0; return e; }
    /* the keep window the shard on the left left open stays active from this shard's first column: the carry area now holds the state
     * after this shard's own triggers, so paint from the imported copy */
    if (!ctx->win.first && ctx->have_saved && ctx->D.n_cols > 0) {
        CG_CHECK(cudaMemcpyAsync(imported, &((CgSavedCarry *)ctx->h_carry_io)->cc, sizeof(CgChainCarry), cudaMemcpyHostToDevice, st));
        k_paint_carry<<<1, 32, 0, st>>>(ctx->D, imported, ctx->win.lo_tid, ctx->win.lo_pos); ctx->launches++;
    }
    cudaEventRecord(ctx->ev[CG_T_D2H][0], ctx->s_d2h);
    for (int k = 0; k < ctx->n_sl; k++) {
        const CgSlice *s = &ctx->sl[k];
        if ((e = slice_B(ctx, s, 2, ctx->shard_timed && k == ctx->n_sl - 1))) { ctx->win_on = 0; return e; }   /* the last slice holds the rewrite */
        if (in && s->r1 > s->r0 && (e = enqueue_d2h(ctx, in, out, s->r0, s->r1, s->chunk))) { ctx->win_on = 0; return e; }
    }
    return finish_streamed(ctx, out, &ctx->win, ctx->shard_timed, NULL);
}

extern "C" int cg_process(cg_ctx *ctx, const cg_batch *in, cg_result *out) {
    if (stream_busy(ctx) || !in) return CG_ERR_STATE;
    return process_streamed(ctx, in, out, NULL, 0);
}

/* One call of a chain (include/crumble_gpu.h): the streamed driver above with a column window.  The column stage runs over all
 * tiles of the batch (columns outside the window come out inert, cg_window_class); the sparse passes of the slice holding the next
 * call's first column stop there, both carries are saved, and the passes finish the rest. */
extern "C" int cg_process_window(cg_ctx *ctx, const cg_batch *in, const cg_window *win, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    if (!win) return CG_ERR_BAD_ARG;
    if (ctx->params.region_tid >= 0) { snprintf(ctx->err, sizeof ctx->err, "chained calls and a -r region do not combine"); return CG_ERR_BAD_ARG; }
    if (!in) return CG_ERR_STATE;
    return process_streamed(ctx, in, out, win, 0);
}

extern "C" int cg_carry_export(cg_ctx *ctx, void *buf) {
    static_assert(sizeof(CgSavedCarry) <= CG_CARRY_BYTES, "carry blob");
    if (!ctx->have_saved) return CG_ERR_STATE;
    CG_CHECK(cudaSetDevice(ctx->device));
    memset(buf, 0, CG_CARRY_BYTES);
    CG_CHECK(cudaMemcpyAsync(buf, ctx->b_saved.p, sizeof(CgSavedCarry), cudaMemcpyDeviceToHost, ctx->stream));
    CG_CHECK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int cg_carry_import(cg_ctx *ctx, const void *buf) {
    CG_CHECK(cudaSetDevice(ctx->device));
    int e = ensure(ctx, &ctx->b_saved, sizeof(CgSavedCarry));
    if (e) return e;
    CG_CHECK(cudaMemcpyAsync(ctx->b_saved.p, buf, sizeof(CgSavedCarry), cudaMemcpyHostToDevice, ctx->stream));
    CG_CHECK(cudaStreamSynchronize(ctx->stream));
    ctx->have_saved = 1;
    return 0;
}
extern "C" int cg_carry_is_neutral(const cg_ctx *ctx, const void *buf, int32_t tid, int32_t lo_pos) {
    CgSavedCarry s; memcpy(&s, buf, sizeof s);
    /* keep-window chain: an open window matters only if it still covers the shard's first column; a trigger beyond
     * max_pos2 resets the state anyway (snp_score.c:1508-1511) and the two prefix-max keys only serve to find segment heads */
    const int open_window = s.cc.has && s.cc.wtid == tid && s.cc.w.min_pos != INT_MAX && s.cc.w.max_pos2 >= lo_pos;
    /* depth average: matters only when the over-depth test could fire at all in that call (run_prep) */
    if (ctx->depth_matters && s.ec.valid && s.ec.tid == tid) return -1;
    return open_window ? 0 : 1;
}

/* ---- a stream of records in GPU memory (include/crumble_gpu.h, DESIGN.md §3.6) ------------------------------------------------------
 * One call: held ++ in as one working batch (dev_stage), its cut planned on the device and read back at the call's one synchronisation
 * together with the checked sums; the held set for later calls is copied out of the pristine working arrays (k_retain) before the chain
 * runs; the chain is process_streamed's window machinery on the resident batch cut to its first m records; k_emit writes the final
 * prefix [e0, f) to qual_out. */
static void stream_close(cg_ctx *ctx) {
    ctx->st_open = 0; ctx->st_unplaced = 0; ctx->st_has_key = 0; ctx->st_kmax = 0;
    ctx->st_n = ctx->st_e0 = ctx->st_padded = ctx->st_cig = ctx->st_qual = ctx->st_seq = 0;
    memset(&ctx->st_win, 0, sizeof ctx->st_win); ctx->st_win.first = 1; ctx->st_win.lo_tid = -1;
}

static int stream_call(cg_ctx *ctx, const cg_dev_batch *in, int last, uint8_t *qual_out, cg_result *out, cg_stream_out *so) {
    cudaStream_t st = ctx->stream;
    const int64_t nh = ctx->st_n, e0 = ctx->st_e0, n = nh + in->n_reads;
    CgScalars *scal = (CgScalars *)ctx->b_scal.p;
    int e;
    if (!ctx->h_stream && cudaHostAlloc((void **)&ctx->h_stream, sizeof(CgScalars::CgStreamScal), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError(); ctx->h_stream = NULL; return CG_ERR_NOMEM;
    }
    uint8_t *keep = NULL;
    e = dev_stage(ctx, in, [&](int64_t *sums) -> int {
        int e2;
        if ((e2 = ensure(ctx, &ctx->b_keep, (size_t)n + 1)) || (e2 = ensure(ctx, &ctx->b_kidx, ((size_t)n + 1) * 4)) ||
            (e2 = ensure(ctx, &ctx->b_koff, ((size_t)n + 1) * 8)) || (e2 = ensure(ctx, &ctx->b_kcig, ((size_t)n + 1) * 4))) return e2;
        scal = (CgScalars *)ctx->b_scal.p;
        keep = (uint8_t *)ctx->b_keep.p;
        CgScalars::CgStreamScal *ss = &scal->stream;
        const CgDev *D = &ctx->D;
        k_stream_init<<<1, 1, 0, st>>>(&ss->red);
        k_prep_read<<<nblk(n, 256), 256, 0, st>>>(*D);
        k_stream_plan<<<nblk(n, 256), 256, 0, st>>>(*D, n, nh, e0, &ss->red);
        k_stream_cut<<<1, 1, 0, st>>>(*D, &ss->red, &ss->cut, n, e0, last, (const int64_t *)ctx->b_qsrc.p, sums + 2);
        k_stream_keep<<<nblk(n, 256), 256, 0, st>>>(*D, &ss->cut, keep, n);
        CG_CHECK(cudaGetLastError());
        LdKeep lk = { keep }; StExcl32of64 sk = { (int32_t *)ctx->b_kidx.p };
        LdKeepPad lp = { keep, D->l_qseq }; StExcl64 sp = { (int64_t *)ctx->b_koff.p };
        LdKeepCig lc = { keep, D->n_cigar }; StExcl32of64 sc = { (int32_t *)ctx->b_kcig.p };
        LdKeepLen ll = { keep, D->l_qseq }; LdKeepHalf lh = { keep, D->l_qseq }; StNone none;
        if ((e2 = run_scan<int64_t, OpSum>(ctx, lk, sk, n, (int64_t)0, &ss->held_n)) || (e2 = run_scan<int64_t, OpSum>(ctx, lp, sp, n, (int64_t)0, &ss->held_padded)) ||
            (e2 = run_scan<int64_t, OpSum>(ctx, lc, sc, n, (int64_t)0, &ss->held_cig)) || (e2 = run_scan<int64_t, OpSum>(ctx, ll, none, n, (int64_t)0, &ss->held_qual)) ||
            (e2 = run_scan<int64_t, OpSum>(ctx, lh, none, n, (int64_t)0, &ss->held_seq))) return e2;
        CG_CHECK(cudaMemcpyAsync(ctx->h_stream, ss, sizeof *ss, cudaMemcpyDeviceToHost, st));
        ctx->launches += 5;
        return 0;
    });
    if (e) return e;
    memset(so, 0, sizeof *so);
    memset(out->counters, 0, sizeof out->counters); out->n_events = 0; out->n_columns = 0;
    if (n == 0) return 0;                                      /* closing an empty stream */
    const CgScalars::CgStreamScal hs = *ctx->h_stream;
    const CgStreamCut c = hs.cut;
    /* the chunk's first pileup record must not sort before the stream's last one, nor after an unplaced record */
    if (hs.red.kmin <= hs.red.kmax && ((ctx->st_has_key && hs.red.kmin < ctx->st_kmax) || ctx->st_unplaced)) {
        snprintf(ctx->err, sizeof ctx->err, "cg_stream_device: this chunk's records sort before records of an earlier chunk");
        return CG_ERR_UNSORTED;
    }
    /* the held set, out of the pristine working arrays, before the chain runs */
    int64_t hn = hs.held_n, hpad = hs.held_padded, hcig = hs.held_cig;
    const CgDev *D = &ctx->D;
    if ((e = ensure(ctx, &ctx->b_htid, (size_t)hn * 4 + 4)) || (e = ensure(ctx, &ctx->b_hpos, (size_t)hn * 4 + 4)) || (e = ensure(ctx, &ctx->b_hflag, (size_t)hn * 2 + 2)) ||
        (e = ensure(ctx, &ctx->b_hmapq, (size_t)hn + 1)) || (e = ensure(ctx, &ctx->b_hlq, (size_t)hn * 4 + 4)) || (e = ensure(ctx, &ctx->b_hnc, (size_t)hn * 2 + 2)) ||
        (e = ensure(ctx, &ctx->b_hcig, (size_t)hcig * 4 + 4)) || (e = ensure(ctx, &ctx->b_hqual, (size_t)hpad + 8)) || (e = ensure(ctx, &ctx->b_hseq, (size_t)hpad / 2 + 8))) return e;
    if ((e = dev_ingest(ctx, in))) return e;
    if (hn > 0) {
        const CgRetain K = { D->tid, D->pos, D->l_qseq, D->flag, D->n_cigar, D->mapq, D->off, D->cigar_off, D->cigar, D->qual, D->seq,
                             (const int32_t *)ctx->b_kidx.p, (const int32_t *)ctx->b_kcig.p, (const int64_t *)ctx->b_koff.p,
                             (int32_t *)ctx->b_htid.p, (int32_t *)ctx->b_hpos.p, (int32_t *)ctx->b_hlq.p, (uint16_t *)ctx->b_hflag.p, (uint16_t *)ctx->b_hnc.p,
                             (uint8_t *)ctx->b_hmapq.p, (uint32_t *)ctx->b_hcig.p, (uint8_t *)ctx->b_hqual.p, (uint8_t *)ctx->b_hseq.p };
        k_retain<<<(unsigned)nblk(n * 32, IO_THREADS), IO_THREADS, 0, st>>>(K, (const uint8_t *)ctx->b_keep.p, n);
        CG_CHECK(cudaGetLastError());
    }
    int64_t n_emit = 0;
    if (!c.skip) {
        /* the chain over records [0, m) with this call's window; columns at/after X wait for later calls */
        cg_window w = ctx->st_win;
        w.hi_tid = c.hi_tid; w.hi_pos = c.hi_pos; w.next_lo_pos = c.S;
        ctx->D.n_reads = c.m;
        ctx->resident = 1; ctx->dump_columns = 0;
        if ((e = process_streamed(ctx, NULL, out, &w, 0))) return e;
        n_emit = c.f - e0;
        if ((e = dev_emit(ctx, e0, c.f, c.q_e0, qual_out))) return e;
        if (c.hi_tid >= 0) { ctx->st_win.first = 0; ctx->st_win.lo_tid = c.hi_tid; ctx->st_win.lo_pos = c.S; ctx->st_win.cnt_pos = c.hi_pos; }
        else { ctx->st_win.first = 1; ctx->st_win.lo_tid = -1; ctx->st_win.lo_pos = ctx->st_win.cnt_pos = 0; }
    } else ctx->resident = 0;                                  /* no chain ran: no events to fetch again */
    if (hs.red.kmin <= hs.red.kmax) { ctx->st_kmax = hs.red.kmax; ctx->st_has_key = 1; }
    ctx->st_unplaced |= hs.red.unplaced;
    ctx->st_n = hn; ctx->st_padded = hpad; ctx->st_cig = hcig; ctx->st_qual = hs.held_qual; ctx->st_seq = hs.held_seq;
    ctx->st_e0 = hn - (n - c.f);                               /* every record from f on is held: the ones before it are the emitted halo */
    so->n_records = n_emit; so->qual_len = n_emit ? c.q_f - c.q_e0 : 0;
    return 0;
}

extern "C" int cg_stream_device(cg_ctx *ctx, const cg_dev_batch *in, int last, uint8_t *qual_out, int64_t qual_cap, cg_result *out, cg_stream_out *so) {
    if (!ctx) return CG_ERR_BAD_ARG;
    cg_dev_batch none; memset(&none, 0, sizeof none);
    if (!in) in = &none;
    if (!out || !so) { snprintf(ctx->err, sizeof ctx->err, "cg_stream_device: no result or no cg_stream_out"); return CG_ERR_BAD_ARG; }
    if (out->columns) { snprintf(ctx->err, sizeof ctx->err, "cg_stream_device: the per-column dump is not available on streams (out->columns must be NULL)"); return CG_ERR_BAD_ARG; }
    if (ctx->params.region_tid >= 0) { snprintf(ctx->err, sizeof ctx->err, "streams and a -r region do not combine"); return CG_ERR_BAD_ARG; }
    if (!ctx->st_open) stream_close(ctx);                      /* the state a new stream starts from */
    if (qual_cap < ctx->st_qual + in->qual_len) {
        snprintf(ctx->err, sizeof ctx->err, "cg_stream_device: qual_cap %lld < %lld held + %lld new quality bytes", (long long)qual_cap, (long long)ctx->st_qual, (long long)in->qual_len);
        return CG_ERR_BAD_ARG;
    }
    CG_CHECK(cudaSetDevice(ctx->device));
    int e;
    if ((e = dev_check(ctx, in, qual_out, qual_cap, out, ctx->st_n + in->n_reads, ctx->st_cig + in->n_cigar_total, ctx->st_qual + in->qual_len))) return e;
    ctx->st_open = 1;
    if (in->n_reads == 0 && !last) {                           /* nothing new: nothing can turn final */
        memset(so, 0, sizeof *so); memset(out->counters, 0, sizeof out->counters); out->n_events = 0; out->n_columns = 0;
        so->held_records = ctx->st_n; so->held_qual_len = ctx->st_qual;
        return 0;
    }
    ctx->win_on = 0;
    if ((e = stream_call(ctx, in, last, qual_out, out, so))) { stream_close(ctx); ctx->resident = 0; ctx->win_on = 0; cudaGetLastError(); return e; }
    if (last) stream_close(ctx);
    so->held_records = ctx->st_n; so->held_qual_len = ctx->st_qual;
    return 0;
}
