/*
 * cg_cells.h — the pileup CELL: what one read contributes to one reference column, as 16 bits.
 *
 * The column stage is split in two (DESIGN.md §3.1):
 *   k_cells   (read-major)    every pileup read is decoded ONCE into a row of cells, one per reference column it covers
 *                             (deletion and ref-skip columns included), written to a cell matrix in global memory in groups
 *                             of 8 cells = 16 bytes.  Row j starts at group cpos8[j]; its first group is the 8-ALIGNED group of
 *                             dense columns that holds the read's first column, so that group g of any row holds columns
 *                             [8g', 8g'+8) of the dense column axis: a 32-column tile of k_column is four whole groups of every row;
 *   k_column  (column-major)  a warp stages the cells of its tile's candidate reads with 16-byte async copies and every lane walks
 *                             its own column down the rows.
 * What a cell carries is everything the per-column loops of the reference read from (read, column):
 * calculate_consensus_pileup's base and effective quality (snp_score.c:588-686) and the flags of the read-set heuristics
 * (1662-1669, 1701-1713).  Functions here are __host__ __device__: tests/emu/ runs the same code on the CPU.
 */
#ifndef CG_CELLS_H
#define CG_CELLS_H

#include "cg_pipeline.h"

#define CELL_VALID   0x8000u
#define CELL_BASE_SH 12         /* bits 14..12: base 0..4 = ACGT*, 5 = N, 6 = ref-skip, 7 = no contribution (l_qseq == 0, or mode B off) */
#define CELL_BASE_M  0x7000u
#define CELL_E_SH    5          /* bits 11..5: effective quality (1..100) == byte offset / 32 of its row in the shared-memory table */
#define CELL_E_M     0x0fe0u
#define CELL_INS     0x0010u    /* an insertion follows this column (indel > 0) in a read that neither starts nor ends here */
#define CELL_CLIP    0x0008u    /* soft-clipped (or inserted) bases hang off this end of the read (snp_score.c:1701-1703) */
#define CELL_INDEL   0x0004u    /* indel != 0 || is_del (1664) */
#define CELL_MID     0x0002u    /* neither the read's first nor its last column (1705) */
#define CELL_LOWMQ   0x0001u    /* mapq <= -m (1663) */

/* one record per pileup read for the cell matrix (16 bytes, read by k_cells and by k_column's staging) */
typedef struct CgCellRec {
    uint32_t cpos8;           /* first 8-cell group of the row */
    int32_t  col0;            /* dense column of the first reference base */
    int32_t  span;            /* reference span */
    uint32_t ngrp;            /* groups of the row: ceil(((col0 & 7) + span) / 8) */
} CgCellRec;

CG_HD uint32_t cg_cell_ngroups(int col0, int span) { return (uint32_t)(((col0 & 7) + span + 7) >> 3); }

/* the cell of compact read j at offset d of its reference span (0 when d is outside): any CIGAR */
CG_HD uint32_t cg_cell_general(const CgDev *D, const CgRead *q, int d, int doB) {
    if ((unsigned)d >= (unsigned)q->span) return 0;
    CgCell cell;
    if (!cg_plp_resolve(D->cigar + q->cig_off, q->n_cigar, d, q->span, &cell)) return 0;
    uint32_t f = CELL_VALID | ((int)q->mapq <= D->P.min_mqual ? CELL_LOWMQ : 0u), base = 7, e = 0;
    if (cell.indel | cell.is_del) f |= CELL_INDEL;
    if (cell.is_refskip) base = 6;
    else {
        if ((cell.is_head && cell.qpos > 0) || (cell.is_tail && cell.qpos + 1 < q->l_qseq)) f |= CELL_CLIP;
        if (!cell.is_tail && !cell.is_head) { f |= CELL_MID; if (cell.indel > 0) f |= CELL_INS; }
        if (q->l_qseq && doB) {
            const int64_t off = CG_OFF(q);
            e = D->T->effB[((int)q->mapq << 8) | D->qual[off + cell.qpos]];
            base = cell.is_del ? 4 : (uint32_t)cg_nt16_to_base((D->seq[(off >> 1) + (cell.qpos >> 1)] >> ((~cell.qpos & 1) << 2)) & 0xf);
        }
    }
    return f | (e << CELL_E_SH) | (base << CELL_BASE_SH);
}

/* eight nt16 codes (one per nibble, lowest nibble first) -> eight base codes (A0 C1 G2 T3, anything else 5) */
CG_HD uint32_t cg_bases8(uint32_t X) {
    const uint32_t M = 0x11111111u;
    const uint32_t p0 = X & M, p1 = (X >> 1) & M, p2 = (X >> 2) & M, p3 = (X >> 3) & M;
    const uint32_t t = (p0 + p1 + p2 + p3) ^ M;                       /* nibble == 0 iff exactly one bit set */
    const uint32_t one = ((t | (t >> 1) | (t >> 2)) & M) ^ M;
    const uint32_t m = one * 15u;
    return ((p1 + p2 * 2u + p3 * 3u) & m) | (0x55555555u & ~m);
}

/* the eight cells of group k of a SIMPLE read (single M/=/X op, l_qseq == span: query offset == column offset), as four 32-bit words
 * of two cells each.  d_first = 8k - (col0 & 7) is the offset inside the read of the group's first cell (negative in the first
 * group of a read that does not start on a group boundary).  Two aligned 64-bit quality loads and two 32-bit sequence loads are
 * funnel-shifted into place (both buffers are padded, see CG_FRONT_PAD), the nt16 codes are mapped to bases in one
 * SIMD-within-register pass, quality x mapq goes through the host-built cell table (effective quality, a pure function of both,
 * snp_score.c:632-642, with the valid and low-mapq bits folded in).  Only the first and last group of a read are ragged. */
CG_HD void cg_cells8_simple(const CgDev *D, const CgRead *q, int d_first, int doB, uint32_t out[4]) {
    const int span = q->span;
    const int ka = -d_first, kb = span - d_first;                        /* cells k in [ka, kb) lie on the read */
    out[0] = out[1] = out[2] = out[3] = 0;
    if (ka >= 8 || kb <= 0) return;
    const int mapq = q->mapq;
    const int64_t A = CG_OFF(q) + d_first;                              /* byte address of the first quality */
    const int64_t Bb = (A >> 1) & ~(int64_t)3;
    const uint32_t *qa = (const uint32_t *)(D->qual + (A & ~(int64_t)7));
    const uint32_t *sa = (const uint32_t *)(D->seq + Bb);
#ifdef __CUDA_ARCH__
    const uint2 w0 = __ldg((const uint2 *)qa), w1 = __ldg((const uint2 *)qa + 1);
    uint32_t v0 = __ldg(sa), v1 = __ldg(sa + 1);
    const uint32_t w0x = w0.x, w0y = w0.y, w1x = w1.x, w1y = w1.y;
#else
    const uint32_t w0x = qa[0], w0y = qa[1], w1x = qa[2], w1y = qa[3];
    uint32_t v0 = sa[0], v1 = sa[1];
#endif
    const int s = (int)(A & 7);
    const uint32_t Wa = (s & 4) ? w0y : w0x, Wb = (s & 4) ? w1x : w0y, Wc = (s & 4) ? w1y : w1x;
    const uint32_t qlo = cg_funnel_r(Wa, Wb, (s & 3) * 8), qhi = cg_funnel_r(Wb, Wc, (s & 3) * 8);
    uint32_t c[4];
    if (doB) {
        const int m0 = (int)(A - (Bb << 1));                            /* first nibble inside the 64-bit word, 0..7 */
        v0 = ((v0 & 0x0f0f0f0fu) << 4) | ((v0 >> 4) & 0x0f0f0f0fu);     /* high nibble first -> little-endian nibbles */
        v1 = ((v1 & 0x0f0f0f0fu) << 4) | ((v1 >> 4) & 0x0f0f0f0fu);
        const uint32_t Bs = cg_bases8(cg_funnel_r(v0, v1, 4 * m0));      /* base of cell k in nibble k */
        const uint16_t *er = D->T->cellB + (mapq << 8);
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
        for (int w = 0; w < 4; w++) {
            const uint32_t qq = w < 2 ? qlo >> (16 * w) : qhi >> (16 * (w - 2));
#ifdef __CUDA_ARCH__
            const uint32_t e0 = __ldg(er + (qq & 0xff)), e1 = __ldg(er + ((qq >> 8) & 0xff));
#else
            const uint32_t e0 = er[qq & 0xff], e1 = er[(qq >> 8) & 0xff];
#endif
            /* the two base nibbles of this word to bits 12..14 and 28..30 */
            const uint32_t bb = (((Bs >> (8 * w)) & 0xffu) * 0x01001000u) & 0x70007000u;
            c[w] = e0 | (e1 << 16) | bb;
        }
    } else {
        const uint32_t rowf = CELL_VALID | (7u << CELL_BASE_SH) | (mapq <= D->P.min_mqual ? CELL_LOWMQ : 0u);   /* no contribution */
        c[0] = c[1] = c[2] = c[3] = rowf | (rowf << 16);
    }
    const uint32_t MIDW = CELL_MID | (CELL_MID << 16);
    if (ka < 0 && kb > 8) {                                              /* interior group: all eight cells valid and "mid" */
        out[0] = c[0] | MIDW; out[1] = c[1] | MIDW; out[2] = c[2] | MIDW; out[3] = c[3] | MIDW;
        return;
    }
    /* ragged ends: valid cells [ka, kb), of which the read's first and last column are not "mid" */
    const int va = ka < 0 ? 0 : ka, vb = kb > 8 ? 8 : kb;
    const int ma = ka + 1 < 0 ? 0 : ka + 1, mb = kb - 1 > 8 ? 8 : kb - 1;
    const uint32_t v8 = ((1u << vb) - 1u) & ~((1u << va) - 1u);
    const uint32_t m8 = mb > ma ? ((1u << mb) - 1u) & ~((1u << ma) - 1u) : 0u;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (int w = 0; w < 4; w++) {
        const uint32_t tv = (v8 >> (2 * w)) & 3u, tm = (m8 >> (2 * w)) & 3u;
        const uint32_t vm = ((tv & 1u) * 0xffffu) | ((tv >> 1) * 0xffff0000u);
        const uint32_t mm = ((tm & 1u) * (uint32_t)CELL_MID) | ((tm >> 1) * ((uint32_t)CELL_MID << 16));
        out[w] = (c[w] & vm) | mm;
    }
}

/* group k of any read */
CG_HD void cg_cells8(const CgDev *D, const CgRead *q, int k, int doB, uint32_t out[4]) {
    const int d_first = 8 * k - (q->col0 & 7);
    if (q->rf & CG_RF_SIMPLE) { cg_cells8_simple(D, q, d_first, doB, out); return; }
    uint32_t c[8];
    for (int i = 0; i < 8; i++) c[i] = cg_cell_general(D, q, d_first + i, doB);
    out[0] = c[0] | c[1] << 16; out[1] = c[2] | c[3] << 16; out[2] = c[4] | c[5] << 16; out[3] = c[6] | c[7] << 16;
}

#endif /* CG_CELLS_H */
