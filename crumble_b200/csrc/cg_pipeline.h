/*
 * cg_pipeline.h — the work-item bodies of the device pipeline.
 *
 * One function per kernel stage, each processing ONE work item (a read, a reference
 * column, a flagged column, a trigger) with no warp collectives, so the same source
 * runs as the body of the sm_100a kernels in cg_device.cu and, for CPU-side debugging of
 * the decomposition, inside tests/emu/ (never shipped).  Stage order (DESIGN.md §pipeline):
 *
 *   prep_read  -> [scan: pileup compaction, dense column coordinates] -> finish_read
 *   tile_index -> column (pileup + consensus + column heuristics)
 *   [compaction of flagged columns] -> flagged (indel spectrum + STR extents)
 *   [depth scan] -> deep ; chain (sequential over trigger columns) -> paint
 *   rewrite (+ P-block) ; events
 */
#ifndef CG_PIPELINE_H
#define CG_PIPELINE_H

#include <string.h>
#include "cg_core.h"
#include "../../include/crumble_gpu.h"

#define CG_RF_PILEUP  1
#define CG_RF_SIMPLE  2       /* single M/=/X op with l_qseq == span (0 < l_qseq < 65535): qpos = column offset, never clipped */

typedef struct CgRead {       /* 32 bytes, one per pileup read (compacted, input order) */
    /* hot half: everything the column kernel needs for a single-M read */
    uint32_t off8;            /* qual byte offset / 8 (seq at off/2) */
    int32_t  col0;            /* dense column of the first reference base */
    int32_t  span;            /* reference span */
    uint32_t pk;              /* min(l_qseq,0xffff) | mapq << 16 | rf << 24 */
    /* cold half */
    int32_t  pos;             /* reference position */
    int32_t  cig_off;
    int32_t  l_qseq;
    uint16_t n_cigar;
    uint8_t  mapq;
    uint8_t  rf;
} __attribute__((aligned(16))) CgRead;    /* two 16-byte loads / stores per record */
#define CG_OFF(q) ((int64_t)(q)->off8 << 3)

typedef struct CgStrItem { int32_t k, j, rpos, is_indel; } CgStrItem;   /* flagged entry, pileup read, 1-based query position (qpos + 1), trigger type */
typedef struct CgIsland { int32_t col_start, tid, pos_start, pad; } CgIsland;
struct CgCellRec;             /* cg_cells.h */

typedef struct CgDev {
    /* sizes */
    int64_t n_reads;          /* records in the batch */
    int32_t n_pile;           /* records entering the pileup */
    int32_t n_cols;           /* covered reference columns (dense) */
    int32_t n_tiles;          /* ceil(n_cols/32) */
    int32_t n_islands;
    int32_t n_flagged;
    int32_t n_trig_cap;
    int64_t n_cigar_total;    /* entries in cigar[] */
    /* batch (SoA) */
    const int32_t *tid, *pos; const uint16_t *flag; const uint8_t *mapq; const int32_t *l_qseq;
    const uint16_t *n_cigar; const int64_t *off; const int32_t *cigar_off;
    const uint32_t *cigar; const uint8_t *seq; const uint8_t *qual;
    uint8_t *qual_out;
    /* per record */
    int32_t *jmap;            /* record -> compact pileup index (exclusive scan of the pileup flag) */
    int32_t *rspan;           /* reference span, 0 when not in the pileup */
    /* per pileup read */
    CgRead  *rd;
    int64_t *ks, *ke;         /* (tid<<32|pos) of start / end; ke becomes its inclusive prefix max */
    int64_t *gap;             /* becomes the inclusive prefix sum of zero-coverage gaps */
    int32_t *pmaxcol;         /* dense inclusive prefix max of end columns */
    int32_t *orig;            /* compact index -> record index */
    uint8_t *r_bf;            /* read overlaps a trigger column: back-fill path in the rewrite */
    int32_t *glist, *n_glist; /* pileup reads with a non-trivial CIGAR (any order), and how many */
    struct CgCellRec *crec;   /* cell matrix: row record per pileup read (cg_cells.h) */
    uint16_t *cells;          /* cell matrix: 16-bit pileup cells in groups of 8 */
    int64_t  K0;              /* key of the first pileup read */
    /* tiles of 32 dense columns */
    int32_t *tile_lo;         /* first pileup read whose prefix-max end column exceeds the tile start */
    int32_t *tile_start;      /* first pileup read starting at/after the tile start; [n_tiles] = n_pile */
    CgIsland *isl;
    /* per dense column */
    uint8_t  *cb; uint16_t *ev; uint32_t *depth;
    cg_column *coldump;       /* optional */
    int64_t *dsum; int32_t *csum;   /* depth scan: inclusive prefix sums of depth / counted flag */
    /* sparse */
    int32_t *fcol;            /* flagged dense columns, ascending */
    CgTrig  *trig;            /* one per flagged column (hasI=hasS=0 when it does not trigger) */
    struct CgStrItem *sitem;  /* (trigger column, read) STR searches of the slice, any order */
    int32_t *n_sitem;         /* how many */
    int64_t sitem_cap;
    unsigned long long *item_bound;   /* running upper bound of the searches the columns processed so far will ask for */
    CgWin   *twin;            /* window state after each flagged column */
    /* scalars on the device */
    unsigned long long *counters;   /* CG_N_COUNTERS */
    int32_t *maxdepth; int32_t *err;
    int32_t *beyond;          /* set when a counted column exists at/after the -r region end (the reference counts one, then breaks) */
    const CgTables *T;
    const cg_bed_reg *bed;    /* -R regions as bed.c:20-40 leaves them (sorted, collapsed) */
    const int64_t *bed_pm;    /* inclusive prefix max of (tid << 32 | end) over bed[] */
    CgDevParams P;
    int32_t want_dump;
    int32_t cons_only;        /* debug */
} CgDev;

CG_HD int64_t cg_key(int32_t tid, int32_t pos) { return ((int64_t)tid << 32) | (uint32_t)pos; }

/* ---- stage: prep_read (one per record) ------------------------------------------------
 * rspan[r] = cg_pileup_span: pileup eligibility as bam_plp_push + pileup_callback (SURVEY §9.2) */
CG_HD void cg_prep_read(const CgDev *D, int64_t r) {
    int n = D->n_cigar[r];
    if (D->cigar_off[r] < 0 || (int64_t)D->cigar_off[r] + n > D->n_cigar_total) { *D->err = CG_ERR_BAD_ARG; D->rspan[r] = 0; return; }   /* a layout that lies about its CIGARs */
    D->rspan[r] = cg_pileup_span(D->tid[r], D->flag[r], D->cigar + D->cigar_off[r], n);
}

/* after the pileup-flag scan: fill compact keys */
CG_HD void cg_prep_keys(const CgDev *D, int64_t r) {
    int span = D->rspan[r];
    if (!span) return;
    int j = D->jmap[r];
    D->orig[j] = (int32_t)r;
    D->ks[j] = cg_key(D->tid[r], D->pos[r]);
    D->ke[j] = cg_key(D->tid[r], D->pos[r] + span);
}

/* gap before pileup read j (after ke[] has become its inclusive prefix max) */
CG_HD int64_t cg_gap_of(const CgDev *D, int j) {
    if (j == 0) return 0;
    int64_t g = D->ks[j] - D->ke[j - 1];
    return g > 0 ? g : 0;
}

/* after both scans: build the read record (one per pileup read) */
CG_HD void cg_finish_read(const CgDev *D, int j, int64_t K0) {
    int64_t r = D->orig[j];
    CgRead q;
    int span = D->rspan[r];
    q.off8 = (uint32_t)(D->off[r] >> 3);
    q.col0 = (int32_t)(D->ks[j] - K0 - D->gap[j]);
    q.span = span;
    q.pos = D->pos[r];
    q.cig_off = D->cigar_off[r];
    q.l_qseq = D->l_qseq[r];
    q.n_cigar = D->n_cigar[r];
    q.mapq = D->mapq[r];
    uint8_t rf = CG_RF_PILEUP;
    if (q.n_cigar == 1 && cg_is_mop(cg_cig_op(D->cigar[q.cig_off])) && q.l_qseq == span && span < 65535) rf |= CG_RF_SIMPLE;
    q.rf = rf;
    q.pk = (uint32_t)(q.l_qseq > 0xffff ? 0xffff : q.l_qseq) | ((uint32_t)q.mapq << 16) | ((uint32_t)rf << 24);
    D->rd[j] = q;
    D->pmaxcol[j] = (int32_t)(D->ke[j] - K0 - D->gap[j]);
    D->r_bf[j] = 0;
    if (j > 0 && D->ks[j] < D->ks[j - 1]) *D->err = CG_ERR_UNSORTED;
}

/* ---- stage: tile_index (one per pileup read): each read "owns" the tile boundaries that
 * fall between its predecessor's coordinate and its own ------------------------------- */
CG_HD void cg_tile_index(const CgDev *D, int j) {
    int c_prev = j ? D->rd[j - 1].col0 : -1;
    int c = D->rd[j].col0;
    for (int t = (c_prev >> 5) + 1; t <= (c >> 5); t++) D->tile_start[t] = j;     /* first read with col0 >= 32t */
    if (j == 0) D->tile_start[0] = 0;
    int p_prev = j ? D->pmaxcol[j - 1] : 0;
    int p = D->pmaxcol[j];
    for (int t = (p_prev + 31) >> 5; t < ((p + 31) >> 5); t++) D->tile_lo[t] = j;  /* first read with pmax > 32t */
}

CG_HD int cg_island_of(const CgDev *D, int c) {
    int lo = 0, hi = D->n_islands - 1;
    while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (D->isl[mid].col_start <= c) lo = mid; else hi = mid - 1; }
    return lo;
}

/* first dense column whose (tid, pos) is at or after the given one; n_cols when there is none */
CG_HD int cg_find_col(const CgDev *D, int tid, int pos) {
    const int64_t K = cg_key(tid, pos);
    int lo = 0, hi = D->n_islands;                         /* first island starting after K */
    while (lo < hi) { int mid = (lo + hi) >> 1; if (cg_key(D->isl[mid].tid, D->isl[mid].pos_start) <= K) lo = mid + 1; else hi = mid; }
    if (lo == 0) return 0;
    const CgIsland I = D->isl[lo - 1];
    const int next = lo < D->n_islands ? D->isl[lo].col_start : D->n_cols;
    if (I.tid != tid) return next;
    const int64_t c = (int64_t)I.col_start + ((int64_t)pos - I.pos_start);
    return c < next ? (int)c : next;
}

/* Chained calls (cg_process_window): 0 = column owned by this call; 1 = replayed (already counted by the previous call,
 * processed again because the cross-column state and the reads still open need it); 2 = not this call's business
 * (before the window: done earlier; at/after its end: reads that cover it have not all arrived yet). */
CG_HD int cg_window_class(const CgDevParams *P, int tid, int pos) {
    if (!P->win_on) return 0;
    if (tid == P->win_lo_tid) { if (pos < P->win_lo_pos) return 2; if (pos < P->win_cnt_pos) return 1; }
    if (P->win_hi_tid >= 0 && (tid > P->win_hi_tid || (tid == P->win_hi_tid && pos >= P->win_hi_pos))) return 2;
    return 0;
}

/* resolve a pileup cell for compact read j at dense column c; false if not covering */
CG_HD bool cg_cell(const CgDev *D, const CgRead *q, int c, CgCell *cell) {
    unsigned d = (unsigned)(c - q->col0);
    if (d >= (unsigned)q->span) return false;
    if (q->rf & CG_RF_SIMPLE) {
        cell->qpos = (int)d; cell->indel = 0; cell->is_del = 0; cell->is_refskip = 0;
        cell->is_head = d == 0; cell->is_tail = (int)d == q->span - 1;
        return true;
    }
    return cg_plp_resolve(D->cigar + q->cig_off, q->n_cigar, (int)d, q->span, cell);
}

CG_HD int cg_seq_nib(const CgDev *D, const CgRead *q, int x) {
    return (D->seq[(CG_OFF(q) >> 1) + (x >> 1)] >> ((~x & 1) << 2)) & 0xf;
}

/* -R keep.bed (snp_score.c:1443-1463): bed_idx only moves forward, past regions with tid < tid or (same tid, end < pos);
 * both conditions are monotone along the sorted column order, so the index reached at a column is the FIRST region with
 * (tid, end) >= (tid, pos) -- found by binary search on the prefix max of the (tid, end) keys -- whatever came before. */
CG_HD int cg_bed_hit(const CgDev *D, int tid, int pos) {
    const int64_t K = ((int64_t)tid << 32) | (uint32_t)pos;
    int lo = 0, hi = D->P.nbed;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (D->bed_pm[mid] < K) lo = mid + 1; else hi = mid; }
    if (lo >= D->P.nbed) return 0;
    const cg_bed_reg b = D->bed[lo];
    return b.tid == tid && b.start <= pos && b.end > pos;
}

/* ---- stage: column (one per dense column) --------------------------------------------
 * transcode's column loop up to the point where cross-column state is needed
 * (snp_score.c:1466-1472, 1490-1500, 1520-1649, 1658-1669, 1694-1713, 1764-1773).
 * Returns a bit mask of CG_CNT_* counters to increment.                                  */
typedef struct CgColOut { uint32_t cnt; int32_t n_plp; int32_t items; /* upper bound of the (column, read) STR searches this column will ask for */ } CgColOut;

template <int MODE_B>
CG_HD void cg_column_cons(const CgDev *D, int c, int lo, int hi, CgCons *out) {
    const CgTables *T = D->T;
    CgConsAcc a; cg_cons_init(&a);
    for (int j = lo; j < hi; j++) {
        const CgRead q = D->rd[j];
        CgCell cell;
        if (!cg_cell(D, &q, c, &cell)) continue;
        if (cell.is_refskip || !q.l_qseq) continue;                       /* 589-595 */
        int nib = cg_seq_nib(D, &q, cell.qpos);
        int base = cell.is_del ? 4 : cg_nt16_to_base(nib);                /* 603-609 */
        uint8_t qv = cg_cap_qual(D->qual[CG_OFF(&q) + cell.qpos], &D->P, T);   /* pileup copy is capped (1325-1332) */
        int eq = MODE_B ? T->effB[((int)q.mapq << 8) | qv] : T->effA[qv];
        cg_cons_add(T, &a, base, eq);
    }
    cg_cons_finalize(T, &a, out);
}

typedef struct CgColStats { int n_plp, n_skip, low_mq, had_indel, indel_cnt, clipped, n_overlap, ins_seen; int cp; /* call_preserve (611-623) */ } CgColStats;

/* everything after the per-read loop: consensus finalisation and the column decisions */
/* cB_ready: the mode-B consensus when the caller has already finalised it (the tuned kernel, cg_column_lean.h); else acc holds the sums */
CG_HD CgColOut cg_column_finish(const CgDev *D, int c, int lo, int hi, const CgColStats *st, CgConsAcc *acc, const CgCons *cB_ready = NULL) {
    const CgDevParams *P = &D->P;
    const CgTables *T = D->T;
    CgColOut o; o.cnt = 0; o.n_plp = 0; o.items = 0;
    const int n_plp = st->n_plp, n_skip = st->n_skip, low_mq = st->low_mq, had_indel = st->had_indel;
    const int clipped = st->clipped, n_overlap = st->n_overlap, ins_seen = st->ins_seen;
    const int doB = P->min_qual_B != 0;
    o.n_plp = n_plp;
    uint16_t ev = 0; uint8_t cb = CG_CB_UNPROC;
    D->depth[c] = (uint32_t)n_plp;
    if (n_plp == 0 || n_skip == n_plp) {                                  /* 1466-1472 (n_plp==0 cannot happen on a dense column) */
        D->cb[c] = (uint8_t)(cb | (D->cb[c] & CG_CB_ACTIVE)); D->ev[c] = 0;
        if (D->want_dump) { cg_column z = {0}; z.tid = -1; D->coldump[c] = z; }
        return o;
    }
    int tid = 0, pos = 0;
    const int need_pos = (P->region_tid >= 0) || D->want_dump || P->nbed || P->win_on;
    if (need_pos) {
        int is = cg_island_of(D, c);
        tid = D->isl[is].tid; pos = D->isl[is].pos_start + (c - D->isl[is].col_start);
    }
    const int wclass = cg_window_class(P, tid, pos);
    if (wclass == 2) {                                                    /* outside this call's column window */
        D->cb[c] = (uint8_t)(cb | (D->cb[c] & CG_CB_ACTIVE)); D->ev[c] = 0;
        if (D->want_dump) { cg_column z = {0}; z.tid = -1; D->coldump[c] = z; }
        return o;
    }
    /* region end acts as a hard stop (the reference breaks out of the loop, 1516-1517) */
    if (P->region_tid >= 0 && pos >= P->region_end) { *D->beyond = 1; D->cb[c] = (uint8_t)(cb | (D->cb[c] & CG_CB_ACTIVE)); D->ev[c] = 0; if (D->want_dump) { cg_column z = {0}; z.tid = -1; D->coldump[c] = z; } return o; }
    ev |= CG_EV_COUNTED;
    o.cnt |= 1u << CG_CNT_COLUMNS;                                        /* 1476 */
    CgCons cB; cB.call = 5; cB.het_call = 0; cB.het_phred = 0; cB.phred = 0; cB.depth = 0; cB.discrep = 0;
    CgCons cA = cB;
    uint32_t dflags = 0;
    if (n_plp > CG_MAX_DEPTH) {                                           /* 1493-1500 */
        ev |= CG_EV_VDEEP;
    } else if (P->region_tid >= 0 && pos < P->region_beg) {               /* 1514-1515 */
        /* counted, not processed */
    } else {
        ev |= CG_EV_PROCESSED;
        dflags |= 8;
        if (doB) { if (cB_ready) cB = *cB_ready; else cg_cons_finalize(T, acc, &cB); }
        if (P->min_qual_A != 0) cg_column_cons<0>(D, c, lo, hi, &cA);
        int hA = 0, sA = 0, hB = 0, sB = 0;
        const CgCons *cc = doB ? &cB : &cA;                                /* B's calls overwrite A's (1534-1543) */
        int code = (doB || P->min_qual_A) ? cg_call_code(cc) : 0;          /* call1=call2=0 matches nothing */
        if (P->min_qual_A) {                                               /* 1576-1583 */
            hA = cA.het_phred > 0 ? cA.het_call : cA.call * 5 + cA.call;
            sA = cA.het_phred > 0 ? cA.het_phred : cA.phred;
        }
        if (doB) {                                                         /* 1584-1591 */
            hB = cB.het_phred > 0 ? cB.het_call : cB.call * 5 + cB.call;
            sB = cB.het_phred > 0 ? cB.het_phred : cB.phred;
        }
        int preserve = 0, perfect = 1;
        if (P->nbed && cg_bed_hit(D, tid, pos)) preserve = 2;               /* 1443-1463: *really* preserve; disallow P-block */
        if (P->min_qual_A && doB && hA != hB) { o.cnt |= 1u << CG_CNT_DIFF; preserve |= 1; }    /* 1593,1624 */
        if (P->min_qual_A) {                                               /* 1594-1609 */
            if (cA.het_phred > 0) { o.cnt |= 1u << CG_CNT_HET_A; if (sA < P->min_qual_A) o.cnt |= 1u << CG_CNT_HET_QUAL_A; }
            else { o.cnt |= 1u << CG_CNT_HOM_A; if (sA < P->min_qual_A) o.cnt |= 1u << CG_CNT_HOM_QUAL_A; }
            if (cA.discrep >= P->min_discrep_A) { o.cnt |= 1u << CG_CNT_DISCREP_A; preserve |= 1; }
            if (sA < P->min_qual_A) preserve |= 1;
            if (st->cp != (1 << cA.call)) perfect = 0;                      /* 1606-1608: evaluated whatever preserve is */
        }
        if (doB) {                                                         /* 1610-1622 */
            if (cB.het_phred > 0) { o.cnt |= 1u << CG_CNT_HET_B; if (sB < P->min_qual_B) o.cnt |= 1u << CG_CNT_HET_QUAL_B; }
            else { o.cnt |= 1u << CG_CNT_HOM_B; if (sB < P->min_qual_B) o.cnt |= 1u << CG_CNT_HOM_QUAL_B; }
            if (cB.discrep >= P->min_discrep_B) { o.cnt |= 1u << CG_CNT_DISCREP_B; preserve |= 1; }
            if (sB < P->min_qual_B) preserve |= 1;
        }
        if (P->any_preserve_qual || P->perfect_col) {                      /* 1630-1649 */
            const int m5 = st->cp & 31;
            const int b2c = (m5 && !(m5 & (m5 - 1))) ? (m5 == 1 ? 0 : m5 == 2 ? 1 : m5 == 4 ? 2 : m5 == 8 ? 3 : 4) : 99;   /* bit2call, 1384-1417 */
            if (P->min_qual_A && !preserve && ((cA.het_phred <= 0 && b2c != cA.call) || (st->cp >> 8))) perfect = 0;
            if (doB && !preserve && ((cB.het_phred <= 0 && b2c != cB.call) || (st->cp >> 8))) perfect = 0;
            if (P->perfect_col && !perfect) preserve = 1;                   /* assignment: a -R hit loses its "2" here, as in the reference */
        }
        if (preserve > 1) ev |= CG_EV_BED;
        if (!perfect) ev |= CG_EV_IMPERFECT;
        int keep = low_mq > P->low_mqual_perc * (n_plp + .01);             /* 1668 */
        if (keep) o.cnt |= 1u << CG_CNT_LOW_MQUAL_PERC;
        if ((clipped - 1.0) >= P->clip_perc * n_overlap) {                 /* 1764-1773 */
            ev |= CG_EV_CLIP; keep = 1; o.cnt |= 1u << CG_CNT_CLIP_PERC;
        }
        if (had_indel) { o.cnt |= 1u << CG_CNT_INDEL; ev |= CG_EV_HADINDEL; }          /* 1761 */
        int lowscore = (P->min_qual_A && sA < P->min_indel_A) || (doB && sB < P->min_indel_B);   /* 1719-1720 */
        if (lowscore) ev |= CG_EV_LOWSCORE;
        int strall = P->str_snp && preserve;
        if (strall) ev |= CG_EV_STRALL;
        if (lowscore && (had_indel || strall)) {
            /* refskip-only "indels" do not trigger (1696-1697): the flagged pass decides per read */
            ev |= CG_EV_FLAGGED;
        }
        if (ins_seen) ev |= CG_EV_FLAGGED;                                 /* indel-size spectrum tests (1777-1819) */
        /* every read that triggers at this column gets one mask_LC_regions search (1718-1739): all of them when str_snp && preserve,
         * else the reads with an indel here; none below the -Y indel fraction (1732).  Sizes the item list of the flagged stage. */
        if (lowscore && (had_indel || strall) && st->indel_cnt >= n_plp * P->indel_fract) o.items = strall ? n_plp : st->indel_cnt;
        cb = (uint8_t)code;
        if (preserve) cb |= CG_CB_PRESERVE;
        if (keep) cb |= CG_CB_KEEP;
        if (preserve) dflags |= 1;
        if (keep) dflags |= 2;
    }
    if (wclass == 1) { ev |= CG_EV_REPLAY; o.cnt = 0; }                   /* counted (and dumped) by the previous call */
    D->cb[c] = (uint8_t)(cb | (D->cb[c] & CG_CB_ACTIVE)); D->ev[c] = ev;
    if (D->want_dump && wclass == 1) { cg_column z = {0}; z.tid = -1; D->coldump[c] = z; }
    else if (D->want_dump) {
        cg_column z;
        const CgCons *cc = doB ? &cB : &cA;
        z.tid = tid; z.pos = pos; z.n_plp = n_plp;
        z.call = cc->call; z.het_call = cc->het_call; z.het_phred = cc->het_phred; z.phred = cc->phred;
        z.discrep = cc->discrep; z.flags = dflags;
        D->coldump[c] = z;
    }
    return o;
}

CG_HD CgColOut cg_column_body(const CgDev *D, int c) {
    const CgDevParams *P = &D->P;
    const CgTables *T = D->T;
    CgColOut o; o.cnt = 0; o.n_plp = 0; o.items = 0;
    const int t = c >> 5;
    const int lo = D->tile_lo[t], hi = D->tile_start[t + 1];
    int n_plp = 0, n_skip = 0, low_mq = 0, had_indel = 0, indel_cnt = 0, clipped = 0, n_overlap = 0;
    int ins_seen = 0, cp = 0;
    CgConsAcc a; cg_cons_init(&a);
    const int doB = P->min_qual_B != 0;
    for (int j = lo; j < hi; j++) {
        const CgRead q = D->rd[j];
        CgCell cell;
        if (!cg_cell(D, &q, c, &cell)) continue;
        n_plp++;
        low_mq += (q.mapq <= P->min_mqual);                               /* 1663 */
        if (cell.indel || cell.is_del) { had_indel = 1; indel_cnt++; }    /* 1664-1665 */
        if (cell.is_refskip) { n_skip++; continue; }
        if ((cell.is_head && cell.qpos > 0) || (cell.is_tail && cell.qpos + 1 < q.l_qseq)) clipped++;   /* 1701-1703 */
        if (!cell.is_tail && !cell.is_head) { n_overlap++; if (cell.indel > 0) ins_seen = 1; }       /* 1705-1708 */
        if (!q.l_qseq) continue;
        int nib = cg_seq_nib(D, &q, cell.qpos);
        int base = cell.is_del ? 4 : cg_nt16_to_base(nib);
        uint8_t qv = cg_cap_qual(D->qual[CG_OFF(&q) + cell.qpos], P, T);
        if (P->any_preserve_qual) {                                        /* 611-623, on the pileup's (capped) copy */
            const int pq = T->preserve_qual[qv];
            if (pq) cp |= 1 << base;
            if (pq > 1) cp |= (1 << base) << 8;
            for (int ins = 1; ins <= cell.indel; ins++)
                if (cell.qpos + ins < q.l_qseq && T->preserve_qual[cg_cap_qual(D->qual[CG_OFF(&q) + cell.qpos + ins], P, T)]) cp |= 1 << 4;
        }
        if (!doB) continue;
        cg_cons_add(T, &a, base, T->effB[((int)q.mapq << 8) | qv]);
    }
    CgColStats st; st.cp = cp; st.n_plp = n_plp; st.n_skip = n_skip; st.low_mq = low_mq; st.had_indel = had_indel; st.indel_cnt = indel_cnt;
    st.clipped = clipped; st.n_overlap = n_overlap; st.ins_seen = ins_seen;
    (void)o;
    return cg_column_finish(D, c, lo, hi, &st, &a);
}

/* ---- stage: flagged (one per flagged column): indel-size spectrum tests and the STR
 * extents of every triggering read (snp_score.c:1690-1762, 1775-1819) ------------------- */
typedef struct CgFlagScratch { uint8_t win[2 * CG_MASK_WIN + 8]; CgRepList reps; int indel_depth[101]; } CgFlagScratch;

CG_HDN uint32_t cg_flagged(const CgDev *D, int k, CgFlagScratch *S) {
    const CgDevParams *P = &D->P;
    const int c = D->fcol[k];
    const int t = c >> 5;
    const int lo = D->tile_lo[t], hi = D->tile_start[t + 1];
    const uint16_t ev = D->ev[c];
    const int n_plp = (int)D->depth[c];
    const int had_indel = (ev & CG_EV_HADINDEL) != 0, lowscore = (ev & CG_EV_LOWSCORE) != 0, strall = (ev & CG_EV_STRALL) != 0;
    uint32_t cnt = 0;
    int is = cg_island_of(D, c);
    const int tid = D->isl[is].tid, pos = D->isl[is].pos_start + (c - D->isl[is].col_start);
    int indel_cnt = 0;
    for (int j = lo; j < hi; j++) {             /* indel_cnt is complete before the trigger loop starts (1662-1666) */
        const CgRead q = D->rd[j]; CgCell cell;
        if (!cg_cell(D, &q, c, &cell)) continue;
        if (cell.indel || cell.is_del) indel_cnt++;
    }
    const int gate = indel_cnt >= n_plp * P->indel_fract;                  /* 1732 */
    int indel_sz = 0; S->indel_depth[0] = 0;
    int m_run = pos, M_run = pos, indel = 0, had_indel_Q = 0;
    CgTrig tr; tr.tid = tid; tr.pos = pos; tr.col = c; tr.hasI = tr.hasS = 0;
    tr.PI = tr.PS = pos; tr.QI = tr.QS = pos;
    for (int j = lo; j < hi; j++) {
        const CgRead q = D->rd[j]; CgCell cell;
        if (!cg_cell(D, &q, c, &cell)) continue;
        if (cell.is_refskip) continue;                                     /* 1696-1697 */
        const int is_indel = (cell.indel || cell.is_del);
        if (!cell.is_head && !cell.is_tail && (cell.indel > 0 || had_indel)) {     /* 1708-1713 */
            while (indel_sz < cell.indel && indel_sz < 100) S->indel_depth[++indel_sz] = 0;
            if (cell.indel >= 0) S->indel_depth[cell.indel < 99 ? cell.indel : 99]++;
        }
        if ((is_indel || strall) && lowscore) {                            /* 1718-1720 */
            if (is_indel) had_indel_Q++;
            if (is_indel) { int v = (cell.indel < 0 ? -cell.indel : cell.indel) + cell.is_del; if (indel < v) indel = v; }
            else indel = 1;                                                /* 1725-1730 */
            if (gate && q.l_qseq > 0) {                                    /* 1732-1739: the two calls are identical in effect */
                int phantom = (q.l_qseq & 1) ? (D->seq[(CG_OFF(&q) >> 1) + (q.l_qseq >> 1)] & 0xf)
                                             : (cg_cap_qual(D->qual[CG_OFF(&q)], P, D->T) >> 4);
                int lo_r = m_run, hi_r = M_run;
                cg_mask_lc(D->seq + (CG_OFF(&q) >> 1), q.l_qseq, phantom, D->cigar + q.cig_off, q.n_cigar, q.pos,
                           cell.qpos + 1, is_indel ? P->iSTR_add : P->sSTR_add, S->win, &S->reps, &lo_r, &hi_r);
                if (S->reps.overflow) *D->err = CG_ERR_OVERFLOW;
#ifdef CG_EMU_CROSSCHECK
                {   /* host emulation only: the bit-parallel search the device runs (k_str_items) must give the same extents on every read the pipeline meets */
                    uint64_t W_[16]; uint32_t ring_[16]; int lo_b = m_run, hi_b = M_run;
                    cg_mask_lc_bits<1, 1>(D->seq + (CG_OFF(&q) >> 1), q.l_qseq, phantom, D->cigar + q.cig_off, q.n_cigar, q.pos,
                                          cell.qpos + 1, is_indel ? P->iSTR_add : P->sSTR_add, W_, ring_, &lo_b, &hi_b);
                    if (!S->reps.overflow && (lo_b != lo_r || hi_b != hi_r)) *D->err = CG_ERR_STATE;
                }
#endif
                m_run = lo_r; M_run = hi_r;
            }
            if (is_indel) { tr.hasI = 1; tr.PI = m_run; tr.QI = M_run; }
            else          { tr.hasS = 1; tr.PS = m_run; tr.QS = M_run; }
        }
    }
    tr.A = m_run; tr.B = M_run; tr.indel = indel;
    D->trig[k] = tr;
    if (had_indel_Q) cnt |= 1u << CG_CNT_INDEL_QUAL;                       /* 1762 */
    uint16_t ev_add = 0; int keep = 0;
    if (indel_sz) {                                                        /* 1777-1819 */
        int qd1 = 0, qd2 = 0, ov = 0;
        for (int i = 0; i <= indel_sz && i < 100; i++) {
            int d = S->indel_depth[i];
            if (!d) continue;
            ov += d;
            if (qd1 < d) { qd2 = qd1; qd1 = d; } else if (qd2 < d) qd2 = d;
        }
        if ((ov - qd1 - qd2) > P->ins_len_perc * (ov + .1)) { ev_add |= CG_EV_INDEL_LEN; keep = 1; cnt |= 1u << CG_CNT_INS_LEN_PERC; }
        if ((double)ov < P->indel_ov_perc * n_plp) { ev_add |= CG_EV_INDEL_COV; keep = 1; cnt |= 1u << CG_CNT_INDEL_OV_PERC; }
    }
    if (tr.hasI || tr.hasS) {
        ev_add |= CG_EV_TRIGGER;
        for (int j = lo; j < hi; j++) {          /* every read of the column is back-filled (1870-1879) */
            const CgRead q = D->rd[j];
            if ((unsigned)(c - q.col0) < (unsigned)q.span) D->r_bf[j] = 1;
        }
    }
    if (ev_add) D->ev[c] = (uint16_t)(ev | ev_add);
    if (keep) D->cb[c] |= CG_CB_KEEP;
    return (ev & CG_EV_REPLAY) ? 0 : cnt;
}

/* ---- stage: chain (sequential, one thread): window state after every flagged column ---- */
CG_HD void cg_chain(const CgDev *D, int n_flagged) {
    CgWin w; cg_win_reset(&w);
    int last_tid = -2;
    for (int k = 0; k < n_flagged; k++) {
        const CgTrig t = D->trig[k];
        if (t.hasI || t.hasS) {
            if (t.tid != last_tid) { cg_win_reset(&w); last_tid = t.tid; }      /* 1478-1485 */
            cg_win_step(&w, &t, &D->P);
        }
        D->twin[k] = w;
    }
}

/* ---- stage: paint (one per flagged column): mark the columns where the keep window opened
 * or extended by trigger k is still active (min_pos != INT_MAX, snp_score.c:1880) ---------- */
CG_HD void cg_paint(const CgDev *D, int k, int n_flagged) {
    const CgTrig t = D->trig[k];
    if (!(t.hasI || t.hasS)) return;
    int64_t end = D->twin[k].max_pos2;                   /* inclusive, reference coordinates */
    for (int k2 = k + 1; k2 < n_flagged; k2++) {         /* next trigger of the same contig takes over from its column */
        const CgTrig *u = &D->trig[k2];
        if (u->tid != t.tid) break;
        if (u->hasI || u->hasS) { if (u->pos - 1 < end) end = u->pos - 1; break; }
    }
    int is = cg_island_of(D, t.col);
    int c = t.col, pos = t.pos;
    for (;;) {
        int isl_end_col = (is + 1 < D->n_islands) ? D->isl[is + 1].col_start : D->n_cols;
        while (c < isl_end_col && pos <= end) { D->cb[c] |= CG_CB_ACTIVE; c++; pos++; }
        if (pos > end || is + 1 >= D->n_islands) break;
        is++;
        if (D->isl[is].tid != t.tid || D->isl[is].pos_start > end) break;
        c = D->isl[is].col_start; pos = D->isl[is].pos_start;
    }
}

/* chained calls: the window the previous call left open stays active over [pos_from, pos_to] of contig tid */
CG_HD void cg_paint_range(const CgDev *D, int tid, int pos_from, int pos_to) {
    int c = cg_find_col(D, tid, pos_from);
    while (c < D->n_cols) {
        const int is = cg_island_of(D, c);
        if (D->isl[is].tid != tid) break;
        const int isl_end_col = (is + 1 < D->n_islands) ? D->isl[is + 1].col_start : D->n_cols;
        int pos = D->isl[is].pos_start + (c - D->isl[is].col_start);
        if (pos > pos_to) break;
        while (c < isl_end_col && pos <= pos_to) { D->cb[c] |= CG_CB_ACTIVE; c++; pos++; }
        if (pos > pos_to) break;                           /* else: on to the next island */
    }
}

/* number of BED events a column emits (none when it was counted by the previous call of a chain) */
CG_HD int cg_event_bits(uint16_t ev) { return (ev & CG_EV_REPLAY) ? 0 : (ev & CG_EV_BEDMASK); }

/* ---- stage: rewrite (one per record): replay of the per-base rewrite loop for ONE read
 * (snp_score.c:1822-1920 seen from the read, SURVEY.md §9.7), tail keep (1939-1940),
 * flush strip + P-block (1090-1100).  Works in place on qual_out.                         */
CG_HD int cg_trig_lower_bound(const CgDev *D, int n_flagged, int col) {
    int lo = 0, hi = n_flagged;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (D->fcol[mid] < col) lo = mid + 1; else hi = mid; }
    return lo;
}

CG_HDN void cg_rewrite(const CgDev *D, int64_t r, int n_flagged) {
    const CgDevParams *P = &D->P;
    const CgTables *T = D->T;
    const int L = D->l_qseq[r];
    const int64_t off = D->off[r];
    const uint8_t *qin = D->qual + off;
    uint8_t *out = D->qual_out + off;
    if (L <= 0) return;
    if (!D->rspan[r]) {
        /* never in the pileup: straight to b_hist; strip bit 7, P-block (1093-1099; 2004-2005) */
        for (int x = 0; x < L; x++) out[x] = qin[x] & 0x7f;
        if (P->pblock) cg_pblock(out, L, P->pblock, P->qcap, T);
        return;
    }
    const int j = D->jmap[r];
    const CgRead q = D->rd[j];
    const uint32_t *cig = D->cigar + q.cig_off;
    /* read-level facts */
    int keep = 0, nopblock = 0;
    for (int c = q.col0; c < q.col0 + q.span; c++) keep |= D->cb[c];
    keep = (keep & CG_CB_KEEP) != 0;
    if (P->region_tid >= 0 && q.pos + q.span - 1 >= P->region_end) keep = 0;      /* tail column never reached */
    if (P->nbed) for (int c = q.col0; c < q.col0 + q.span; c++) if (D->ev[c] & CG_EV_BED) nopblock = 1;     /* 1890-1892 */
    const int apq = P->any_preserve_qual;
    const int head_proc = !(D->cb[q.col0] & CG_CB_UNPROC);
    const uint8_t init_or = (head_proc && q.mapq <= P->min_mqual) ? 0x80 : 0;     /* 1852-1859 */
    for (int x = 0; x < L; x++) out[x] = qin[x] | init_or;
    /* visits in column order */
    {
        int c = q.col0, y = 0;
        for (int k = 0; k < q.n_cigar; k++) {
            int op = cg_cig_op(cig[k]), l = cg_cig_len(cig[k]);
            if (cg_is_mop(op)) {
                for (int i = 0; i < l; i++) {
                    int x = y + i;
                    out[x] = cg_visit(out[x], D->cb[c + i], cg_cap_qual(qin[x], P, T), cg_seq_nib(D, &q, x), P, T,
                                      apq && (D->ev[c + i] & CG_EV_IMPERFECT));
                }
                c += l; y += l;
            } else if (op == 2 || op == 3) {
                if (y < L) {
                    uint8_t oc = cg_cap_qual(qin[y], P, T); int nib = cg_seq_nib(D, &q, y); uint8_t v = out[y];
                    for (int i = 0; i < l; i++) v = cg_visit(v, D->cb[c + i], oc, nib, P, T, apq && (D->ev[c + i] & CG_EV_IMPERFECT));
                    out[y] = v;
                }
                c += l;
            } else if (op == 1 || op == 4) y += l;
        }
    }
    /* -S (1894-1904): at the read's head column the bases before qpos, at its tail column the bases after qpos, are
     * binned in place unless that column set keep_qual.  Only back-fills reach those bases: the head column's own
     * back-fill comes before the binning, those of later trigger columns after it. */
    int head_bin = 0, tail_bin = 0, qh = 0, qt = L - 1;
    if (P->softclip) {
        CgCell ch, ct;
        const uint8_t cbh = D->cb[q.col0], cbt = D->cb[q.col0 + q.span - 1];
        if (cg_cell(D, &q, q.col0, &ch)) { qh = ch.qpos; head_bin = !(cbh & (CG_CB_UNPROC | CG_CB_KEEP)) && qh > 0; }
        if (q.span > 1 && cg_cell(D, &q, q.col0 + q.span - 1, &ct)) { qt = ct.qpos; tail_bin = !(cbt & (CG_CB_UNPROC | CG_CB_KEEP)); }
    }
    /* back-fills from trigger columns under this read (1870-1879) */
    if (D->r_bf[j]) {
        for (int k = cg_trig_lower_bound(D, n_flagged, q.col0); k < n_flagged && D->fcol[k] < q.col0 + q.span; k++) {
            const CgTrig *t = &D->trig[k];
            if (head_bin && t->col > q.col0) { for (int x = 0; x < qh && x < L; x++) out[x] = T->bin2[out[x]]; head_bin = 0; }
            if (!(t->hasI || t->hasS)) continue;
            CgCell cell;
            if (!cg_cell(D, &q, t->col, &cell)) continue;
            int x0 = cg_ref2query_pos(cig, q.n_cigar, q.pos, D->twin[k].min_pos2);
            for (int x = x0; x <= cell.qpos && x < L; x++) out[x] = (uint8_t)(cg_cap_qual(qin[x], P, T) | 0x80);
        }
    }
    if (head_bin) for (int x = 0; x < qh && x < L; x++) out[x] = T->bin2[out[x]];
    if (tail_bin) for (int x = qt + 1; x < L; x++) out[x] = T->bin2[out[x]];
    if (keep) for (int x = 0; x < L; x++) out[x] = cg_cap_qual(qin[x], P, T);      /* 1939-1940 */
    for (int x = 0; x < L; x++) out[x] &= 0x7f;                                     /* 1093-1096 */
    if (P->pblock && !nopblock) cg_pblock(out, L, P->pblock, P->qcap, T);           /* 1098-1099 */
}

/* ---- stage: deep (one per dense column) after the depth scan: over-depth test
 * (snp_score.c:1490-1491, 1673-1687).  tdepth/tcol are total_depth/total_col as they stand
 * at the test, i.e. including this column.                                                */
CG_HD uint32_t cg_deep_test(const CgDev *D, int c, int64_t tdepth, int64_t tcol) {
    const uint16_t ev = D->ev[c];
    if (!(ev & CG_EV_PROCESSED)) return 0;
    int64_t n = D->depth[c];
    if ((double)(n * (tcol + 1)) > D->P.over_depth * (double)(tdepth + 1)) {
        D->ev[c] = (uint16_t)(ev | CG_EV_DEEP);
        D->cb[c] |= CG_CB_KEEP;
        return (ev & CG_EV_REPLAY) ? 0 : 1u << CG_CNT_OVER_DEPTH;
    }
    return 0;
}

/* ---- stages: ingest / emit (cg_process_device) -------------------------------------------
 * Records in GPU memory arrive as "concatenated BAM fields" (cg_dev_batch): qualities and sequences back to back at any byte
 * offset.  ingest moves them into the padded working layout the chain reads (qual at off[r], seq at off[r] / 2, off 8-aligned),
 * emit moves the rewritten qualities back.  Every access on the working side is an aligned 8- or 4-byte word; the caller's side
 * is read as whole aligned 32-bit words joined by funnel shifts, and only words holding at least one byte of the record are read. */
CG_HD uint32_t cg_ld_word(const uint8_t *aligned) {
#ifdef __CUDA_ARCH__
    return *(const uint32_t *)aligned;
#else
    uint32_t v; memcpy(&v, aligned, 4); return v;
#endif
}
CG_HD void cg_st_word(uint8_t *aligned, uint32_t v) {
#ifdef __CUDA_ARCH__
    *(uint32_t *)aligned = v;
#else
    memcpy(aligned, &v, 4);
#endif
}
CG_HD void cg_st_dword(uint8_t *aligned, uint64_t v) {
#ifdef __CUDA_ARCH__
    *(uint64_t *)aligned = v;
#else
    memcpy(aligned, &v, 8);
#endif
}
CG_HD uint32_t cg_funnel_r(uint32_t lo, uint32_t hi, unsigned sh) {    /* sh in 0..31 (also used by cg_cells.h) */
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}
/* bytes [p, p + n), 1 <= n <= 8, as a little-endian word, zero above byte n: the (at most three) aligned words that hold them */
CG_HD uint64_t cg_gather8(const uint8_t *p, int n) {
    const uintptr_t a = (uintptr_t)p & ~(uintptr_t)3, end = (uintptr_t)p + (uintptr_t)n;
    const uint32_t sh = ((uint32_t)(uintptr_t)p & 3u) * 8u;
    const uint8_t *w = (const uint8_t *)a;
    const uint32_t w0 = cg_ld_word(w), w1 = a + 4 < end ? cg_ld_word(w + 4) : 0u, w2 = a + 8 < end ? cg_ld_word(w + 8) : 0u;
    const uint64_t v = (uint64_t)cg_funnel_r(w0, w1, sh) | ((uint64_t)cg_funnel_r(w1, w2, sh) << 32);
    return n >= 8 ? v : v & ((1ull << (8 * n)) - 1);
}

typedef struct CgIngest {
    const int32_t *l_qseq; const int64_t *off;       /* working layout: off[] = running sum of (l_qseq + 7) & ~7 */
    const int64_t *qsrc, *ssrc;                      /* running sums of l_qseq and (l_qseq + 1) / 2: record r in the caller's arrays */
    const uint8_t *qual_in, *seq_in;                 /* the caller's concatenated arrays */
    uint8_t *qual, *seq;                             /* working arrays (past their front padding) */
    int64_t qbase, sbase;                            /* qsrc / ssrc of the caller's first record (a stream: the held records come first) */
} CgIngest;

/* ingest, one item per (record r, group k < (l_qseq + 7) / 8): working qual bytes [off + 8k, off + 8k + 8) and seq bytes
 * [off/2 + 4k, off/2 + 4k + 4).  Bytes past the record are zero, as the host batcher leaves its padding (cg_host.cpp, cgb_add);
 * the record's last seq byte is copied whole, so an odd-length record keeps its phantom low nibble (SURVEY §9.3). */
CG_HD void cg_ingest_group(const CgIngest *I, int64_t r, int k) {
    const int L = I->l_qseq[r];
    const int64_t o = I->off[r];
    const int nq = L - 8 * k;
    uint64_t q = 0; uint32_t s = 0;
    if (nq > 0) {
        const int ns = ((L + 1) >> 1) - 4 * k;                                  /* > 0 whenever nq > 0 */
        q = cg_gather8(I->qual_in + (I->qsrc[r] - I->qbase) + 8 * k, nq < 8 ? nq : 8);
        s = (uint32_t)cg_gather8(I->seq_in + (I->ssrc[r] - I->sbase) + 4 * k, ns < 4 ? ns : 4);
    }
    cg_st_dword(I->qual + o + 8 * k, q);
    cg_st_word(I->seq + (o >> 1) + 4 * k, s);
}

typedef struct CgEmit {
    const int32_t *l_qseq; const int64_t *off, *qdst;   /* qdst = qsrc of CgIngest: the concatenated layout */
    const uint8_t *qout;                               /* rewritten qualities, working layout */
    uint8_t *qual_out;                                 /* the caller's concatenated array */
    int64_t qbase;                                     /* qdst of the record that goes to qual_out[0] */
} CgEmit;

/* emit, one item per (record r, j < cg_emit_words): the 8-byte aligned words of the caller's array that hold bytes of record r.
 * A word wholly inside the record takes one aligned store; the first and last word, shared with the neighbours, take byte stores. */
CG_HD int cg_emit_words(const CgEmit *E, int64_t r) {
    const int L = E->l_qseq[r];
    if (L <= 0) return 0;
    const uintptr_t d0 = (uintptr_t)(E->qual_out + (E->qdst[r] - E->qbase));
    return (int)(((d0 + (uintptr_t)L - 1) >> 3) - (d0 >> 3) + 1);
}
CG_HD void cg_emit_word(const CgEmit *E, int64_t r, int j) {
    const int64_t L = E->l_qseq[r];
    uint8_t *dst = E->qual_out + (E->qdst[r] - E->qbase);
    const int64_t x = -(int64_t)((uintptr_t)dst & 7) + 8 * (int64_t)j;        /* record byte at the word's first address */
    const int64_t x0 = x > 0 ? x : 0, x1 = x + 8 < L ? x + 8 : L;
    const uint64_t v = cg_gather8(E->qout + E->off[r] + x0, (int)(x1 - x0));
    if (x0 == x && x1 == x + 8) cg_st_dword(dst + x, v);
    else for (int64_t b = x0; b < x1; b++) dst[b] = (uint8_t)(v >> (8 * (b - x0)));
}

/* ---- streams (cg_stream_device, DESIGN.md §3.6) ----------------------------------------------------------------------------------
 * One call works on held ++ in (n records; the first e0 of them were emitted by earlier calls).  Every quantity of the cut is a min or
 * max over the records, so the device reduces them with atomics and the emulation with plain loops over the same per-record body. */
typedef struct CgStreamRed {
    int32_t mmax;             /* last record whose key differs from the last record's (-1: none): m = mmax + 1 */
    int32_t mtid;             /* the same among records on the last record's contig: the held-back run continues record m-1's contig iff equal */
    int32_t smin;             /* smallest start of a pileup record on the last record's contig that ends beyond its position (INT_MAX: none) */
    int32_t fmin;             /* first such record at or after e0 (INT_MAX: none) */
    uint64_t kmin, kmax;      /* smallest / largest key of the pileup records of `in` (kmin > kmax: none) */
    int32_t unplaced;         /* `in` holds a record with tid < 0 */
    int32_t pad;
} CgStreamRed;

CG_HD void cg_stream_red_init(CgStreamRed *R) {
    R->mmax = -1; R->mtid = -1; R->smin = 0x7fffffff; R->fmin = 0x7fffffff; R->kmin = ~0ull; R->kmax = 0; R->unplaced = 0; R->pad = 0;
}
/* A record is open at the cut (cut_tid, limit): a pileup record (span = cg_pileup_span) on contig cut_tid that ends beyond limit.
 * With limit = X it is not final yet; with limit = S it belongs to the next call's read halo. */
CG_HD bool cg_open_at(int32_t tid, int32_t pos, int32_t span, int32_t cut_tid, int32_t limit) {
    return span && tid == cut_tid && (int64_t)pos + span > limit;
}

/* record r's contribution (identities where it has none); rspan[] as cg_prep_read leaves it, so the end is the pileup's own */
CG_HD CgStreamRed cg_stream_plan_item(const CgDev *D, int64_t r, int64_t n, int64_t n_held, int64_t e0) {
    CgStreamRed c; cg_stream_red_init(&c);
    const int32_t tL = D->tid[n - 1], pL = D->pos[n - 1], t = D->tid[r], p = D->pos[r], sp = D->rspan[r];
    if (t != tL || p != pL) { c.mmax = (int32_t)r; if (t == tL) c.mtid = (int32_t)r; }
    if (cg_open_at(t, p, sp, tL, pL)) { c.smin = p; if (r >= e0) c.fmin = (int32_t)r; }
    if (r >= n_held) {
        if (sp) c.kmin = c.kmax = (uint64_t)cg_key(t, p);
        if (t < 0) c.unplaced = 1;
    }
    return c;
}
CG_HD void cg_stream_red_merge(CgStreamRed *a, const CgStreamRed *b) {
    if (b->mmax > a->mmax) a->mmax = b->mmax;
    if (b->mtid > a->mtid) a->mtid = b->mtid;
    if (b->smin < a->smin) a->smin = b->smin;
    if (b->fmin < a->fmin) a->fmin = b->fmin;
    if (b->kmin < a->kmin) a->kmin = b->kmin;
    if (b->kmax > a->kmax) a->kmax = b->kmax;
    a->unplaced |= b->unplaced;
}

typedef struct CgStreamCut {
    int32_t m;                /* the call covers records [0, m); [m, n) is the held-back run */
    int32_t f;                /* records [e0, f) are final and emitted */
    int32_t hi_tid, hi_pos;   /* X: the columns at/after it are left to later calls (hi_tid < 0: none) */
    int32_t S;                /* next_lo_pos: the smallest start of a record of the call reaching beyond X (X if none) */
    int32_t skip;             /* m <= e0: the call covers no record that is not emitted yet; it runs nothing and holds everything */
    int64_t q_e0, q_f;        /* concatenated quality offsets of records e0 and f */
} CgStreamCut;

/* the cut from the reductions; qsrc[] = running sum of l_qseq over the working batch, q_total its total */
CG_HD CgStreamCut cg_stream_cut(const CgDev *D, const CgStreamRed *R, int64_t n, int64_t e0, int last, const int64_t *qsrc, int64_t q_total) {
    CgStreamCut c; memset(&c, 0, sizeof c);
    c.hi_tid = -1;
    c.m = (int32_t)n;
    if (!last && n > 0 && D->tid[n - 1] >= 0) {              /* after an unplaced record only unplaced ones follow: nothing to hold back */
        c.m = R->mmax + 1;
        if (R->mmax >= 0 && R->mtid == R->mmax) { c.hi_tid = D->tid[n - 1]; c.hi_pos = D->pos[n - 1]; }
    }
    c.S = c.hi_tid >= 0 && R->smin < c.hi_pos ? R->smin : c.hi_pos;
    c.f = c.hi_tid >= 0 && R->fmin < c.m ? R->fmin : c.m;
    c.skip = c.m <= e0;
    if (c.skip) c.f = (int32_t)e0;
    c.q_e0 = e0 < n ? qsrc[e0] : q_total;
    c.q_f = c.f < n ? qsrc[c.f] : q_total;
    return c;
}

/* record r stays for later calls: the read halo before f (pileup records on hi_tid reaching beyond S), then everything from f on */
CG_HD int cg_stream_keep(const CgDev *D, int64_t r, const CgStreamCut *c) {
    if (c->skip || r >= c->f) return 1;
    const int32_t sp = D->rspan[r];
    return sp && cg_open_at(D->tid[r], D->pos[r], sp, c->hi_tid, c->S);    /* rspan first: tid and pos are loaded for pileup records only */
}

typedef struct CgRetain {
    const int32_t *tid, *pos, *l_qseq; const uint16_t *flag, *n_cigar; const uint8_t *mapq;
    const int64_t *off; const int32_t *cigar_off; const uint32_t *cigar; const uint8_t *qual, *seq;   /* working batch */
    const int32_t *didx, *dcig; const int64_t *doff;                   /* where kept record r goes: exclusive scans over the keep flag */
    int32_t *h_tid, *h_pos, *h_lq; uint16_t *h_flag, *h_nc; uint8_t *h_mapq;
    uint32_t *h_cigar; uint8_t *h_qual, *h_seq;                        /* the held store, in the working layout */
} CgRetain;

/* one item per (kept record r, j < cg_retain_items): item 0 moves the per-record fields; item j moves the j-th 8-byte word of the padded
 * qualities, the j-th 4-byte word of the sequence and the j-th CIGAR operation, where they exist */
CG_HD int cg_retain_items(const CgRetain *K, int64_t r) {
    const int w = (K->l_qseq[r] + 7) >> 3, nc = K->n_cigar[r];
    const int v = w > nc ? w : nc;
    return v > 1 ? v : 1;
}
CG_HD void cg_retain_item(const CgRetain *K, int64_t r, int j) {
    const int64_t d = K->didx[r];
    if (j == 0) {
        K->h_tid[d] = K->tid[r]; K->h_pos[d] = K->pos[r]; K->h_lq[d] = K->l_qseq[r];
        K->h_flag[d] = K->flag[r]; K->h_nc[d] = K->n_cigar[r]; K->h_mapq[d] = K->mapq[r];
    }
    if (j < K->n_cigar[r]) K->h_cigar[K->dcig[r] + j] = K->cigar[K->cigar_off[r] + j];
    if (j < (K->l_qseq[r] + 7) >> 3) {
        const int64_t s = K->off[r] + 8 * (int64_t)j, t = K->doff[r] + 8 * (int64_t)j;
#ifdef __CUDA_ARCH__
        *(uint64_t *)(K->h_qual + t) = *(const uint64_t *)(K->qual + s);
        *(uint32_t *)(K->h_seq + (t >> 1)) = *(const uint32_t *)(K->seq + (s >> 1));
#else
        memcpy(K->h_qual + t, K->qual + s, 8);
        memcpy(K->h_seq + (t >> 1), K->seq + (s >> 1), 4);
#endif
    }
}

#endif /* CG_PIPELINE_H */
