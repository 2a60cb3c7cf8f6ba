/*
 * cg_core.h — per-cell / per-column / per-read building blocks of the device path.
 *
 * Every function here is `__host__ __device__` so the very same source is compiled
 * (a) by nvcc into the sm_100a kernels of cg_device.cu — the product path — and
 * (b) by g++ into tests/emu/, a host emulation of the kernel decomposition used only
 * by the CPU test-suite to debug the decomposition where no GPU exists.  (b) is never
 * linked into libcrumble_gpu.so.
 *
 * Each block cites the reference lines whose behaviour it reproduces.  Floating point:
 * compile device code with -fmad=false; all double arithmetic below is written so that
 * the sequence of IEEE operations equals the reference's (SURVEY.md §8 "a3 contract").
 */
#ifndef CG_CORE_H
#define CG_CORE_H

#include <stdint.h>
#include <limits.h>
#include <float.h>
#include <math.h>

#ifdef __CUDACC__
#define CG_HD __host__ __device__ __forceinline__
#define CG_HDN __host__ __device__ __noinline__
#else
#define CG_HD static inline
#define CG_HDN static __attribute__((unused))
#endif

#define CG_MAX_DEPTH   20000      /* snp_score.c:92  */
#define CG_MASK_WIN    250        /* snp_score.c:1229 */
#define CG_BED_DIST    50         /* snp_score.c:149 */
#define CG_REP_CAP     640        /* upper bound on live repeats in a 501-base window */

/* ---- tables built on the host with libm and uploaded (consensus_init, snp_score.c:378-489;
 *      q2p/mqual_pow 564-574; bin2 234-247) ------------------------------------------ */
typedef struct CgTables {
    double  lprior15[16];
    double  MM[128];          /* pMM[q] - p__[q]            (snp_score.c:645) */
    double  _M[128];          /* p_M[q] - p__[q]            (snp_score.c:646) */
    double  q2p[128];         /* 10^(-q/10)                 (snp_score.c:565) */
    double  omq2p[128];       /* 1 - q2p[q]                 (snp_score.c:651) */
    double  e_tab[1002];      /* exp(i),    i = -500..500, index i+500 (snp_score.c:381-382) */
    double  e_tab2[1002];     /* exp(i/10.)                              (snp_score.c:383-384) */
    double  min_e_exp;        /* DBL_MIN_EXP*log(2)+1       (snp_score.c:540) */
    double  log_c1, log_c2;   /* (double)(-1.0f/3), (double)(2.0f/3)    (snp_score.c:515) */
    uint8_t effB[65536];      /* [mapq<<8|qual] -> max(1, (uint8_t)ph_log(1-(_m*_p+(1-_m)/4))) (632-642), qual capped first (1325-1332) */
    uint16_t cellB[65536];    /* [mapq<<8|qual] -> the read-and-quality part of a pileup cell (cg_cells.h): valid | effB << 5 | (mapq <= -m) */
    uint8_t effA[256];        /* mode A: max(1,qual), clamped to the table size */
    uint8_t bin2[256];        /* snp_score.c:234-247 (values are < 256 for sane -l/-u) */
    uint8_t preserve_qual[256];
} CgTables;

/* device-side copy of the options that the kernels need */
typedef struct CgDevParams {
    int32_t reduce_qual, binary_qual;
    int32_t iSTR_add, sSTR_add;
    double  iSTR_mul, sSTR_mul;
    int32_t qlow, qhigh, qcap, qcutoff;
    int32_t min_mqual;
    double  indel_fract;
    int32_t min_qual_A, min_indel_A; double min_discrep_A;
    int32_t min_qual_B, min_indel_B; double min_discrep_B;
    double  low_mqual_perc, clip_perc, ins_len_perc, over_depth, indel_ov_perc;
    int32_t pblock, softclip, perfect_col;
    int32_t region_tid, region_beg, region_end;
    int32_t str_snp;          /* sSTR_add || sSTR_mul (snp_score.c:1345) */
    int32_t any_preserve_qual;
    int32_t nbed;             /* -R regions (snp_score.c:1443-1463) */
    /* column window of a chained call (cg_process_window, include/crumble_gpu.h): which columns this call owns */
    int32_t win_on, win_lo_tid, win_lo_pos, win_cnt_pos, win_hi_tid, win_hi_pos;
} CgDevParams;

#include <stddef.h>
#ifdef __cplusplus
static_assert(offsetof(CgTables, e_tab2) == offsetof(CgTables, e_tab) + 1002 * sizeof(double), "cg_fast_exp indexes e_tab2 through e_tab");
#endif

/* ---- CIGAR ------------------------------------------------------------------------- */
CG_HD int cg_cig_op(uint32_t c)  { return (int)(c & 0xf); }
CG_HD int cg_cig_len(uint32_t c) { return (int)(c >> 4); }
CG_HD int cg_cig_type(int op)    { return (0x3C1A7 >> (op << 1)) & 3; }   /* bit0 query, bit1 ref */
CG_HD bool cg_is_refop(int op)   { return op == 0 || op == 2 || op == 3 || op == 7 || op == 8; }
CG_HD bool cg_is_mop(int op)     { return op == 0 || op == 7 || op == 8; }

/* A record's pileup span, the one definition every cut, halo and batch end derives from (its end is pos + span): 0 outside the pileup
 * (unplaced, unmapped, or no op consumes the reference; bam_plp_push + pileup_callback snp_score.c:1125-1149), else the reference
 * span, at least 1 (bam_endpos: pos+1 when the ops that consume the reference have length 0) */
CG_HD int cg_pileup_span(int32_t tid, int flag, const uint32_t *cig, int n) {
    int span = 0, hasref = 0;
    for (int k = 0; k < n; k++)
        if (cg_cig_type(cg_cig_op(cig[k])) & 2) { span += cg_cig_len(cig[k]); hasref = 1; }
    if (tid < 0 || (flag & 4) || !hasref) return 0;
    return span ? span : 1;
}

/* One pileup cell: what htslib's bam_plp_auto reports for (read, column) — restated in
 * oracle/shim/plp.c from SURVEY.md §9.2; d = column - read start on the reference. */
typedef struct CgCell {
    int32_t qpos, indel;
    uint8_t is_del, is_refskip, is_head, is_tail;
} CgCell;

CG_HD bool cg_plp_resolve(const uint32_t *cig, int n_cigar, int d, int span, CgCell *c) {
    int x = 0, y = 0;
    for (int k = 0; k < n_cigar; k++) {
        int op = cg_cig_op(cig[k]), l = cg_cig_len(cig[k]);
        if (cg_is_refop(op)) {
            if (d < x + l) {
                c->indel = 0; c->is_del = 0; c->is_refskip = 0;
                if (x + l - 1 == d && k + 1 < n_cigar) {
                    int op2 = cg_cig_op(cig[k + 1]), l2 = cg_cig_len(cig[k + 1]);
                    if (op2 == 2) c->indel = -l2;
                    else if (op2 == 1) c->indel = l2;
                    else if (op2 == 6 && k + 2 < n_cigar) {
                        int l3 = 0;
                        for (int j = k + 2; j < n_cigar; j++) {
                            int o3 = cg_cig_op(cig[j]);
                            if (o3 == 1) l3 += cg_cig_len(cig[j]);
                            else if (cg_is_refop(o3)) break;
                        }
                        if (l3 > 0) c->indel = l3;
                    }
                }
                if (cg_is_mop(op)) c->qpos = y + (d - x);
                else { c->is_del = 1; c->qpos = y; c->is_refskip = (op == 3); }
                c->is_head = (d == 0); c->is_tail = (d == span - 1);
                return true;
            }
            x += l;
            if (cg_is_mop(op)) y += l;
        } else if (op == 1 || op == 4) y += l;
    }
    return false;
}

/* ref2query_pos, snp_score.c:1156-1179 (pos/rpos are absolute reference coordinates) */
CG_HD int cg_ref2query_pos(const uint32_t *cig, int n, int rpos, int pos) {
    int p = rpos, q = 0;
    for (int i = 0; i < n; i++) {
        int op = cg_cig_op(cig[i]), l = cg_cig_len(cig[i]), t = cg_cig_type(op);
        if (p + ((t & 2) ? l : 0) < pos) {
            if (t & 1) q += l;
            if (t & 2) p += l;
            continue;
        }
        if (t & 1) q += (pos - p);
        return q >= 0 ? q : 0;
    }
    return q;
}

/* bam_qpos2rpos, snp_score.c:1205-1219 */
CG_HD int cg_qpos2rpos(const uint32_t *cig, int n, int rpos0, int qpos) {
    int rpos = rpos0, aq = 0;
    for (int k = 0; k < n && aq < qpos; k++) {
        int op = cg_cig_op(cig[k]), l = cg_cig_len(cig[k]), t = cg_cig_type(op);
        if (t & 2) rpos += (l <= qpos - aq) ? l : qpos - aq;
        if (t & 1) aq += l;
    }
    return rpos;
}

/* ---- fast math (snp_score.c:491-527) ------------------------------------------------ */
CG_HD double cg_fast_exp(const CgTables *T, double y) {
    /* one load from the pair of adjacent tables (e_tab2 follows e_tab): the index is selected, not the value */
    const bool fine = y >= -50 && y <= 50;
    double yc = y < -500 ? -500 : y;
    if (yc > 500) yc = 500;
    const int idx = fine ? 1002 + 500 + (int)(y * 10) : 500 + (int)yc;
    return T->e_tab[idx];
}

/* the same for y <= 0 (a genotype sum minus the largest one): the upper clamps of fast_exp are dead and drop out */
CG_HD double cg_fast_exp_neg(const CgTables *T, double y) {
    const bool fine = y >= -50;
    const double t = fine ? y * 10 : (y < -500 ? -500 : y);
    return T->e_tab[(fine ? 1002 + 500 : 500) + (int)t];
}

CG_HD double cg_fast_log2(const CgTables *T, double val) {
    union { double d; int64_t i; } u;
    u.d = val;
    int64_t x = u.i;
    const int log_2 = (int)((x >> 52) & 2047) - 1024;
    x &= ~(2047LL << 52);
    x += 1023LL << 52;
    u.i = x;
    val = u.d;
    val = (T->log_c1 * val + 2) * val - T->log_c2;
    return val + log_2;
}
#define CG_TENLOG2OVERLOG10 3.0103
CG_HD double cg_ph_log(const CgTables *T, double x) { return -CG_TENLOG2OVERLOG10 * cg_fast_log2(T, x); }

/* ---- consensus (calculate_consensus_pileup, snp_score.c:533-797) --------------------- */
typedef struct CgConsAcc {
    double S[15];
    double sumsC[5];
    double sumsE;
    int depth, nN;
} CgConsAcc;

CG_HD void cg_cons_init(CgConsAcc *a) {
#ifdef __CUDACC__
#pragma unroll
#endif
    for (int j = 0; j < 15; j++) a->S[j] = 0;
#ifdef __CUDACC__
#pragma unroll
#endif
    for (int j = 0; j < 5; j++) a->sumsC[j] = 0;
    a->sumsE = 0; a->depth = 0; a->nN = 0;
}

/* nt16 -> ACGT*N index (table L[] at snp_score.c:603-605) */
CG_HD int cg_nt16_to_base(int nib) {
    return (0x5555555355525105ULL >> (nib << 2)) & 0xf;   /* {5,0,1,5, 2,5,5,5, 3,5,5,5, 5,5,5,5} */
}

/* one read into the accumulators; eq = effective quality (>= 1) (snp_score.c:644-685).
 * Slot order of S[]: AA AC AG AT A* CC CG CT C* GG GT G* TT T* **                        */
CG_HD void cg_cons_add(const CgTables *T, CgConsAcc *a, int base, int eq) {
    const double MM = T->MM[eq], _M = T->_M[eq];
    a->sumsE += T->q2p[eq];
    const double om = T->omq2p[eq];
    if (base < 5) {
        const bool b0 = base == 0, b1 = base == 1, b2 = base == 2, b3 = base == 3, b4 = base == 4;
        if (b0) a->sumsC[0] += om;
        if (b1) a->sumsC[1] += om;
        if (b2) a->sumsC[2] += om;
        if (b3) a->sumsC[3] += om;
        if (b4) a->sumsC[4] += om;
        if (b0) a->S[0] += MM;
        if (b0 || b1) a->S[1] += _M;
        if (b0 || b2) a->S[2] += _M;
        if (b0 || b3) a->S[3] += _M;
        if (b0 || b4) a->S[4] += _M;
        if (b1) a->S[5] += MM;
        if (b1 || b2) a->S[6] += _M;
        if (b1 || b3) a->S[7] += _M;
        if (b1 || b4) a->S[8] += _M;
        if (b2) a->S[9] += MM;
        if (b2 || b3) a->S[10] += _M;
        if (b2 || b4) a->S[11] += _M;
        if (b3) a->S[12] += MM;
        if (b3 || b4) a->S[13] += _M;
        if (b4) a->S[14] += MM;
    } else {
        /* N: MM to every non-pad combination, _M to the pad-containing ones, nothing to ** (677-682) */
        a->S[0] += MM; a->S[1] += MM; a->S[2] += MM; a->S[3] += MM; a->S[4] += _M;
        a->S[5] += MM; a->S[6] += MM; a->S[7] += MM; a->S[8] += _M;
        a->S[9] += MM; a->S[10] += MM; a->S[11] += _M;
        a->S[12] += MM; a->S[13] += _M;
        a->nN++;
    }
    a->depth++;
}

typedef struct CgCons {
    int32_t call, het_call, het_phred, phred, depth;
    float discrep;
} CgCons;

/* "and speculate" (snp_score.c:690-794) */
CG_HD void cg_cons_finalize(const CgTables *T, CgConsAcc *a, CgCons *o) {
    double S[15], norm[15];
    double shift = -DBL_MAX, mx = -DBL_MAX, mx_het = -DBL_MAX;
    int call = 0, het_call = 0;
#ifdef __CUDACC__
#pragma unroll
#endif
    for (int j = 0; j < 15; j++) {
        S[j] = a->S[j] + T->lprior15[j];
        if (shift < S[j]) shift = S[j];
        if (j != 0 && j != 5 && j != 9 && j != 12 && j != 14) {
            if (mx_het < S[j]) { mx_het = S[j]; het_call = j; }
        } else {
            if (mx < S[j]) { mx = S[j]; call = j; }
        }
    }
#ifdef __CUDACC__
#pragma unroll
#endif
    for (int j = 0; j < 15; j++) {
        S[j] -= shift;
        double e = cg_fast_exp(T, S[j]);
        S[j] = (S[j] > T->min_e_exp) ? e : DBL_MIN;
        norm[j] = 0;
    }
    double tot1 = 0, tot2 = 0;
#ifdef __CUDACC__
#pragma unroll
#endif
    for (int j = 0; j < 15; j++) {
        norm[j] += tot1;
        norm[14 - j] += tot2;
        tot1 += S[j];
        tot2 += S[14 - j];
    }
    if (a->depth && a->depth != a->nN) {
        const int map_sing[15] = { 0, 5, 5, 5, 5, 1, 5, 5, 5, 2, 5, 5, 3, 5, 4 };
        const int map_het[15]  = { 0, 1, 2, 3, 4, 6, 7, 8, 9, 12, 13, 14, 18, 19, 24 };
        double ncall = 0, nhet = 0, shet = 0;
        int cs = 5, ch = 0;
#ifdef __CUDACC__
#pragma unroll
#endif
        for (int j = 0; j < 15; j++) {          /* static indexing keeps S/norm in registers */
            if (j == call) { ncall = norm[j]; cs = map_sing[j]; }
            if (j == het_call) { nhet = norm[j]; shet = S[j]; ch = map_het[j]; }
        }
        o->depth = a->depth;
        o->call = cs;
        if (ncall == 0) ncall = DBL_MIN;
        int ph = (int)(cg_ph_log(T, ncall) + .5);
        o->phred = ph > 255 ? 255 : (ph < 0 ? 0 : ph);
        o->het_call = ch;
        if (nhet == 0) nhet = DBL_MIN;
        ph = (int)(CG_TENLOG2OVERLOG10 * (cg_fast_log2(T, shet) - cg_fast_log2(T, nhet)) + .5);
        o->het_phred = ph;
        double m = a->sumsC[0] + a->sumsC[1] + a->sumsC[2] + a->sumsC[3] + a->sumsC[4];
        double c;
        if (o->het_phred > 0) {
            double c1 = 0, c2 = 0; int h1 = ch % 5, h2 = ch / 5;
#ifdef __CUDACC__
#pragma unroll
#endif
            for (int j = 0; j < 5; j++) { if (j == h1) c1 = a->sumsC[j]; if (j == h2) c2 = a->sumsC[j]; }
            c = c1 + c2;
        } else {
            c = 0;
#ifdef __CUDACC__
#pragma unroll
#endif
            for (int j = 0; j < 5; j++) if (j == cs) c = a->sumsC[j];
        }
        o->discrep = (float)((m - c) / sqrt(m));
    } else {
        o->call = 5; o->het_call = 0; o->het_phred = 0; o->phred = 0; o->depth = 0; o->discrep = 0;
    }
}

/* ---- column record encodings shared by the kernels ------------------------------------ */
/* cb[c] (u8): what the per-read rewrite needs from a column */
#define CG_CB_CALL_MASK   0x0f      /* nt16 codes of call1 | call2 (A=1 C=2 G=4 T=8; '*' and N match no base) */
#define CG_CB_UNPROC      0x10      /* column not processed (all ref-skip, VDEEP, outside -r) */
#define CG_CB_PRESERVE    0x20      /* snp_score.c:1624-1628,1648-1649 */
#define CG_CB_ACTIVE      0x40      /* min_pos != INT_MAX at this column (snp_score.c:1880) */
#define CG_CB_KEEP        0x80      /* keep_qual (snp_score.c:1668,1679,1771,1805,1816) */
/* ev[c] (u16): sparse facts */
#define CG_EV_VDEEP       0x0001
#define CG_EV_DEEP        0x0002
#define CG_EV_CLIP        0x0004
#define CG_EV_INDEL_LEN   0x0008
#define CG_EV_INDEL_COV   0x0010
#define CG_EV_BEDMASK     0x001f
#define CG_EV_FLAGGED     0x0020    /* second (sparse) pass needed: had_indel or trigger */
#define CG_EV_TRIGGER     0x0040    /* some read opens/extends a keep window here */
#define CG_EV_COUNTED     0x0080    /* not all-refskip, before region end: enters total_depth/total_col */
#define CG_EV_LOWSCORE    0x0100    /* score < min_indel (snp_score.c:1719-1720) */
#define CG_EV_STRALL      0x0200    /* str_snp && preserve: every read triggers (snp_score.c:1718) */
#define CG_EV_HADINDEL    0x0400
#define CG_EV_PROCESSED   0x0800
#define CG_EV_BED         0x1000    /* preserve > 1: column inside a -R region, reads seen here skip the P-block (snp_score.c:1461,1890-1892) */
#define CG_EV_IMPERFECT   0x2000    /* !perfect: preserved quality values disagree with the call (snp_score.c:1606-1608,1633-1645) */
#define CG_EV_REPLAY      0x4000    /* chained call: column already counted by the previous call; processed again for the cross-column state only */

/* call1 | call2 as the set of nt16 codes a base must equal to agree with the call (snp_score.c:1526-1542, 1906-1910):
 * calls 0..3 are A C G T; call 4 ('*' = 16) and 5 (N = 32) never equal an nt16 base code */
CG_HD int cg_call_code(const CgCons *c) {
    int c1, c2;
    if (c->het_phred > 0) { c1 = c->het_call / 5; c2 = c->het_call % 5; }
    else { c1 = c2 = c->call; }
    return ((c1 < 4) ? (1 << c1) : 0) | ((c2 < 4) ? (1 << c2) : 0);
}

/* ---- per-byte visit of the rewrite loop (snp_score.c:1880-1919), see SURVEY.md §9.7 ---- */
CG_HD uint8_t cg_visit(uint8_t val, uint8_t cbv, uint8_t orig_capped, int nib,
                       const CgDevParams *P, const CgTables *T, int imperfect = 0) {
    if (cbv & CG_CB_UNPROC) return val;
    if (cbv & CG_CB_ACTIVE) val = (uint8_t)(orig_capped | 0x80);
    /* 1885: preserve || preserve_qual[*qual & 0x7f] >= 1 + perfect */
    if ((cbv & CG_CB_PRESERVE) || (P->any_preserve_qual && T->preserve_qual[val & 0x7f] >= 2 - imperfect)) val |= 0x80;
    if (!(val & 0x80)) {
        /* base == call1 || base == call2: an nt16 code equals a one-hot call mask iff it is one-hot and inside the set */
        bool match = nib && !(nib & (nib - 1)) && (nib & cbv & CG_CB_CALL_MASK);
        if (match) val = (uint8_t)P->qhigh;
        else if (P->reduce_qual) val = P->binary_qual ? T->bin2[val] : (uint8_t)P->qlow;
    }
    return val;
}

CG_HD uint8_t cg_cap_qual(uint8_t q, const CgDevParams *P, const CgTables *T) {   /* cap_quality, snp_score.c:1325-1332 */
    return (q > P->qcap && !T->preserve_qual[q]) ? (uint8_t)P->qcap : q;
}

/* ---- P-block (pblock, snp_score.c:803-834), in place on qual[0..len) --------------------
 * A run whose bytes all equal the value it would be filled with is left alone (same result, no stores);
 * HASP = 0 when the preserve_qual table is all zero (no -k/-K), which removes the per-byte table lookups. */
template <int HASP>
CG_HD void cg_pblock_t(uint8_t *qual, int len, int level, int qcap, const CgTables *T) {
    int i, j, qmin = INT_MAX, qmax = INT_MIN, last_qmin = 0, last_qmax = 0, mid;
    level *= 2;
    for (i = j = 0; i < len; i++) {
        int q = qual[i];
        if (qmin > q) qmin = q;
        if (qmax < q) qmax = q;
        if (qmax - qmin > level || (HASP && T->preserve_qual[q])) {
            mid = (last_qmin + last_qmax) / 2;
            if (mid > qcap) mid = qcap;
            if (last_qmin != last_qmax || mid != last_qmin) for (int k = j; k < i; k++) qual[k] = (uint8_t)mid;
            if (HASP) while (i < len && T->preserve_qual[qual[i]]) i++;
            if (i < len) qmin = qmax = qual[i];        /* the reference reads qual[len] here; value unused when i==len */
            j = i;
        }
        last_qmin = qmin; last_qmax = qmax;
    }
    mid = (last_qmin + last_qmax) / 2;
    if (last_qmin != last_qmax) for (int k = j; k < i && k < len; k++) qual[k] = (uint8_t)mid;
}
CG_HD void cg_pblock(uint8_t *qual, int len, int level, int qcap, const CgTables *T) { cg_pblock_t<1>(qual, len, level, qcap, T); }

/* ---- STR finder (find_STR / add_rep, str_finder.c:34-189) on 2-bit codes ---------------- */
typedef struct CgRepList { int n; int overflow; int16_t start[CG_REP_CAP]; int16_t end[CG_REP_CAP]; } CgRepList;   /* window positions: 0..500 */

/* seq_nt16_str char -> L[] of str_finder.c:15-32: C->1, G->2, T->3, everything else 0 */
CG_HD uint8_t cg_nt16_to_2bit(int nib) { return nib == 2 ? 1 : nib == 4 ? 2 : nib == 8 ? 3 : 0; }

CG_HD void cg_add_rep(CgRepList *L, const uint8_t *s, int clen, int pos, int rlen) {
    if (L->n) {                                             /* str_finder.c:41-45 */
        int t = L->n - 1;
        if (L->start[t] <= pos - rlen * 2 + 1 && L->end[t] >= pos) return;
    }
    int c1 = pos - rlen + 1, c2 = pos + 1;                  /* str_finder.c:49-74 (no pads in read windows) */
    while (c2 < clen && s[c1] == s[c2]) { c1++; c2++; }
    int el_end = c2 - 1;                                    /* str_finder.c:79 */
    int el_start = pos + 1 - 2 * rlen;                      /* str_finder.c:80-87 */
    /* drop older items contained in the new one (str_finder.c:106-122) */
    int k = L->n - 1;
    while (k >= 0 && L->end[k] >= el_start) k--;
    int w = k + 1;
    for (int i = k + 1; i < L->n; i++)
        if (L->start[i] < el_start) { L->start[w] = L->start[i]; L->end[w] = L->end[i]; w++; }
    if (w >= CG_REP_CAP) { L->overflow = 1; L->n = w; return; }
    L->start[w] = (int16_t)el_start; L->end[w] = (int16_t)el_end;
    L->n = w + 1;
}

CG_HDN void cg_find_str(const uint8_t *s, int len, CgRepList *L) {
    int i, j; uint32_t w = 0;
    L->n = 0; L->overflow = 0;
    for (i = j = 0; i < len && j < 15; i++) {               /* str_finder.c:140-162 */
        w <<= 2; w |= s[i];
        if (j >= 1  && (w & 0x0003) == ((w >> 2)  & 0x0003)) cg_add_rep(L, s, len, i, 1);
        if (j >= 3  && (w & 0x000f) == ((w >> 4)  & 0x000f)) cg_add_rep(L, s, len, i, 2);
        if (j >= 5  && (w & 0x003f) == ((w >> 6)  & 0x003f)) cg_add_rep(L, s, len, i, 3);
        if (j >= 7  && (w & 0x00ff) == ((w >> 8)  & 0x00ff)) cg_add_rep(L, s, len, i, 4);
        if (j >= 9  && (w & 0x03ff) == ((w >> 10) & 0x03ff)) cg_add_rep(L, s, len, i, 5);
        if (j >= 11 && (w & 0x0fff) == ((w >> 12) & 0x0fff)) cg_add_rep(L, s, len, i, 6);
        if (j >= 13 && (w & 0x3fff) == ((w >> 14) & 0x3fff)) cg_add_rep(L, s, len, i, 7);
        j++;
    }
    for (; i < len; i++) {                                   /* str_finder.c:164-186 */
        w <<= 2; w |= s[i];
        if      ((w & 0xffff) == ((w >> 16) & 0xffff)) cg_add_rep(L, s, len, i, 8);
        else if ((w & 0x3fff) == ((w >> 14) & 0x3fff)) cg_add_rep(L, s, len, i, 7);
        else if ((w & 0x0fff) == ((w >> 12) & 0x0fff)) cg_add_rep(L, s, len, i, 6);
        else if ((w & 0x03ff) == ((w >> 10) & 0x03ff)) cg_add_rep(L, s, len, i, 5);
        else if ((w & 0x00ff) == ((w >> 8)  & 0x00ff)) cg_add_rep(L, s, len, i, 4);
        else if ((w & 0x003f) == ((w >> 6)  & 0x003f)) cg_add_rep(L, s, len, i, 3);
        else if ((w & 0x000f) == ((w >> 4)  & 0x000f)) cg_add_rep(L, s, len, i, 2);
        else if ((w & 0x0003) == ((w >> 2)  & 0x0003)) cg_add_rep(L, s, len, i, 1);
    }
}

/* mask_LC_regions (snp_score.c:1230-1290): reference extents [*lo,*hi] of the repeats
 * overlapping rpos +- add in one read.  seq4 = packed 4-bit sequence, phantom = nibble that
 * the reference reads at index l_qseq (SURVEY.md §9.3 item 1).  lo/hi are only narrowed/
 * widened (callers start them at INT_MAX / 0 or at the running min_pos / max_pos).       */
CG_HDN void cg_mask_lc(const uint8_t *seq4, int l_qseq, int phantom, const uint32_t *cig, int n_cigar,
                       int read_pos, int rpos, int add, uint8_t *win /* >= 501 bytes */, CgRepList *L,
                       int *lo, int *hi) {
    int start = rpos - CG_MASK_WIN; if (start < 0) start = 0;
    int end = rpos + CG_MASK_WIN;   if (end > l_qseq) end = l_qseq;
    int len = end - start + 1;
    for (int i = start; i <= end; i++) {
        int nib = (i < l_qseq) ? ((seq4[i >> 1] >> ((~i & 1) << 2)) & 0xf) : phantom;
        win[i - start] = cg_nt16_to_2bit(nib);
    }
    cg_find_str(win, len, L);
    for (int k = 0; k < L->n; k++) {
        if (!(rpos + add >= L->start[k] + start && rpos - add <= L->end[k] + start)) continue;
        int s = cg_qpos2rpos(cig, n_cigar, read_pos, L->start[k] + start);
        int e = cg_qpos2rpos(cig, n_cigar, read_pos, L->end[k] + start);
        if (*lo > s) *lo = s;
        if (*hi < e) *hi = e;
    }
}

/* mask_LC_regions again, without the repeat list (the device path: one thread per (trigger column, read)).
 * What the caller wants from find_STR's list is only min start / max end over the FINAL entries that overlap Q = [rpos - add,
 * rpos + add].  Three facts about add_rep (str_finder.c:34-127) make the list unnecessary:
 *  1. the skip test (41-45) looks at the LAST entry only, i.e. the most recently added repeat;
 *  2. the pruning (106-122) drops exactly the earlier entries whose start is >= the new entry's start, and every such entry starts
 *     within the last 15 positions (a repeat found at position i with period p starts at i + 1 - 2p >= i - 15).  Entries that start
 *     before i - 15 are therefore final; at most one live entry exists per start value, so the live ones fit 16 slots indexed by
 *     start mod 16 (an older entry with the same start is itself dropped by the rule);
 *  3. a repeat found at position i starts at >= i - 15, so nothing found beyond rpos + add + 15 can overlap Q, and nothing found
 *     there can prune an entry that does (its start would have to be <= rpos + add): the scan stops there.
 * qpos2rpos is monotone in qpos, so mapping the two extreme window positions equals taking min / max over the mapped entries.
 * live: 16 slots (value = end of the live entry with that start mod 16, -1 = none), LS = stride between slots. */
template <int LS>
CG_HD void cg_mask_lc_lean(const uint8_t *seq4, int l_qseq, int phantom, const uint32_t *cig, int n_cigar,
                           int read_pos, int rpos, int add, int16_t *live, int *lo, int *hi) {
    int start = rpos - CG_MASK_WIN; if (start < 0) start = 0;
    int end = rpos + CG_MASK_WIN;   if (end > l_qseq) end = l_qseq;
    const int len = end - start + 1;
    const int qlo = rpos - start - add, qhi = rpos - start + add;          /* Q in window coordinates */
    int imax = qhi + 15; if (imax > len - 1) imax = len - 1;
    const uint32_t ph2 = cg_nt16_to_2bit(phantom);
#define CG_B2(wi_) (((wi_) + start) < l_qseq ? (uint32_t)cg_nt16_to_2bit((seq4[((wi_) + start) >> 1] >> ((~((wi_) + start) & 1) << 2)) & 0xf) : ph2)
    for (int k = 0; k < 16; k++) live[k * LS] = -1;
    int tail_s = INT_MAX, tail_e = -1;                                     /* no entry yet: the skip test fails */
    int rlo = INT_MAX, rhi = -1;
    uint32_t w = 0;
    for (int i = 0; i <= imax; i++) {
        {   /* the entry that started at i - 16 can no longer be pruned: final */
            const int en = live[(i & 15) * LS];
            if (en >= 0) { const int st = i - 16; if (qhi >= st && qlo <= en) { if (rlo > st) rlo = st; if (rhi < en) rhi = en; } live[(i & 15) * LS] = -1; }
        }
        w = (w << 2) | CG_B2(i);
        /* candidate periods at this position: all matching ones (shortest first) while fewer than 15 bases have been consumed
         * (str_finder.c:140-162), only the longest afterwards (164-186) */
        uint32_t cand = 0;
        if (i < 15) {
            for (int p = 1; p <= 7; p++) if (i >= 2 * p - 1 && ((w ^ (w >> (2 * p))) & ((1u << (2 * p)) - 1u)) == 0) cand |= 1u << p;
        } else {
            for (int p = 8; p >= 1; p--) if (((w ^ (w >> (2 * p))) & (p == 16 ? 0xffffffffu : ((1u << (2 * p)) - 1u))) == 0) { cand = 1u << p; break; }
        }
        while (cand) {
#ifdef __CUDA_ARCH__
            const int p = __ffs((int)cand) - 1;
#else
            const int p = __builtin_ctz(cand);
#endif
            cand &= cand - 1;
            const int ps = i + 1 - 2 * p;
            if (tail_s <= ps && tail_e >= i) continue;                     /* str_finder.c:41-45 */
            int c1 = i - p + 1, c2 = i + 1;                                /* 49-74 */
            while (c2 < len && CG_B2(c1) == CG_B2(c2)) { c1++; c2++; }
            const int en = c2 - 1;
            for (int x = ps; x < i; x++) live[(x & 15) * LS] = -1;         /* 106-122: earlier entries starting at or after ps */
            live[(ps & 15) * LS] = (int16_t)en;
            tail_s = ps; tail_e = en;
        }
    }
    for (int k = 0; k < 16; k++) {                                         /* whatever is still live at the end of the scan */
        const int en = live[k * LS];
        if (en < 0) continue;
        const int st = imax - ((imax - k) & 15);
        if (qhi >= st && qlo <= en) { if (rlo > st) rlo = st; if (rhi < en) rhi = en; }
    }
#undef CG_B2
    if (rhi >= 0) {
        const int s = cg_qpos2rpos(cig, n_cigar, read_pos, rlo + start);
        const int e = cg_qpos2rpos(cig, n_cigar, read_pos, rhi + start);
        if (*lo > s) *lo = s;
        if (*hi < e) *hi = e;
    }
}

/* ---- mask_LC_regions, bit-parallel ------------------------------------------------------------------------------------------------
 * The list-free form above still walks the window base by base, and on the device one thread does that per work item: the lanes of a
 * warp sit at different bases of different reads, so the (rare, long) candidate handling of one lane stalls the other 31.  Here the
 * per-base part becomes word arithmetic on the window held as 2-bit codes, 32 bases per 64-bit word, and the only loop left runs over
 * the candidate positions themselves:
 *   eq_p(x)  = base x equals base x - p                    (one XOR + fold per 32 bases and period)
 *   R_p(i)   = eq_p holds at i, i-1, .., i-p+1             = the test of str_finder.c:140-186 for period p at position i
 *   ext(i,p) = first x > i where eq_p fails or x = len     = the extension loop of add_rep (str_finder.c:49-74)
 * add_rep's list is a stack sorted by start (a new entry drops exactly the entries on top that start at or after it), entries that
 * start more than 15 bases back can no longer be dropped, so a 16-entry ring of (start, end) is enough; what leaves the ring at the
 * bottom is final and folded into the answer straight away.  W: >= (len + 31) / 32 words (16 for the 501-base maximum), stride WS;
 * ring: 16 words, stride RS. */
#if defined(__CUDA_ARCH__)
#define CG_CTZ64(x_) (__ffsll((long long)(x_)) - 1)
#define CG_CTZ32(x_) (__ffs((int)(x_)) - 1)
#define CG_MSB32(x_) (31 - __clz((int)(x_)))
#else
#define CG_CTZ64(x_) __builtin_ctzll(x_)
#define CG_CTZ32(x_) __builtin_ctz(x_)
#define CG_MSB32(x_) (31 - __builtin_clz(x_))
#endif

/* 16 consecutive bases of a packed 4-bit sequence from base index s on, as 2-bit codes of str_finder.c:15-32 (C 1, G 2, T 3, all else 0),
 * base s + j at bits 2j..2j+1.  Bytes beyond last_byte are not touched (the caller overrides or ignores those bases). */
CG_HD uint32_t cg_b2x16(const uint8_t *seq4, int s, int last_byte) {
    const int b0 = s >> 1;
    uint64_t n = 0;
    for (int k = 0; k < 8; k++) { int idx = b0 + k; if (idx > last_byte) idx = last_byte; n |= (uint64_t)seq4[idx] << (8 * k); }
    n = ((n & 0x0f0f0f0f0f0f0f0fULL) << 4) | ((n >> 4) & 0x0f0f0f0f0f0f0f0fULL);          /* nibble j = base 2 * b0 + j */
    if (s & 1) { int idx = b0 + 8; if (idx > last_byte) idx = last_byte; n = (n >> 4) | ((uint64_t)(seq4[idx] >> 4) << 60); }
    const uint64_t M1 = 0x1111111111111111ULL;
    const uint64_t e0 = n & M1, e1 = (n >> 1) & M1, e2 = (n >> 2) & M1, e3 = (n >> 3) & M1;
    const uint64_t is2 = e1 & ~(e0 | e2 | e3), is4 = e2 & ~(e0 | e1 | e3), is8 = e3 & ~(e0 | e1 | e2);
    uint64_t x = (is2 | is8) | ((is4 | is8) << 1);                                         /* the code in the low 2 bits of every nibble */
    x = (x | (x >> 2)) & 0x0f0f0f0f0f0f0f0fULL;
    x = (x | (x >> 4)) & 0x00ff00ff00ff00ffULL;
    x = (x | (x >> 8)) & 0x0000ffff0000ffffULL;
    x = (x | (x >> 16)) & 0x00000000ffffffffULL;
    return (uint32_t)x;
}

template <int WS, int RS>
CG_HD void cg_mask_lc_bits(const uint8_t *seq4, int l_qseq, int phantom, const uint32_t *cig, int n_cigar,
                           int read_pos, int rpos, int add, uint64_t *W, uint32_t *ring, int *lo, int *hi) {
    int start = rpos - CG_MASK_WIN; if (start < 0) start = 0;
    int end = rpos + CG_MASK_WIN;   if (end > l_qseq) end = l_qseq;
    const int len = end - start + 1;
    if (len <= 0 || l_qseq <= 0) return;
    const int qlo = rpos - start - add, qhi = rpos - start + add;          /* Q in window coordinates */
    int imax = qhi + 15; if (imax > len - 1) imax = len - 1;
    const int nw = (len + 31) >> 5, last_byte = (l_qseq - 1) >> 1;
    for (int c = 0; c < nw; c++)
        W[c * WS] = (uint64_t)cg_b2x16(seq4, start + 32 * c, last_byte) | ((uint64_t)cg_b2x16(seq4, start + 32 * c + 16, last_byte) << 32);
    if (end == l_qseq) {                                                   /* the window's last base is the one past the read (SURVEY.md 9.3) */
        const int x = len - 1;
        W[(x >> 5) * WS] = (W[(x >> 5) * WS] & ~(3ULL << (2 * (x & 31)))) | ((uint64_t)cg_nt16_to_2bit(phantom) << (2 * (x & 31)));
    }
    const uint64_t M5 = 0x5555555555555555ULL;
    int tail_s = INT_MAX, tail_e = -1, rlo = INT_MAX, rhi = -1;
    int rb = 0, rn = 0;                                                    /* ring: bottom index, entries */
#define CG_FOLD(e_) do { const int st_ = (int)((e_) >> 16), en_ = (int)((e_) & 0xffffu); \
        if (qhi >= st_ && qlo <= en_) { if (rlo > st_) rlo = st_; if (rhi < en_) rhi = en_; } } while (0)
    for (int b = 0; 16 * b <= imax; b++) {
        /* V: the block's 16 bases in the upper half, the 16 before them in the lower half */
        const uint64_t Wc = W[(b >> 1) * WS];
        const uint64_t V = (b & 1) ? Wc : ((b ? (W[((b >> 1) - 1) * WS] >> 32) : 0ULL) | (Wc << 32));
        uint32_t R[9];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int p = 1; p <= 8; p++) {
            const uint64_t X = V ^ (V << (2 * p));
            uint64_t eq = ~(X | (X >> 1)) & M5;
            if (b == 0) eq &= ~0ULL << (2 * (16 + p));                     /* bases before the window have no partner */
            uint64_t r = eq;
            if (p >= 2) r &= r << 2;                                       /* runs of 2 */
            if (p >= 4) r &= r << 4;                                       /* runs of 4 */
            if (p == 3) r &= eq << 4;
            if (p == 5) r &= eq << 8;
            if (p == 6) r &= (eq & (eq << 2)) << 8;
            if (p == 7) r &= r << 6;                                       /* 4 + 4 overlapping by one */
            if (p == 8) r &= r << 8;
            R[p] = (uint32_t)(r >> 32);
        }
        uint32_t U = R[1] | R[2] | R[3] | R[4] | R[5] | R[6] | R[7] | R[8];
        const int nvalid = imax - 16 * b + 1;
        if (nvalid < 16) U &= (1u << (2 * nvalid)) - 1u;
        while (U) {
            const int j2 = CG_CTZ32(U); U &= U - 1;
            const int i = 16 * b + (j2 >> 1);
            uint32_t m = 0;                                                /* periods matching at i */
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int p = 1; p <= 8; p++) m |= ((R[p] >> j2) & 1u) << p;
            if (i >= 15) m = 1u << CG_MSB32(m);                            /* str_finder.c:164-186: the longest only */
            while (m) {
                const int p = CG_CTZ32(m); m &= m - 1;
                const int ps = i + 1 - 2 * p;
                if (tail_s <= ps && tail_e >= i) continue;                 /* str_finder.c:41-45 */
                int x = i + 1, xe = len;                                   /* 49-74: first x where base x differs from base x - p */
                for (int c = x >> 5; c < nw; c++) {
                    const uint64_t A = W[c * WS], Bp = c ? W[(c - 1) * WS] : 0ULL;
                    const uint64_t Y = A ^ ((A << (2 * p)) | (Bp >> (64 - 2 * p)));
                    uint64_t ne = (Y | (Y >> 1)) & M5;
                    if (c == (x >> 5)) ne &= ~0ULL << (2 * (x & 31));
                    if (ne) { xe = 32 * c + (CG_CTZ64(ne) >> 1); break; }
                }
                if (xe > len) xe = len;
                const int en = xe - 1;
                while (rn > 0 && (int)(ring[((rb + rn - 1) & 15) * RS] >> 16) >= ps) rn--;   /* 106-122 */
                if (rn == 16) { CG_FOLD(ring[rb * RS]); rb = (rb + 1) & 15; rn--; }
                ring[((rb + rn) & 15) * RS] = ((uint32_t)ps << 16) | (uint32_t)en;
                rn++;
                tail_s = ps; tail_e = en;
            }
        }
    }
    for (int k = 0; k < rn; k++) CG_FOLD(ring[((rb + k) & 15) * RS]);
#undef CG_FOLD
    if (rhi >= 0) {
        const int s = cg_qpos2rpos(cig, n_cigar, read_pos, rlo + start);
        const int e = cg_qpos2rpos(cig, n_cigar, read_pos, rhi + start);
        if (*lo > s) *lo = s;
        if (*hi < e) *hi = e;
    }
}

/* ---- keep-window chain (snp_score.c:1508-1511,1741-1755) --------------------------------
 * Per trigger column the device pre-reduces, independently of the incoming state:
 *   A/B   = min/max over pos and every triggered read's STR extents,
 *   PI/QI = running min/max as seen by the LAST indel-type trigger, PS/QS = same for SNP-type.
 * Because pos-(pos-m)*mul-add is monotone in m (mul >= 0) the sequential per-read MIN/MAX
 * with double->int truncation collapses to one evaluation per type (DESIGN.md §chain).     */
typedef struct CgTrig {
    int32_t tid, pos;
    int32_t A, B, PI, QI, PS, QS;
    int32_t hasI, hasS;
    int32_t indel;            /* column variable `indel` (snp_score.c:1725-1730) */
    int32_t col;              /* dense column */
    int32_t jI, jS;           /* device path: last indel-type / SNP-type triggering read (pileup index), -1 if none */
} CgTrig;

typedef struct CgWin { int32_t min_pos, max_pos, min_pos2, max_pos2; } CgWin;

CG_HD void cg_win_reset(CgWin *w) { w->min_pos = INT_MAX; w->max_pos = 0; w->min_pos2 = INT_MAX; w->max_pos2 = 0; }

CG_HD int cg_min_id(int a, double b) { return (int)((a < b) ? (double)a : b); }   /* MIN(int,double) -> int */
CG_HD int cg_max_id(int a, double b) { return (int)((a > b) ? (double)a : b); }

CG_HD void cg_win_step(CgWin *w, const CgTrig *t, const CgDevParams *P) {
    const int pos = t->pos;
    if (pos > w->max_pos2) cg_win_reset(w);                                      /* 1508-1511 */
    if (t->hasI) {
        int m = w->min_pos < t->PI ? w->min_pos : t->PI;
        int M = w->max_pos > t->QI ? w->max_pos : t->QI;
        w->min_pos2 = cg_min_id(w->min_pos2, pos - (pos - m) * P->iSTR_mul - P->iSTR_add);   /* 1746-1749 */
        w->max_pos2 = cg_max_id(w->max_pos2, pos + (M - pos) * P->iSTR_mul + P->iSTR_add);
    }
    if (t->hasS) {
        int m = w->min_pos < t->PS ? w->min_pos : t->PS;
        int M = w->max_pos > t->QS ? w->max_pos : t->QS;
        w->min_pos2 = cg_min_id(w->min_pos2, pos - (pos - m) * P->sSTR_mul - P->sSTR_add);   /* 1751-1754 */
        w->max_pos2 = cg_max_id(w->max_pos2, pos + (M - pos) * P->sSTR_mul + P->sSTR_add);
    }
    if (w->min_pos > t->A) w->min_pos = t->A;
    if (w->max_pos < t->B) w->max_pos = t->B;
}

#endif /* CG_CORE_H */
