/*
 * cg_host.cpp — host-side pieces of the C ABI that need no CUDA: option defaults and
 * level presets, the libm-built lookup tables that are uploaded to the device, and the
 * record batcher (decoded BAM records -> structure-of-arrays).
 */
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <math.h>
#include <float.h>
#include <pthread.h>
#include <unistd.h>
#include "cg_pipeline.h"
#include "cg_host.h"
#include "crumble_host.h"

/* Which option combinations the device path implements today. */
int cg_params_check(const cg_params *p, const char **why) {
    static const char *w_mul = "negative -i/-s STR multipliers";
    static const char *w_bed = "-R regions must be sorted by (tid, start) as bed_load leaves them";
    if (p->iSTR_mul < 0 || p->sSTR_mul < 0) { if (why) *why = w_mul; return CG_ERR_UNSUPPORTED; }
    if (p->nbed < 0 || (p->nbed > 0 && !p->bed)) { if (why) *why = w_bed; return CG_ERR_BAD_ARG; }
    for (int i = 1; i < p->nbed; i++)
        if (p->bed[i].tid < p->bed[i - 1].tid || (p->bed[i].tid == p->bed[i - 1].tid && p->bed[i].start < p->bed[i - 1].start)) { if (why) *why = w_bed; return CG_ERR_BAD_ARG; }
    return 0;
}

/* Options the hand-tuned kernels do not cover (-S, -k/-K/-y, -N, -R): the chain then runs the one-item-per-thread
 * bodies of cg_pipeline.h for the column and rewrite stages (same results, lower throughput). */
int cg_params_generic(const cg_params *p) {
    if (p->softclip || p->perfect_col || p->nbed) return 1;
    for (int i = 0; i < 256; i++) if (p->preserve_qual[i]) return 1;
    return 0;
}

/* inclusive prefix max of the (tid, end) keys: see cg_bed_hit */
void cg_bed_prefix_max(const cg_bed_reg *bed, int n, int64_t *pm) {
    int64_t m = INT64_MIN;
    for (int i = 0; i < n; i++) { int64_t k = ((int64_t)bed[i].tid << 32) | (uint32_t)bed[i].end; if (k > m) m = k; pm[i] = m; }
}

void cg_devparams_from(CgDevParams *d, const cg_params *p) {
    memset(d, 0, sizeof(*d));
    d->reduce_qual = p->reduce_qual; d->binary_qual = p->binary_qual;
    d->iSTR_add = p->iSTR_add; d->sSTR_add = p->sSTR_add; d->iSTR_mul = p->iSTR_mul; d->sSTR_mul = p->sSTR_mul;
    d->qlow = p->qlow; d->qhigh = p->qhigh; d->qcap = p->qcap; d->qcutoff = p->qcutoff;
    d->min_mqual = p->min_mqual; d->indel_fract = p->indel_fract;
    d->min_qual_A = p->min_qual_A; d->min_indel_A = p->min_indel_A; d->min_discrep_A = p->min_discrep_A;
    d->min_qual_B = p->min_qual_B; d->min_indel_B = p->min_indel_B; d->min_discrep_B = p->min_discrep_B;
    d->low_mqual_perc = p->low_mqual_perc; d->clip_perc = p->clip_perc; d->ins_len_perc = p->ins_len_perc;
    d->over_depth = p->over_depth; d->indel_ov_perc = p->indel_ov_perc;
    d->pblock = p->pblock; d->softclip = p->softclip; d->perfect_col = p->perfect_col;
    d->region_tid = p->region_tid; d->region_beg = p->region_beg; d->region_end = p->region_end;
    d->str_snp = (p->sSTR_add || p->sSTR_mul != 0.0);                   /* snp_score.c:1345 */
    for (int i = 0; i < 256; i++) if (p->preserve_qual[i]) d->any_preserve_qual = 1;
    d->nbed = p->nbed;
}

/* ---- tables (host libm; never recomputed on the device) ----------------------------------- */
static double host_fast_log2(double val, double c1, double c2) {       /* snp_score.c:506-518 */
    union { double d; int64_t i; } u; u.d = val;
    int64_t x = u.i;
    const int log_2 = (int)((x >> 52) & 2047) - 1024;
    x &= ~(2047LL << 52);
    x += 1023LL << 52;
    u.i = x; val = u.d;
    val = (c1 * val + 2) * val - c2;
    return val + log_2;
}

void cg_tables_init(CgTables *T, const cg_params *p) {
    memset(T, 0, sizeof(*T));
    const double p_het = 1e-6;                                          /* P_HET, snp_score.c:283 */
    for (int i = -500; i <= 500; i++) T->e_tab[i + 500] = exp((double)i);            /* 381-382 */
    for (int i = -500; i <= 500; i++) T->e_tab2[i + 500] = exp(i / 10.);             /* 383-384 */
    double prior[25];
    for (int i = 0; i < 25; i++) prior[i] = p_het / 20;                              /* 389-391 */
    prior[0] = prior[6] = prior[12] = prior[18] = prior[24] = (1 - p_het) / 5;
    static const int pidx[15] = { 0, 1, 2, 3, 4, 6, 7, 8, 9, 12, 13, 14, 18, 19, 24 };
    for (int j = 0; j < 15; j++) {                                                   /* 393-407 */
        int hom = (pidx[j] % 6) == 0;
        T->lprior15[j] = hom ? log(prior[pidx[j]]) : log(prior[pidx[j]] * 2);
    }
    double pMM[101], p__[101], p_M[101];
    for (int i = 1; i < 101; i++) {                                                  /* 412-413, 464-466 */
        double prob = 1 - pow(10, -i / 10.0);
        pMM[i] = log(prob / 5);
        p__[i] = log((1 - prob) / 20);
        p_M[i] = log((exp(pMM[i]) + exp(p__[i])) / 2);
        /* STECH_SOLEXA: tech_undercall == 1.00, the *= chain at 470-474 is the identity */
    }
    pMM[0] = pMM[1]; p__[0] = p__[1]; p_M[0] = p_M[1];                               /* 478-480 */
    double q2p[101], mqual_pow[256];
    for (int i = 0; i <= 100; i++) q2p[i] = pow(10, -i / 10.0);                      /* 564-566 */
    for (int i = 0; i < 255; i++) mqual_pow[i] = 1 - pow(10, -(i / 2 + .05) / 10.0); /* 568-572: integer i/2 */
    mqual_pow[255] = mqual_pow[10];                                                  /* 574 */
    for (int q = 0; q < 128; q++) {
        int qq = q > 100 ? 100 : q;
        T->MM[q] = pMM[qq] - p__[qq];                                                /* 644-646 */
        T->_M[q] = p_M[qq] - p__[qq];
        T->q2p[q] = q2p[qq];                                                         /* 649 */
        T->omq2p[q] = 1 - q2p[qq];                                                   /* 651 */
    }
    T->min_e_exp = DBL_MIN_EXP * log(2) + 1;                                         /* 540 */
    T->log_c1 = (double)(-1.0f / 3);                                                 /* 515 */
    T->log_c2 = (double)(2.0f / 3);
    for (int mq = 0; mq < 256; mq++)
        for (int q = 0; q < 256; q++) {                                              /* 632-642 */
            /* the pileup copy is capped before the consensus sees it (cap_quality, 1325-1332): fold it into the table */
            int qc = (q > p->qcap && !p->preserve_qual[q]) ? p->qcap : q;
            if (qc < 0) qc = 0;
            if (qc > 255) qc = 255;
            double _p = mqual_pow[qc], _m = mqual_pow[mq];
            uint8_t e = (uint8_t)(-3.0103 * host_fast_log2(1 - (_m * _p + (1 - _m) / 4), T->log_c1, T->log_c2));
            if (e < 1) e = 1;
            if (e > 100) e = 100;          /* the reference would index past its 101-entry tables here */
            T->effB[(mq << 8) | q] = e;
            T->cellB[(mq << 8) | q] = (uint16_t)(0x8000u | ((unsigned)e << 5) | (mq <= p->min_mqual ? 1u : 0u));   /* CELL_VALID | e << CELL_E_SH | CELL_LOWMQ */
        }
    for (int q = 0; q < 256; q++) { int qc = (q > p->qcap && !p->preserve_qual[q]) ? p->qcap : q; int e = qc < 1 ? 1 : (qc > 100 ? 100 : qc); T->effA[q] = (uint8_t)e; }
    for (int i = 0; i < 256; i++) {                                                  /* init_bins 234-247 */
        int v = i < p->qcutoff ? p->qlow : p->qhigh;
        if (p->preserve_qual[i] > 1) v = i;
        T->bin2[i] = (uint8_t)v;
        T->preserve_qual[i] = p->preserve_qual[i];
    }
}

/* ---- batch builder ----------------------------------------------------------------------- */
void *(*cg_pinned_alloc_hook)(size_t) = NULL;
void (*cg_pinned_free_hook)(void *) = NULL;

extern "C" void *cg_host_alloc(size_t bytes) {
    cg_enable_pinned();                                     /* installs the hooks when a device exists; they stay for the life of the process */
    return cg_pinned_alloc_hook ? cg_pinned_alloc_hook(bytes) : malloc(bytes);
}
extern "C" void cg_host_free(void *p) {
    if (!p) return;
    if (cg_pinned_free_hook) cg_pinned_free_hook(p); else free(p);
}

template <class T> struct vec {
    T *p; size_t n, cap; int pinned;
    void init(int pin) { p = NULL; n = cap = 0; pinned = pin; }
    void release() {
        if (!p) return;
        if (pinned && cg_pinned_free_hook) cg_pinned_free_hook(p); else free(p);
        p = NULL; n = cap = 0;
    }
    int reserve(size_t want) {
        if (want <= cap) return 0;
        size_t nc = cap ? cap + (cap >> 1) : 1024;
        if (nc < want) nc = want;
        T *np;
        if (pinned && cg_pinned_alloc_hook) {
            np = (T *)cg_pinned_alloc_hook(nc * sizeof(T));
            if (!np) return -1;
            if (p) { memcpy(np, p, n * sizeof(T)); cg_pinned_free_hook(p); }
        } else {
            np = (T *)realloc(p, nc * sizeof(T));
            if (!np) return -1;
        }
        p = np; cap = nc;
        return 0;
    }
};

struct cg_batch_builder {
    vec<int32_t> tid, pos, l_qseq, cigar_off; vec<uint16_t> flag, n_cigar; vec<uint8_t> mapq; vec<int64_t> off;
    vec<uint32_t> cigar; vec<uint8_t> seq, qual;
    vec<uint8_t> seq2, qualp; vec<uint64_t> seq_exc;        /* compact planes (cgb_pack) */
    vec<int32_t> pmax;                                      /* running max of pos + span inside the contig */
    vec<uint64_t> tid_runs, pos_abs; vec<uint8_t> pos_d8, lq8, nc8; vec<uint32_t> cigar_x;   /* compact planes of the per-record arrays (cgb_pack) */
    int have_meta; int32_t lq_dict[256];
    int have_pack, qual_bits; uint8_t qual_dict[16];
    int64_t last_key; int unsorted; int seen_unplaced;
};

extern "C" cg_batch_builder *cgb_create(int pinned) {
    cg_batch_builder *b = (cg_batch_builder *)calloc(1, sizeof(*b));
    if (!b) return NULL;
    if (pinned) cg_enable_pinned();
    int pin = pinned && cg_pinned_alloc_hook;
    b->tid.init(pin); b->pos.init(pin); b->l_qseq.init(pin); b->cigar_off.init(pin); b->flag.init(pin); b->n_cigar.init(pin);
    b->mapq.init(pin); b->off.init(pin); b->cigar.init(pin); b->seq.init(pin); b->qual.init(pin);
    b->seq2.init(pin); b->qualp.init(pin); b->seq_exc.init(pin); b->pmax.init(0);
    b->tid_runs.init(pin); b->pos_abs.init(pin); b->pos_d8.init(pin); b->lq8.init(pin); b->nc8.init(pin); b->cigar_x.init(pin);
    b->last_key = INT64_MIN;
    return b;
}
extern "C" void cgb_reset(cg_batch_builder *b) {
    b->tid.n = b->pos.n = b->l_qseq.n = b->cigar_off.n = b->flag.n = b->n_cigar.n = b->mapq.n = b->off.n = 0;
    b->cigar.n = b->seq.n = b->qual.n = 0;
    b->seq2.n = b->qualp.n = b->seq_exc.n = 0; b->have_pack = 0; b->qual_bits = 0; b->pmax.n = 0;
    b->tid_runs.n = b->pos_abs.n = b->pos_d8.n = b->lq8.n = b->nc8.n = b->cigar_x.n = 0; b->have_meta = 0;
    b->last_key = INT64_MIN; b->unsorted = 0; b->seen_unplaced = 0;
}
extern "C" void cgb_destroy(cg_batch_builder *b) {
    if (!b) return;
    b->tid.release(); b->pos.release(); b->l_qseq.release(); b->cigar_off.release(); b->flag.release(); b->n_cigar.release();
    b->mapq.release(); b->off.release(); b->cigar.release(); b->seq.release(); b->qual.release();
    b->seq2.release(); b->qualp.release(); b->seq_exc.release(); b->pmax.release();
    b->tid_runs.release(); b->pos_abs.release(); b->pos_d8.release(); b->lq8.release(); b->nc8.release(); b->cigar_x.release();
    free(b);
}

extern "C" int cgb_add(cg_batch_builder *b, int32_t tid, int32_t pos, uint16_t flag, uint8_t mapq, int32_t l_qseq,
                       uint32_t n_cigar, const uint32_t *cigar, const uint8_t *seq4, const uint8_t *qual) {
    size_t i = b->tid.n;
    if (n_cigar > 65535 || l_qseq < 0) return CG_ERR_BAD_ARG;
    b->have_pack = 0; b->have_meta = 0;
    if (b->tid.reserve(i + 1) || b->pos.reserve(i + 1) || b->l_qseq.reserve(i + 1) || b->cigar_off.reserve(i + 1) ||
        b->flag.reserve(i + 1) || b->n_cigar.reserve(i + 1) || b->mapq.reserve(i + 1) || b->off.reserve(i + 1)) return CG_ERR_NOMEM;
    /* quality bytes padded to 8 so that off is 8-aligned and seq sits at off/2 */
    size_t qoff = b->qual.n, qpad = ((size_t)l_qseq + 7) & ~(size_t)7;
    if (b->qual.reserve(qoff + qpad + 8) || b->seq.reserve((qoff + qpad) / 2 + 8) || b->cigar.reserve(b->cigar.n + n_cigar + 1)) return CG_ERR_NOMEM;
    memcpy(b->qual.p + qoff, qual, (size_t)l_qseq);
    memset(b->qual.p + qoff + l_qseq, 0, qpad - (size_t)l_qseq);
    size_t sbytes = ((size_t)l_qseq + 1) >> 1;
    memcpy(b->seq.p + qoff / 2, seq4, sbytes);
    memset(b->seq.p + qoff / 2 + sbytes, 0, qpad / 2 - sbytes);
    memcpy(b->cigar.p + b->cigar.n, cigar, 4u * (size_t)n_cigar);
    b->tid.p[i] = tid; b->pos.p[i] = pos; b->flag.p[i] = flag; b->mapq.p[i] = mapq; b->l_qseq.p[i] = l_qseq;
    b->n_cigar.p[i] = (uint16_t)n_cigar; b->off.p[i] = (int64_t)qoff; b->cigar_off.p[i] = (int32_t)b->cigar.n;
    b->qual.n = qoff + qpad; b->seq.n = (qoff + qpad) / 2; b->cigar.n += n_cigar;
    b->tid.n = b->pos.n = b->l_qseq.n = b->cigar_off.n = b->flag.n = b->n_cigar.n = b->mapq.n = b->off.n = i + 1;
    {   /* running max of the record ends inside the contig (cg_batch.pmax_end) */
        if (b->pmax.reserve(i + 1)) return CG_ERR_NOMEM;
        const int32_t e = pos + cg_pileup_span(tid, flag, cigar, (int)n_cigar);
        b->pmax.p[i] = (i > 0 && b->tid.p[i - 1] == tid && b->pmax.p[i - 1] > e) ? b->pmax.p[i - 1] : e;
        b->pmax.n = i + 1;
    }
    /* sortedness of what enters the pileup (htslib's pileup aborts on unsorted input) */
    if (tid >= 0 && !(flag & 4)) {
        int64_t key = cg_key(tid, pos);
        if (key < b->last_key || b->seen_unplaced) b->unsorted = 1;
        b->last_key = key;
    } else if (tid < 0) b->seen_unplaced = 1;
    return 0;
}

/* size the (pinned) arrays once: growing a pinned allocation means a new cudaHostAlloc and a copy */
extern "C" int cgb_reserve(cg_batch_builder *b, int64_t n_reads, int64_t qual_bytes, int64_t n_cigar) {
    if (n_reads < 0 || qual_bytes < 0 || n_cigar < 0) return CG_ERR_BAD_ARG;
    size_t i = (size_t)n_reads, q = (size_t)qual_bytes + 8 * (size_t)n_reads + 16;
    if (b->tid.reserve(i) || b->pos.reserve(i) || b->l_qseq.reserve(i) || b->cigar_off.reserve(i) || b->flag.reserve(i) ||
        b->n_cigar.reserve(i) || b->mapq.reserve(i) || b->off.reserve(i) || b->qual.reserve(q) || b->seq.reserve(q / 2 + 16) ||
        b->cigar.reserve((size_t)n_cigar + 2)) return CG_ERR_NOMEM;
    return 0;
}

extern "C" int cgb_add_bam_stream(cg_batch_builder *b, const uint8_t *buf, size_t len) {
    if (len < 12 || memcmp(buf, "BAM\1", 4)) return CG_ERR_BAD_ARG;
    size_t p = 4; uint32_t lt, nref;
    memcpy(&lt, buf + p, 4); p += 4 + lt;
    if (p + 4 > len) return CG_ERR_BAD_ARG;
    memcpy(&nref, buf + p, 4); p += 4;
    for (uint32_t i = 0; i < nref; i++) { uint32_t ln; if (p + 4 > len) return CG_ERR_BAD_ARG; memcpy(&ln, buf + p, 4); p += 4 + ln + 4; }
    {   /* size everything once (pinned allocations are expensive to grow) */
        size_t q = p, nrec = 0, qb = 0, nc = 0;
        while (q + 4 <= len) {
            uint32_t bs; memcpy(&bs, buf + q, 4);
            if (bs < 32 || q + 4 + bs > len) return CG_ERR_BAD_ARG;
            int32_t lseq; uint16_t ncig; memcpy(&lseq, buf + q + 4 + 16, 4); memcpy(&ncig, buf + q + 4 + 12, 2);
            if (lseq < 0) return CG_ERR_BAD_ARG;
            nrec++; qb += ((size_t)lseq + 7) & ~(size_t)7; nc += ncig;
            q += 4 + bs;
        }
        size_t i = b->tid.n + nrec;
        if (b->tid.reserve(i) || b->pos.reserve(i) || b->l_qseq.reserve(i) || b->cigar_off.reserve(i) || b->flag.reserve(i) ||
            b->n_cigar.reserve(i) || b->mapq.reserve(i) || b->off.reserve(i) || b->qual.reserve(b->qual.n + qb + 16) ||
            b->seq.reserve((b->qual.n + qb) / 2 + 16) || b->cigar.reserve(b->cigar.n + nc + 2)) return CG_ERR_NOMEM;
    }
    while (p + 4 <= len) {
        uint32_t bs; memcpy(&bs, buf + p, 4);
        if (bs < 32 || p + 4 + bs > len) return CG_ERR_BAD_ARG;
        const uint8_t *r = buf + p + 4;
        int32_t tid, pos, lseq; memcpy(&tid, r, 4); memcpy(&pos, r + 4, 4); memcpy(&lseq, r + 16, 4);
        uint8_t lname = r[8], mapq = r[9];
        uint16_t ncig, flag; memcpy(&ncig, r + 12, 2); memcpy(&flag, r + 14, 2);
        const uint8_t *cig = r + 32 + lname;
        const uint8_t *seq = cig + 4u * ncig;
        const uint8_t *qual = seq + ((lseq + 1) >> 1);
        if ((size_t)(qual + lseq - r) > bs) return CG_ERR_BAD_ARG;
        uint32_t cigbuf[64], *cg = cigbuf;
        if (ncig > 64) cg = (uint32_t *)malloc(4u * ncig);
        memcpy(cg, cig, 4u * ncig);                 /* records are not 4-byte aligned in the stream */
        int e = cgb_add(b, tid, pos, flag, mapq, lseq, ncig, cg, seq, qual);
        if (cg != cigbuf) free(cg);
        if (e) return e;
        p += 4 + bs;
    }
    return 0;
}

extern "C" int cgb_finish(cg_batch_builder *b, cg_batch *o) {
    if (b->unsorted) return CG_ERR_UNSORTED;
    memset(o, 0, sizeof(*o));
    o->n_reads = (int64_t)b->tid.n;
    o->tid = b->tid.p; o->pos = b->pos.p; o->flag = b->flag.p; o->mapq = b->mapq.p; o->l_qseq = b->l_qseq.p;
    o->n_cigar = b->n_cigar.p; o->off = b->off.p; o->cigar_off = b->cigar_off.p;
    o->cigar = b->cigar.p; o->n_cigar_total = (int64_t)b->cigar.n;
    o->seq = b->seq.p; o->seq_bytes = (int64_t)b->seq.n;
    o->qual = b->qual.p; o->qual_bytes = (int64_t)b->qual.n;
    o->packed = 1;                                   /* cgb_add lays records out back to back */
    o->pmax_end = b->pmax.p;
    if (b->have_pack) {
        o->seq2 = b->seq2.p; o->seq2_bytes = (int64_t)b->seq2.n;
        o->seq_exc = b->seq_exc.p; o->n_seq_exc = (int64_t)b->seq_exc.n;
        o->qual_bits = b->qual_bits;
        if (b->qual_bits) { o->qualp = b->qualp.p; o->qualp_bytes = (int64_t)b->qualp.n; memcpy(o->qual_dict, b->qual_dict, 16); }
    }
    if (b->have_meta) {
        o->meta_planes = 1;
        o->tid_runs = b->tid_runs.p; o->n_tid_runs = (int64_t)b->tid_runs.n;
        o->pos_d8 = b->pos_d8.p; o->pos_abs = b->pos_abs.p; o->n_pos_abs = (int64_t)b->pos_abs.n;
        o->lq8 = b->lq8.p; memcpy(o->lq_dict, b->lq_dict, sizeof b->lq_dict);
        o->nc8 = b->nc8.p; o->cigar_x = b->cigar_x.p; o->n_cigar_x = (int64_t)b->cigar_x.n;
    }
    return 0;
}

/* ---- compact planes -------------------------------------------------------------------------
 * Workers own contiguous ranges of RECORDS; a range's positions are a contiguous, 8-aligned range of the quality buffer, so the
 * planes are written without overlap (8 positions = 2 bytes of seq2, 2 or 4 bytes of qualp).  Exceptions are collected per worker
 * and concatenated in worker order, which is position order. */
struct pack_job {
    cg_batch_builder *b; size_t r0, r1; int pass; int bits; const uint8_t *code;     /* code[value] -> dictionary code */
    uint64_t seen[4]; uint64_t *exc; size_t n_exc, cap_exc; int err;
};
static void *pack_worker(void *v) {
    pack_job *J = (pack_job *)v;
    cg_batch_builder *b = J->b;
    if (J->pass == 0) {                                  /* which quality values occur (real bases only, not the padding) */
        for (size_t r = J->r0; r < J->r1; r++) {
            const uint8_t *q = b->qual.p + b->off.p[r]; const int l = b->l_qseq.p[r];
            for (int x = 0; x < l; x++) J->seen[q[x] >> 6] |= 1ULL << (q[x] & 63);
        }
        return NULL;
    }
    static const uint8_t n2[16] = { 0xff, 0, 1, 0xff, 2, 0xff, 0xff, 0xff, 3, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff };   /* nt16 -> 2 bit */
    for (size_t r = J->r0; r < J->r1; r++) {
        const size_t o = (size_t)b->off.p[r]; const int l = b->l_qseq.p[r], lp = (l + 7) & ~7;
        const uint8_t *q = b->qual.p + o, *s4 = b->seq.p + o / 2;
        uint8_t *s2 = b->seq2.p + o / 4;
        for (int x = 0; x < lp; x += 4) {
            unsigned byte = 0;
            for (int k = 0; k < 4; k++) {
                const int xx = x + k;
                if (xx >= l) continue;                   /* padding: A */
                const unsigned nib = (s4[xx >> 1] >> ((~xx & 1) << 2)) & 0xf;
                unsigned c = n2[nib];
                if (c == 0xff) {
                    c = 0;
                    if (J->n_exc == J->cap_exc) {
                        size_t nc = J->cap_exc ? J->cap_exc * 2 : 1024;
                        uint64_t *ne = (uint64_t *)realloc(J->exc, nc * 8);
                        if (!ne) { J->err = 1; return NULL; }
                        J->exc = ne; J->cap_exc = nc;
                    }
                    J->exc[J->n_exc++] = ((uint64_t)(o + (size_t)xx) << 4) | nib;
                }
                byte |= c << (2 * k);
            }
            s2[x >> 2] = (uint8_t)byte;
        }
        if (J->bits == 2) {
            uint8_t *qp = b->qualp.p + o / 4;
            for (int x = 0; x < lp; x += 4) {
                unsigned byte = 0;
                for (int k = 0; k < 4; k++) if (x + k < l) byte |= (unsigned)J->code[q[x + k]] << (2 * k);
                qp[x >> 2] = (uint8_t)byte;
            }
        } else if (J->bits == 4) {
            uint8_t *qp = b->qualp.p + o / 2;
            for (int x = 0; x < lp; x += 2) {
                unsigned byte = 0;
                if (x < l) byte |= J->code[q[x]];
                if (x + 1 < l) byte |= (unsigned)J->code[q[x + 1]] << 4;
                qp[x >> 1] = (uint8_t)byte;
            }
        }
    }
    return NULL;
}

/* compact planes of the per-record arrays (cg_batch.meta_planes); 0 = built, 1 = this batch does not qualify (the plain arrays travel) */
static int pack_meta(cg_batch_builder *b) {
    const size_t n = b->tid.n;
    b->have_meta = 0;
    b->tid_runs.n = b->pos_abs.n = b->cigar_x.n = 0;
    if (n == 0 || n >= (1ULL << 31)) return 1;
    if (b->pos_d8.reserve(n) || b->lq8.reserve(n) || b->nc8.reserve(n)) return CG_ERR_NOMEM;
    int nd = 0; memset(b->lq_dict, 0, sizeof b->lq_dict);
    int last_code = -1; int32_t last_lq = -1;
    for (size_t i = 0; i < n; i++) {
        const int32_t tid = b->tid.p[i], pos = b->pos.p[i], lq = b->l_qseq.p[i];
        const uint32_t nc = b->n_cigar.p[i];
        if (i == 0 || tid != b->tid.p[i - 1]) {
            if (b->tid_runs.reserve(b->tid_runs.n + 1)) return CG_ERR_NOMEM;
            b->tid_runs.p[b->tid_runs.n++] = ((uint64_t)i << 32) | (uint32_t)tid;
        }
        const int64_t d = i ? (int64_t)pos - b->pos.p[i - 1] : -1;
        if (i == 0 || tid != b->tid.p[i - 1] || d < 0 || d > 254) {
            if (b->pos_abs.reserve(b->pos_abs.n + 1)) return CG_ERR_NOMEM;
            b->pos_abs.p[b->pos_abs.n++] = ((uint64_t)i << 32) | (uint32_t)pos;
            b->pos_d8.p[i] = 255;
        } else b->pos_d8.p[i] = (uint8_t)d;
        if (lq != last_lq) {
            int c = 0;
            while (c < nd && b->lq_dict[c] != lq) c++;
            if (c == nd) { if (nd == 256) return 1; b->lq_dict[nd++] = lq; }
            last_code = c; last_lq = lq;
        }
        b->lq8.p[i] = (uint8_t)last_code;
        if (nc > 254) return 1;
        const uint32_t *cg = b->cigar.p + b->cigar_off.p[i];
        if (nc == 1 && cg[0] == ((uint32_t)lq << 4)) b->nc8.p[i] = 255;                 /* one M of l_qseq bases: implied */
        else {
            b->nc8.p[i] = (uint8_t)nc;
            if (b->cigar_x.reserve(b->cigar_x.n + nc + 1)) return CG_ERR_NOMEM;
            memcpy(b->cigar_x.p + b->cigar_x.n, cg, 4u * (size_t)nc); b->cigar_x.n += nc;
        }
    }
    if (b->pos_abs.n > n / 8 + 64 || b->tid_runs.n > n / 8 + 64) return 1;              /* not a coordinate-sorted stream: the per-record searches would cost more than the bytes saved */
    b->pos_d8.n = b->lq8.n = b->nc8.n = n;
    b->have_meta = 1;
    return 0;
}

extern "C" int cgb_pack(cg_batch_builder *b, int threads) {
    const size_t n = b->tid.n;
    b->have_pack = 0; b->qual_bits = 0;
    { const int me = pack_meta(b); if (me < 0) return me; }
    if (threads <= 0) threads = (int)sysconf(_SC_NPROCESSORS_ONLN);
    if (threads < 1) threads = 1;
    if (threads > 64) threads = 64;
    if ((size_t)threads > n) threads = n ? (int)n : 1;
    if (b->seq2.reserve(b->qual.n / 4 + 16) || b->qualp.reserve(b->qual.n / 2 + 16)) return CG_ERR_NOMEM;
    pack_job jobs[64]; pthread_t th[64];
    uint8_t code[256]; memset(code, 0, sizeof code);
    int bits = 0;
    for (int pass = 0; pass < 2; pass++) {
        for (int t = 0; t < threads; t++) {
            pack_job *J = &jobs[t];
            if (pass == 0) { memset(J, 0, sizeof *J); J->b = b; J->r0 = n * (size_t)t / (size_t)threads; J->r1 = n * (size_t)(t + 1) / (size_t)threads; }
            J->pass = pass; J->bits = bits; J->code = code;
            if (pthread_create(&th[t], NULL, pack_worker, J) != 0) { pack_worker(J); th[t] = 0; }
        }
        for (int t = 0; t < threads; t++) if (th[t]) pthread_join(th[t], NULL);
        if (pass == 0) {
            uint64_t seen[4] = { 0, 0, 0, 0 };
            for (int t = 0; t < threads; t++) for (int k = 0; k < 4; k++) seen[k] |= jobs[t].seen[k];
            int nv = 0; uint8_t dict[256];
            for (int v = 0; v < 256; v++) if (seen[v >> 6] >> (v & 63) & 1) dict[nv++] = (uint8_t)v;
            bits = nv <= 4 ? 2 : (nv <= 16 ? 4 : 0);
            memset(b->qual_dict, 0, 16);
            if (bits) for (int k = 0; k < nv; k++) { b->qual_dict[k] = dict[k]; code[dict[k]] = (uint8_t)k; }
        }
    }
    size_t ne = 0; int err = 0;
    for (int t = 0; t < threads; t++) { ne += jobs[t].n_exc; err |= jobs[t].err; }
    if (err || b->seq_exc.reserve(ne + 1)) { for (int t = 0; t < threads; t++) free(jobs[t].exc); return CG_ERR_NOMEM; }
    ne = 0;
    for (int t = 0; t < threads; t++) { if (jobs[t].n_exc) memcpy(b->seq_exc.p + ne, jobs[t].exc, jobs[t].n_exc * 8); ne += jobs[t].n_exc; free(jobs[t].exc); }
    b->seq_exc.n = ne;
    b->seq2.n = b->qual.n / 4;
    b->qual_bits = bits;
    b->qualp.n = bits == 2 ? b->qual.n / 4 : (bits == 4 ? b->qual.n / 2 : 0);
    b->have_pack = 1;
    return 0;
}

extern "C" int64_t cgb_bytes(const cg_batch_builder *b) {
    return (int64_t)(b->tid.n * (4 + 4 + 4 + 4 + 2 + 2 + 1 + 8) + b->cigar.n * 4 + b->seq.n + b->qual.n);
}

extern "C" int32_t cg_record_end(int32_t tid, int32_t pos, uint16_t flag, const uint32_t *cigar, int n_cigar) {
    return pos + cg_pileup_span(tid, flag, cigar, n_cigar);
}
static int batch_span(const cg_batch *in, int64_t i) {
    return cg_pileup_span(in->tid[i], in->flag[i], in->cigar + in->cigar_off[i], in->n_cigar[i]);
}
extern "C" void cg_batch_ends(const cg_batch *in, int32_t *end_out) {
    for (int64_t i = 0; i < in->n_reads; i++) end_out[i] = in->pos[i] + batch_span(in, i);
}
extern "C" int64_t cg_algorithmic_bytes(const cg_batch *in) {           /* SURVEY.md §8(d) */
    int64_t s = 0;
    for (int64_t i = 0; i < in->n_reads; i++)
        if (batch_span(in, i)) { int64_t l = in->l_qseq[i]; s += ((l + 1) >> 1) + 2 * l + 4 * (int64_t)in->n_cigar[i] + 16; }
    return s;
}
extern "C" int64_t cg_aligned_bases(const cg_batch *in) {
    int64_t s = 0;
    for (int64_t i = 0; i < in->n_reads; i++) if (batch_span(in, i)) s += in->l_qseq[i];
    return s;
}
