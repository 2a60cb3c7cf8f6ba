/*
 * transcode_gpu.c — host driver with the reference's transcode() contract
 * (snp_score.c:1336-2029): read records, hand them to the device path through the C ABI
 * of include/crumble_gpu.h, write them back in input order with rewritten qualities.
 *
 * What stays on the host, as in the reference: record I/O, the BED text lines
 * (snp_score.c:1496-1498 etc.), the -v counters, the read-count check (2021-2026).
 * Everything between "record decoded" and "record ready to write" runs on the GPU.
 *
 * The stream is processed in bounded memory as a CHAIN of device calls (cg_process_window): the host cuts the
 * coordinate-sorted input every CRUMBLE_BATCH_READS records (default 512 Ki), keeps the reads that straddle a cut
 * as the next call's halo, and writes records out in input order as they become final.  The reference does the same
 * thing with its streaming loop and the two RB-trees of in-flight reads (snp_score.c:1113-1153, 1926-1975); here the
 * unit is a region shard instead of a column.  With -r the region is one call (cg_process).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <inttypes.h>
#include <limits.h>
#include <pthread.h>
#include <time.h>
#include "htslib/sam.h"
#include "crumble_host.h"

/* ---- record queues: a reader thread decodes ahead of the device, a writer thread encodes behind it ---------------- */
#define RQ_CHUNK 4096
#define RQ_SLOTS 256                                         /* <= 1 Mi records queued on either side */
typedef struct { bam1_t **v; int n; } rchunk;
typedef struct {
    pthread_mutex_t mu; pthread_cond_t cv;
    rchunk ring[RQ_SLOTS]; int head, count, closed, status;  /* status < 0: the producer / consumer failed */
} recq;

static void rq_init(recq *q) { memset(q, 0, sizeof *q); pthread_mutex_init(&q->mu, NULL); pthread_cond_init(&q->cv, NULL); }
static int rq_put(recq *q, rchunk c) {                       /* blocks while full; -1 if the other side has failed */
    pthread_mutex_lock(&q->mu);
    while (q->count == RQ_SLOTS && q->status >= 0) pthread_cond_wait(&q->cv, &q->mu);
    int st = q->status;
    if (st >= 0) { q->ring[(q->head + q->count) % RQ_SLOTS] = c; q->count++; pthread_cond_broadcast(&q->cv); }
    pthread_mutex_unlock(&q->mu);
    return st < 0 ? -1 : 0;
}
static int rq_get(recq *q, rchunk *c) {                      /* 1 = chunk, 0 = closed and drained */
    pthread_mutex_lock(&q->mu);
    while (q->count == 0 && !q->closed) pthread_cond_wait(&q->cv, &q->mu);
    int got = 0;
    if (q->count) { *c = q->ring[q->head]; q->head = (q->head + 1) % RQ_SLOTS; q->count--; got = 1; pthread_cond_broadcast(&q->cv); }
    pthread_mutex_unlock(&q->mu);
    return got;
}
static void rq_close(recq *q, int status) {
    pthread_mutex_lock(&q->mu);
    q->closed = 1; if (status < 0) q->status = status;
    pthread_cond_broadcast(&q->cv);
    pthread_mutex_unlock(&q->mu);
}
static void rq_fail(recq *q) { pthread_mutex_lock(&q->mu); q->status = -1; pthread_cond_broadcast(&q->cv); pthread_mutex_unlock(&q->mu); }

typedef struct { recq q; samFile *fp; bam_hdr_t *header; hts_itr_t *itr; crumble_opts *o; } io_thread;

static void *reader_main(void *v) {
    io_thread *t = (io_thread *)v;
    int status = 0;
    for (;;) {
        rchunk c; c.n = 0; c.v = (bam1_t **)malloc(sizeof(bam1_t *) * RQ_CHUNK);
        if (!c.v) { status = -1; break; }
        int r = 0;
        while (c.n < RQ_CHUNK) {
            bam1_t *b = bam_init1();
            r = t->itr ? sam_itr_next(t->fp, t->itr, b) : sam_read1(t->fp, t->header, b);
            if (r < 0) { bam_destroy1(b); break; }
            c.v[c.n++] = b;
        }
        if (c.n) { if (rq_put(&t->q, c) < 0) { for (int i = 0; i < c.n; i++) bam_destroy1(c.v[i]); free(c.v); break; } }
        else free(c.v);
        if (r < -1) { fprintf(stderr, "Error reading input\n"); status = -1; }
        if (r < 0) break;
    }
    rq_close(&t->q, status);
    return NULL;
}
static void *writer_main(void *v) {
    io_thread *t = (io_thread *)v;
    rchunk c;
    int bad = 0;
    while (rq_get(&t->q, &c)) {
        for (int i = 0; i < c.n; i++) {
            if (!bad) {
                crumble_purge_tags(t->o, c.v[i]);                               /* snp_score.c:1088 */
                if (sam_write1(t->fp, t->header, c.v[i]) < 0) { bad = 1; rq_fail(&t->q); }
            }
            bam_destroy1(c.v[i]);
        }
        free(c.v);
    }
    return NULL;
}

/* one record in flight: read but not yet written, or written but still part of a later call's halo */
typedef struct {
    bam1_t  *b;             /* NULL once written and destroyed (then oq/meta below serve the halo) */
    uint8_t *oq;            /* original qualities, saved when the record turns final while later calls still need it */
    int32_t  end;           /* cg_record_end: pos + pileup span, pos itself outside the pileup */
    uint8_t  final, is_new;
    int64_t  slot;          /* index in the current batch, -1 when not part of it */
} live_rec;

typedef struct { live_rec *v; size_t n, cap, head; } live_q;

static int lq_push(live_q *q, bam1_t *b) {
    if (q->n == q->cap) {
        if (q->head > 0) {                                  /* drop the written prefix */
            memmove(q->v, q->v + q->head, (q->n - q->head) * sizeof(*q->v));
            q->n -= q->head; q->head = 0;
        }
        if (q->n == q->cap) {
            size_t nc = q->cap ? q->cap * 2 : 4096;
            live_rec *nv = (live_rec *)realloc(q->v, nc * sizeof(*nv));
            if (!nv) return -1;
            q->v = nv; q->cap = nc;
        }
    }
    live_rec *r = &q->v[q->n++];
    memset(r, 0, sizeof(*r));
    r->b = b; r->is_new = 1; r->slot = -1;
    r->end = cg_record_end(b->core.tid, b->core.pos, b->core.flag, bam_get_cigar(b), (int)b->core.n_cigar);
    return 0;
}

/* r is open at the cut (tid, limit): a pileup record (end > pos) on contig tid that ends beyond limit.  With limit = the cut's
 * position the record is not final yet; with limit = S it belongs to the next call's read halo. */
static int reaches(const live_rec *r, int32_t tid, int32_t limit) {
    return r->b->core.tid == tid && r->end > r->b->core.pos && r->end > limit;
}

static void lq_free(live_q *q) {
    for (size_t i = q->head; i < q->n; i++) { if (q->v[i].b) bam_destroy1(q->v[i].b); free(q->v[i].oq); }
    free(q->v);
}

static void write_bed(crumble_opts *o, bam_hdr_t *header, const cg_result *res) {
    /* BED lines, in column order (snp_score.c:1496-1498,1676-1678,1768-1770,1802-1804,1810-1812) */
    static const char *tag[5] = { "VDEEP", "DEEP", "CLIP", "INDEL_LEN", "INDEL_COVERAGE" };
    if (!o->bed_fp) return;
    for (int64_t i = 0; i < res->n_events; i++) {
        const cg_bed_event *e = &res->events[i];
        int s = e->pos - 50; if (s < 0) s = 0;
        fprintf(o->bed_fp, "%s\t%d\t%d\t%s\n", header->target_name[e->tid], s, e->pos + 50, tag[e->tag]);
    }
}

static int grow_result(cg_result *res, int64_t *qcap, int64_t qual_bytes) {
    if (qual_bytes + 16 > *qcap) {                           /* page-locked: the download of a slice overlaps the kernels of the next (nothing to keep from the last call) */
        int64_t nc = qual_bytes + (qual_bytes >> 2) + 4096;
        cg_host_free(res->qual_out); res->qual_out = NULL; *qcap = 0;
        uint8_t *nq = (uint8_t *)cg_host_alloc((size_t)nc);
        if (!nq) return -1;
        res->qual_out = nq; *qcap = nc;
    }
    return 0;
}

int transcode_gpu(crumble_opts *o, samFile *in, samFile *out, bam_hdr_t *header, hts_itr_t *h_iter) {
    int ret = -1, err = 0;
    live_q lq = {0};
    cg_batch_builder *bb = NULL;
    cg_ctx *ctx = NULL;
    cg_multi *mg = NULL;                                    /* CRUMBLE_GPUS > 1: every call of the chain is spread over the GPUs of the box (cg_multi.c) */
    cg_result res; memset(&res, 0, sizeof(res));
    int64_t qcap = 0;
    int64_t count_in = 0, count_out = 0;
    bam1_t *nx = NULL;                                      /* the record after the current cut */
    float device_ms = 0;
    io_thread rd, wr; pthread_t rd_th, wr_th; int rd_on = 0, wr_on = 0;
    struct timespec t_0, t_1; clock_gettime(CLOCK_MONOTONIC, &t_0);
    double t_gather = 0, t_build = 0, t_dev = 0, t_out = 0; int64_t n_calls = 0, n_halo = 0;
#define TICK() (clock_gettime(CLOCK_MONOTONIC, &t_1), (t_1.tv_sec - t_0.tv_sec) + 1e-9 * (t_1.tv_nsec - t_0.tv_nsec))
    rchunk rc = { NULL, 0 }; int rc_i = 0;                  /* chunk being consumed from the reader */
    rchunk wc = { NULL, 0 };                                /* chunk being filled for the writer */

    cg_params p = o->p;
    if (h_iter) { p.region_tid = h_iter->tid; p.region_beg = h_iter->beg; p.region_end = h_iter->end; }
    int64_t batch_reads = 512 << 10;
    const char *ev = getenv("CRUMBLE_BATCH_READS");
    if (ev && atoll(ev) > 0) batch_reads = atoll(ev);
    int n_gpus = 1;
    if (getenv("CRUMBLE_GPUS") && atoi(getenv("CRUMBLE_GPUS")) > 1 && !h_iter) {
        n_gpus = atoi(getenv("CRUMBLE_GPUS"));
        if (n_gpus > cg_device_count()) n_gpus = cg_device_count();
        if (n_gpus < 1) n_gpus = 1;
        if (!(ev && atoll(ev) > 0)) batch_reads *= n_gpus;  /* one shard of the usual size per device */
    }
    if (h_iter) batch_reads = INT64_MAX;                    /* a -r region is one call: the region logic owns the column limits */

    if (!(bb = cgb_create(1))) goto done;
    {   /* pre-size the pinned arrays for one shard (capped: a huge CRUMBLE_BATCH_READS just grows them on demand) */
        const int64_t rsv = (batch_reads < (4 << 20) ? batch_reads : (4 << 20)) + 4096;
        if (!h_iter && cgb_reserve(bb, rsv, rsv * 160, rsv * 2) != 0) goto done;
    }
    if (n_gpus > 1) {
        mg = cgm_create(&p, n_gpus, NULL, &err);
        if (!mg) { fprintf(stderr, "crumble: cannot create %d GPU contexts: %s\n", n_gpus, cg_strerror(err)); goto done; }
    } else {
        ctx = cg_create(&p, o->device, &err);
        if (!ctx) { fprintf(stderr, "crumble: cannot create GPU context: %s\n", cg_strerror(err)); goto done; }
    }
    res.events_cap = 1 << 16;
    if (getenv("CRUMBLE_EVENTS_CAP") && atoll(getenv("CRUMBLE_EVENTS_CAP")) > 0) res.events_cap = atoll(getenv("CRUMBLE_EVENTS_CAP"));   /* tests: force the regrow path */
    res.events = (cg_bed_event *)malloc(sizeof(cg_bed_event) * (size_t)res.events_cap);
    if (!res.events) goto done;

    rq_init(&rd.q); rd.fp = in; rd.header = header; rd.itr = h_iter; rd.o = o;
    rq_init(&wr.q); wr.fp = out; wr.header = header; wr.itr = NULL; wr.o = o;
    if (pthread_create(&rd_th, NULL, reader_main, &rd) != 0) goto done;
    rd_on = 1;
    if (pthread_create(&wr_th, NULL, writer_main, &wr) != 0) goto done;
    wr_on = 1;

    int eof = 0, first = 1;
    int32_t lo_tid = -1, lo_pos = 0, cnt_pos = 0;
    int64_t last_key = INT64_MIN; int seen_unplaced = 0;
    while (!eof || nx || lq.head < lq.n) {
        /* ---- gather the new records of this call ---- */
        double tk0 = TICK();
        int64_t n_new = 0;
        int32_t last_tid = -2;
        for (;;) {
            if (!nx && !eof) {
                if (rc_i >= rc.n) { free(rc.v); rc.v = NULL; rc.n = rc_i = 0; if (!rq_get(&rd.q, &rc)) { rc.v = NULL; rc.n = 0; } }
                if (rc_i < rc.n) nx = rc.v[rc_i++];
                else { eof = 1; if (rd.q.status < 0) goto done; }
                if (nx) {
                    count_in++;
                    if (nx->core.tid >= 0 && !(nx->core.flag & BAM_FUNMAP)) {       /* sortedness across calls (cgb_add checks inside one) */
                        int64_t key = ((int64_t)nx->core.tid << 32) | (uint32_t)nx->core.pos;
                        if (key < last_key || seen_unplaced) { fprintf(stderr, "crumble: %s\n", cg_strerror(CG_ERR_UNSORTED)); goto done; }
                        last_key = key;
                    } else if (nx->core.tid < 0) seen_unplaced = 1;
                }
            }
            if (!nx) break;
            if (n_new >= batch_reads) break;
            if (lq_push(&lq, nx) < 0) goto done;
            last_tid = nx->core.tid;
            nx = NULL; n_new++;
        }
        if (n_new == 0) break;
        double tk1 = TICK(); t_gather += tk1 - tk0;

        /* ---- this call's column window ---- */
        cg_window win; memset(&win, 0, sizeof win);
        win.first = first; win.lo_tid = lo_tid; win.lo_pos = lo_pos; win.cnt_pos = cnt_pos; win.hi_tid = -1;
        if (nx && nx->core.tid >= 0 && nx->core.tid == last_tid) { win.hi_tid = nx->core.tid; win.hi_pos = nx->core.pos; }
        /* ---- the batch: halo (earlier records of lo_tid that reach beyond lo_pos) + new records, in input order ---- */
        cgb_reset(bb);
        int64_t nb = 0;
        int32_t S = win.hi_pos;
        for (size_t i = lq.head; i < lq.n; i++) {
            live_rec *r = &lq.v[i];
            r->slot = -1;
            if (!r->is_new && !(r->b && !first && reaches(r, lo_tid, lo_pos))) continue;
            const bam1_t *b = r->b;
            int e = cgb_add(bb, b->core.tid, b->core.pos, b->core.flag, b->core.qual, b->core.l_qseq, b->core.n_cigar,
                            bam_get_cigar(b), bam_get_seq(b), r->oq ? r->oq : bam_get_qual(b));
            if (e) { fprintf(stderr, "crumble: %s\n", cg_strerror(e)); goto done; }
            r->slot = nb++;
            if (reaches(r, win.hi_tid, win.hi_pos) && b->core.pos < S) S = b->core.pos;
        }
        win.next_lo_pos = S;
        cg_batch batch;
        if ((err = cgb_finish(bb, &batch)) != 0) { fprintf(stderr, "crumble: %s\n", cg_strerror(err)); goto done; }
        if (grow_result(&res, &qcap, batch.qual_bytes) < 0) goto done;

        double tk2 = TICK(); t_build += tk2 - tk1; n_calls++; n_halo += nb - n_new;
        /* ---- device ---- */
        if (h_iter) {
            for (;;) {
                err = cg_process(ctx, &batch, &res);
                if (err == CG_OK && res.n_events > res.events_cap) {            /* event buffer too small: grow and redo */
                    res.events_cap = res.n_events;
                    cg_bed_event *ne = (cg_bed_event *)realloc(res.events, sizeof(cg_bed_event) * (size_t)res.events_cap);
                    if (!ne) goto done;
                    res.events = ne;
                    continue;
                }
                break;
            }
        } else {
            err = mg ? cgm_process_window(mg, &batch, &win, &res) : cg_process_window(ctx, &batch, &win, &res);
            if (err == CG_OK && res.n_events > res.events_cap) {                /* the chain's state has moved on: fetch again, do not redo */
                res.events_cap = res.n_events;
                cg_bed_event *ne = (cg_bed_event *)realloc(res.events, sizeof(cg_bed_event) * (size_t)res.events_cap);
                if (!ne) goto done;
                res.events = ne;
                if (mg) cgm_events(mg, res.events, res.events_cap);
                else { uint8_t *q = res.qual_out; res.qual_out = NULL; err = cg_download(ctx, &res); res.qual_out = q; }
            }
        }
        if (err) { fprintf(stderr, "crumble: GPU path failed: %s (%s)\n", cg_strerror(err), mg ? cgm_last_error(mg) : cg_last_error(ctx)); goto done; }
        device_ms += mg ? cgm_last_ms(mg) : cg_last_ms(ctx, CG_T_TOTAL);
        double tk3 = TICK(); t_dev += tk3 - tk2;
        write_bed(o, header, &res);
        for (int i = 0; i < CG_N_COUNTERS; i++) o->counters[i] += res.counters[i];

        /* ---- records that are final now: everything except pileup records reaching the first incomplete column ---- */
        for (size_t i = lq.head; i < lq.n; i++) {
            live_rec *r = &lq.v[i];
            r->is_new = 0;
            if (r->final || r->slot < 0) continue;
            bam1_t *b = r->b;
            if (reaches(r, win.hi_tid, win.hi_pos)) continue;
            if (b->core.l_qseq) {
                if (reaches(r, win.hi_tid, S)) {                                /* part of the next halo */
                    r->oq = (uint8_t *)malloc((size_t)b->core.l_qseq);
                    if (!r->oq) goto done;
                    memcpy(r->oq, bam_get_qual(b), (size_t)b->core.l_qseq);
                }
                memcpy(bam_get_qual(b), res.qual_out + batch.off[r->slot], (size_t)b->core.l_qseq);
            }
            r->final = 1;
        }
        /* ---- write the final prefix in input order; forget what no later call needs ---- */
        {
            size_t i = lq.head;
            int blocked = 0;
            for (; i < lq.n; i++) {
                live_rec *r = &lq.v[i];
                if (!r->final) blocked = 1;
                if (!blocked && r->final != 2) {
                    /* to the writer thread, which owns what it gets; a record the next call still needs as halo goes as a copy */
                    const int needed = reaches(r, win.hi_tid, S);
                    bam1_t *w = needed ? bam_dup1(r->b) : r->b;
                    if (!w) goto done;
                    if (!needed) r->b = NULL;
                    if (!wc.v && !(wc.v = (bam1_t **)malloc(sizeof(bam1_t *) * RQ_CHUNK))) { if (needed) bam_destroy1(w); else r->b = w; goto done; }
                    wc.v[wc.n++] = w;
                    count_out++;
                    if (wc.n == RQ_CHUNK) { if (rq_put(&wr.q, wc) < 0) goto done; wc.v = NULL; wc.n = 0; }
                    r->final = 2;                                               /* handed over */
                }
            }
            /* records kept for an earlier halo that the next call no longer needs */
            for (i = lq.head; i < lq.n; i++) {
                live_rec *r = &lq.v[i];
                if (r->final != 2 || !r->b) continue;
                if (!reaches(r, win.hi_tid, S)) { bam_destroy1(r->b); r->b = NULL; }
            }
            /* drop from the head every written record the next call does not need as halo */
            while (lq.head < lq.n) {
                live_rec *r = &lq.v[lq.head];
                if (r->final != 2) break;
                if (r->b) break;                                                /* kept for the next call's halo */
                free(r->oq); r->oq = NULL;
                lq.head++;
            }
        }
        t_out += TICK() - tk3;
        /* ---- next call ---- */
        if (win.hi_tid >= 0) { first = 0; lo_tid = win.hi_tid; lo_pos = S; cnt_pos = win.hi_pos; }
        else { first = 1; lo_tid = -1; lo_pos = cnt_pos = 0; }
    }
    if (wc.n) { if (rq_put(&wr.q, wc) < 0) goto done; wc.v = NULL; wc.n = 0; }
    rq_close(&wr.q, 0);
    pthread_join(wr_th, NULL); wr_on = 0;
    if (wr.q.status < 0) goto done;                                      /* write failure: -1 as snp_score.c:2007 */
    if (count_in != count_out) {                                         /* snp_score.c:2021-2026 */
        fprintf(stderr, "ERROR: lost a read?\nRead  %" PRId64 " reads\nWrote %" PRId64 " reads\n\n", count_in, count_out);
        ret = 1;
    } else ret = 0;
    o->last_device_ms = device_ms;
    if (getenv("CRUMBLE_TIMING"))
        fprintf(stderr, "[transcode_gpu] %" PRId64 " records in %" PRId64 " calls (%" PRId64 " halo records re-sent), wall %.3f s: waiting for the reader %.3f, "
                "batching %.3f, device calls %.3f (kernel chain %.3f), finalise+hand to writer %.3f, writer drain %.3f\n",
                count_in, n_calls, n_halo, TICK(), t_gather, t_build, t_dev, device_ms * 1e-3, t_out, TICK() - (t_gather + t_build + t_dev + t_out));

done:
    if (wr_on) { rq_close(&wr.q, 0); pthread_join(wr_th, NULL); }
    if (rd_on) { rq_fail(&rd.q); pthread_join(rd_th, NULL); rchunk c; while (rq_get(&rd.q, &c)) { for (int i = 0; i < c.n; i++) bam_destroy1(c.v[i]); free(c.v); } }
    for (int i = rc_i; i < rc.n; i++) bam_destroy1(rc.v[i]);
    free(rc.v);
    for (int i = 0; i < wc.n; i++) bam_destroy1(wc.v[i]);
    free(wc.v);
    if (nx) bam_destroy1(nx);
    lq_free(&lq);
    cg_host_free(res.qual_out); free(res.events);
    if (ctx) cg_destroy(ctx);
    if (mg) cgm_destroy(mg);
    if (bb) cgb_destroy(bb);
    return ret;
}
