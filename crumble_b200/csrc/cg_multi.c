/*
 * cg_multi.c — one batch over the GPUs of a box: region shards with a read halo, scheduled from plain C.
 *
 * The reference's only way to use more than one core is one process per `-r` region (snp_score.c:2616-2626); inside a
 * region everything is one sequential streaming loop whose state crosses every column (keep-window chain 1508-1511,
 * 1741-1755; depth average 1490-1491, 1673-1687).  Here one coordinate-sorted batch (any number of contigs) is cut into
 * as many shards as there are devices, of about equal size, at record boundaries.  A shard's batch is its own records plus
 * the READ HALO: the earlier records of the same contig that still cover its first columns.  Every device runs the part of
 * the kernel chain that needs no carried state at the same time (cg_shard_begin: upload, pileup, consensus, column
 * decisions, STR searches: ~3/4 of the work); the 128-byte state then travels from shard to shard through cg_shard_carry
 * (prefix sums, epochs, window chain: microseconds per shard), and the rest (over-depth test, painting, rewrite, downloads)
 * runs on all devices at once again (cg_shard_end).  No speculation, no re-runs, bit-identical to cg_process at every level.
 * Results land in the caller's buffers as cg_process would leave them: every device downloads its own byte range of
 * qual_out directly, the few halo records that turn final in a later shard come through small side buffers.
 * No device collective is involved: shards are independent given the halo and the carry (SURVEY.md §8e).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include "crumble_host.h"

typedef struct {
    struct cg_multi *m; int k;
    int64_t h0, r0, r1;                     /* records [h0, r0) = halo, [r0, r1) = the shard's own */
    cg_batch sub; cg_window win; cg_result res;
    int64_t *off2; int32_t *coff2; uint64_t *exc2;
    const cg_batch *parent; int64_t exc_first;  /* rebasing of the offset arrays and the exception list happens in the shard's own thread */
    uint8_t *head; int64_t head_bytes;
    int needs_left, has_right;
    int status;                             /* error code of this shard */
    int carry_ready;                        /* 1 = carry_out is valid, -1 = this shard failed before producing it */
    unsigned char carry_out[CG_CARRY_BYTES];
    pthread_t th; int started;
    float ms_total;
} cgm_shard;

struct cg_multi {
    int n; cg_ctx **ctx; cg_params p; char err[768];
    unsigned char carry[CG_CARRY_BYTES]; int have_carry;    /* chained calls: the state the last call's last shard saved */
    pthread_mutex_t mu; pthread_cond_t cv;
    cgm_shard *sh; int n_sh;
    unsigned char carry_in0[CG_CARRY_BYTES]; int first_needs_carry;
    float last_ms; int64_t last_h2d;
    cg_bed_event *ev; int64_t n_ev, cap_ev;                  /* all BED events of the last call, in order */
};

const char *cgm_last_error(const cg_multi *m) { return m ? m->err : "no context"; }
int cgm_n_devices(const cg_multi *m) { return m ? m->n : 0; }
float cgm_last_ms(const cg_multi *m) { return m ? m->last_ms : -1.f; }
int64_t cgm_last_h2d_bytes(const cg_multi *m) { return m ? m->last_h2d : 0; }
cg_ctx *cgm_context(cg_multi *m, int i) { return (m && i >= 0 && i < m->n) ? m->ctx[i] : NULL; }

void cgm_destroy(cg_multi *m) {
    if (!m) return;
    for (int i = 0; i < m->n; i++) if (m->ctx && m->ctx[i]) cg_destroy(m->ctx[i]);
    free(m->ctx); free(m->sh); free(m->ev);
    pthread_mutex_destroy(&m->mu); pthread_cond_destroy(&m->cv);
    free(m);
}

cg_multi *cgm_create(const cg_params *p, int n_devices, const int *devices, int *err) {
    const int avail = cg_device_count();
    if (n_devices <= 0) n_devices = avail;
    /* an explicit device list may name a device more than once (several contexts on one GPU: how the 1-GPU tests drive this code) */
    if (avail <= 0 || (!devices && n_devices > avail)) { if (err) *err = CG_ERR_NO_DEVICE; return NULL; }
    if (n_devices > 64) { if (err) *err = CG_ERR_BAD_ARG; return NULL; }
    cg_multi *m = (cg_multi *)calloc(1, sizeof *m);
    if (!m) { if (err) *err = CG_ERR_NOMEM; return NULL; }
    pthread_mutex_init(&m->mu, NULL); pthread_cond_init(&m->cv, NULL);
    m->n = n_devices; m->p = *p;
    m->ctx = (cg_ctx **)calloc((size_t)n_devices, sizeof(cg_ctx *));
    m->sh = (cgm_shard *)calloc((size_t)n_devices, sizeof(cgm_shard));
    if (!m->ctx || !m->sh) { if (err) *err = CG_ERR_NOMEM; cgm_destroy(m); return NULL; }
    for (int i = 0; i < n_devices; i++) {
        int e = 0;
        m->ctx[i] = cg_create(p, devices ? devices[i] : i, &e);
        if (!m->ctx[i]) { if (err) *err = e; cgm_destroy(m); return NULL; }
    }
    if (err) *err = 0;
    return m;
}

/* records [i0, i1) of a batch as a batch of their own: the big arrays are shared, the offsets rebased */
static int sub_batch(const cg_batch *in, int64_t i0, int64_t i1, cgm_shard *s) {
    cg_batch *b = &s->sub;
    const int64_t n = in->n_reads, cnt = i1 - i0;
    const int64_t q0 = i0 < n ? in->off[i0] : in->qual_bytes, q1 = i1 < n ? in->off[i1] : in->qual_bytes;
    const int64_t c0 = i0 < n ? in->cigar_off[i0] : in->n_cigar_total, c1 = i1 < n ? in->cigar_off[i1] : in->n_cigar_total;
    memset(b, 0, sizeof *b);
    s->off2 = (int64_t *)malloc(sizeof(int64_t) * (size_t)(cnt + 1));
    s->coff2 = (int32_t *)malloc(sizeof(int32_t) * (size_t)(cnt + 1));
    if (!s->off2 || !s->coff2) return CG_ERR_NOMEM;
    s->parent = in;                                          /* the arrays are filled by sub_batch_rebase in the shard's thread: two stores per record, all shards at once */
    b->n_reads = cnt;
    b->tid = in->tid + i0; b->pos = in->pos + i0; b->flag = in->flag + i0; b->mapq = in->mapq + i0; b->l_qseq = in->l_qseq + i0;
    b->n_cigar = in->n_cigar + i0; b->off = s->off2; b->cigar_off = s->coff2;
    b->cigar = in->cigar + c0; b->n_cigar_total = c1 - c0;
    b->seq = in->seq + q0 / 2; b->seq_bytes = (q1 - q0) / 2;
    b->qual = in->qual + q0; b->qual_bytes = q1 - q0;
    b->packed = in->packed;                                  /* running sums stay running sums after rebasing */
    if (in->seq2) {                                          /* compact planes: positions are quality-buffer offsets and rebase with q0 */
        b->seq2 = in->seq2 + q0 / 4; b->seq2_bytes = (q1 - q0) / 4;
        int64_t lo = 0, hi = in->n_seq_exc, e0, e1;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)(in->seq_exc[mid] >> 4) < q0) lo = mid + 1; else hi = mid; }
        e0 = lo; hi = in->n_seq_exc;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)(in->seq_exc[mid] >> 4) < q1) lo = mid + 1; else hi = mid; }
        e1 = lo;
        if (e1 > e0) {
            s->exc2 = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(e1 - e0));
            if (!s->exc2) return CG_ERR_NOMEM;
            s->exc_first = e0;
            b->seq_exc = s->exc2; b->n_seq_exc = e1 - e0;
        }
        b->qual_bits = in->qual_bits;
        if (in->qual_bits) { b->qualp = in->qualp + q0 * in->qual_bits / 8; b->qualp_bytes = (q1 - q0) * in->qual_bits / 8; memcpy(b->qual_dict, in->qual_dict, 16); }
    }
    return 0;
}

static void sub_batch_rebase(cgm_shard *s) {
    const cg_batch *in = s->parent;
    const int64_t i0 = s->h0, cnt = s->sub.n_reads, n = in->n_reads;
    const int64_t q0 = i0 < n ? in->off[i0] : in->qual_bytes;
    const int64_t c0 = i0 < n ? in->cigar_off[i0] : in->n_cigar_total;
    for (int64_t i = 0; i < cnt; i++) { s->off2[i] = in->off[i0 + i] - q0; s->coff2[i] = (int32_t)(in->cigar_off[i0 + i] - c0); }
    for (int64_t i = 0; i < s->sub.n_seq_exc; i++) s->exc2[i] = in->seq_exc[s->exc_first + i] - ((uint64_t)q0 << 4);
}

static void shard_free(cgm_shard *s) {
    free(s->off2); free(s->coff2); free(s->exc2); free(s->head); free(s->res.events);
    s->off2 = NULL; s->coff2 = NULL; s->exc2 = NULL; s->head = NULL; s->res.events = NULL;
}

static void publish_carry(cgm_shard *s, int state) {
    pthread_mutex_lock(&s->m->mu);
    s->carry_ready = state;
    pthread_cond_broadcast(&s->m->cv);
    pthread_mutex_unlock(&s->m->mu);
}

static void *shard_main(void *v) {
    cgm_shard *s = (cgm_shard *)v;
    cg_multi *m = s->m;
    cg_ctx *ctx = m->ctx[s->k];
    sub_batch_rebase(s);
    int e = cg_shard_begin(ctx, &s->sub, &s->win, &s->res);
    const unsigned char *cin = NULL;
    if (!e && s->needs_left) {
        if (s->k == 0) cin = m->carry_in0;                   /* a chained call: the state the previous call saved */
        else {
            cgm_shard *l = &m->sh[s->k - 1];
            pthread_mutex_lock(&m->mu);
            while (!l->carry_ready) pthread_cond_wait(&m->cv, &m->mu);
            const int ok = l->carry_ready > 0;
            pthread_mutex_unlock(&m->mu);
            if (!ok) e = CG_ERR_STATE; else cin = l->carry_out;
        }
    }
    if (!e) e = cg_shard_carry(ctx, cin, s->has_right ? s->carry_out : NULL);
    if (e) { s->status = e; publish_carry(s, -1); return NULL; }
    publish_carry(s, 1);
    for (;;) {
        e = cg_shard_end(ctx, &s->res);
        if (!e && s->res.n_events > s->res.events_cap) {      /* event buffer too small: the state has moved on, fetch again */
            cg_bed_event *ne = (cg_bed_event *)realloc(s->res.events, sizeof(cg_bed_event) * (size_t)s->res.n_events);
            if (!ne) { e = CG_ERR_NOMEM; break; }
            s->res.events = ne; s->res.events_cap = s->res.n_events;
            cg_result r2 = s->res; r2.qual_out = NULL; r2.qual_head = NULL;
            e = cg_download(ctx, &r2);
            s->res.n_events = r2.n_events;
        }
        break;
    }
    s->ms_total = cg_last_ms(ctx, CG_T_TOTAL);
    s->status = e;
    return NULL;
}

/* record i is open at the cut (tid, limit): a pileup record (end > pos) on contig tid that ends beyond limit */
static int open_at(const cg_batch *in, int64_t i, int32_t tid, int32_t limit) {
    if (in->tid[i] != tid) return 0;
    const int32_t e = cg_record_end(in->tid[i], in->pos[i], in->flag[i], in->cigar + in->cigar_off[i], in->n_cigar[i]);
    return e > in->pos[i] && e > limit;
}
/* first record of contig tid (records are sorted by (tid, pos), unplaced ones last) at or after index lo */
static int64_t contig_start(const cg_batch *in, int32_t tid, int64_t hi) {
    int64_t lo = 0;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; const int32_t t = in->tid[mid]; if (t >= 0 && t < tid) lo = mid + 1; else hi = mid; }
    return lo;
}
/* first record in [a, b) (one contig) whose end exceeds `limit`; b when none.  pmax = running max of the ends inside the contig */
static int64_t first_reaching(const int32_t *pmax, int64_t a, int64_t b, int32_t limit) {
    while (a < b) { const int64_t mid = (a + b) >> 1; if (pmax[mid] > limit) b = mid; else a = mid + 1; }
    return a;
}

/* win == NULL: the whole batch, fresh state (cg_process).  Otherwise one call of a chain (cg_process_window): the first shard
 * continues from the state this object kept from the previous call, the last one saves the state for the next. */
int cgm_process_window(cg_multi *m, const cg_batch *in, const cg_window *win, cg_result *out) {
    const int64_t n = in->n_reads;
    int N = m->n, err = 0;
    if (n < N) N = n > 0 ? (int)n : 1;
    /* running max of pos + span inside each contig: the batcher keeps it (cg_batch.pmax_end); a caller's own batch gets it here */
    int32_t *own_pmax = NULL;
    const int32_t *pmax = in->pmax_end;
    if (!pmax && n > 0) {
        own_pmax = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
        if (!own_pmax) return CG_ERR_NOMEM;
        for (int64_t i = 0; i < n; i++) {
            const int32_t e = cg_record_end(in->tid[i], in->pos[i], in->flag[i], in->cigar + in->cigar_off[i], in->n_cigar[i]);
            own_pmax[i] = (i > 0 && in->tid[i] == in->tid[i - 1] && own_pmax[i - 1] > e) ? own_pmax[i - 1] : e;
        }
        pmax = own_pmax;
    }
    m->n_sh = N; m->first_needs_carry = 0;
    memset(m->sh, 0, sizeof(cgm_shard) * (size_t)m->n);
    /* ---- plan: equal record counts; a cut inside a contig gets a halo and a window, a cut between contigs (or before unplaced
     * records) separates independent pieces.  X = position of the first record after the cut, S = start of the first record before
     * it that reaches X (S = X if none): the shard owns the columns below X, the next one replays [S, X) (include/crumble_gpu.h). ---- */
    int have_lo = 0; int32_t lo_tid = -1, lo_S = 0, lo_X = 0;
    if (win && !win->first) { have_lo = 1; lo_tid = win->lo_tid; lo_S = win->lo_pos; lo_X = win->cnt_pos; }
    for (int k = 0; k < N; k++) {
        cgm_shard *s = &m->sh[k];
        s->m = m; s->k = k;
        s->r0 = n * k / N; s->r1 = n * (k + 1) / N; s->h0 = s->r0;
        cg_window *w = &s->win; memset(w, 0, sizeof *w);
        w->first = 1; w->lo_tid = -1; w->hi_tid = -1;
        if (have_lo) {
            w->first = 0; w->lo_tid = lo_tid; w->lo_pos = lo_S; w->cnt_pos = lo_X; s->needs_left = 1;
            if (k > 0) s->h0 = first_reaching(pmax, contig_start(in, lo_tid, s->r0), s->r0, lo_S);   /* halo: the earlier records of that contig from the first one reaching beyond S */
        }
        have_lo = 0;
        const int last = k == N - 1;
        if (!last && s->r1 > 0 && s->r1 < n && in->tid[s->r1] >= 0 && in->tid[s->r1] == in->tid[s->r1 - 1]) {
            const int32_t t = in->tid[s->r1], X = in->pos[s->r1];
            int64_t a = contig_start(in, t, s->r1);
            if (a < s->h0) a = s->h0;
            const int64_t iS = first_reaching(pmax, a, s->r1, X);
            /* pmax may carry an end from before `a`: the first record of [a, r1) that really reaches X */
            int64_t ii = iS; while (ii < s->r1 && !open_at(in, ii, t, X)) ii++;
            int32_t S = ii < s->r1 ? in->pos[ii] : X;
            /* a chained call whose first shards hold nothing but halo records: a cut below the first column this CALL owns (X < cnt_pos) must
             * neither make the next shard count the columns in between again (the previous call of the chain counted them), nor start its
             * replay below the call's own: the records that reach such a cut but start below lo_pos were finalised by the previous call, and
             * the state this call received already contains every column below lo_pos */
            const int chained_here = win && !win->first && t == win->lo_tid;
            if (chained_here && S < win->lo_pos) S = win->lo_pos;
            w->hi_tid = t; w->hi_pos = X; w->next_lo_pos = S; s->has_right = 1;
            have_lo = 1; lo_tid = t; lo_S = S; lo_X = X;
            if (chained_here && lo_X < win->cnt_pos) lo_X = win->cnt_pos;
        } else if (last && win && win->hi_tid >= 0) {
            w->hi_tid = win->hi_tid; w->hi_pos = win->hi_pos; w->next_lo_pos = win->next_lo_pos; s->has_right = 1;
        }
        if ((err = sub_batch(in, s->h0, s->r1, s))) goto fail;
        s->head_bytes = (s->r0 < n ? in->off[s->r0] : in->qual_bytes) - (s->h0 < n ? in->off[s->h0] : in->qual_bytes);
        if (s->head_bytes > 0 && !(s->head = (uint8_t *)malloc((size_t)s->head_bytes))) { err = CG_ERR_NOMEM; goto fail; }
        s->res.qual_out = out->qual_out ? out->qual_out + (s->h0 < n ? in->off[s->h0] : in->qual_bytes) : NULL;
        s->res.qual_head = s->head; s->res.head_bytes = s->head_bytes;
        s->res.events_cap = 1 << 14;
        s->res.events = (cg_bed_event *)malloc(sizeof(cg_bed_event) * (size_t)s->res.events_cap);
        if (!s->res.events) { err = CG_ERR_NOMEM; goto fail; }
    }
    if (m->sh[0].needs_left) {
        if (!m->have_carry) { snprintf(m->err, sizeof m->err, "chained call without a saved state"); err = CG_ERR_STATE; goto fail; }
        memcpy(m->carry_in0, m->carry, CG_CARRY_BYTES);
    }
    /* ---- run: one thread per shard / device ---- */
    for (int k = 0; k < N; k++) {
        if (pthread_create(&m->sh[k].th, NULL, shard_main, &m->sh[k]) != 0) { m->sh[k].status = CG_ERR_NOMEM; publish_carry(&m->sh[k], -1); }
        else m->sh[k].started = 1;
    }
    for (int k = 0; k < N; k++) if (m->sh[k].started) pthread_join(m->sh[k].th, NULL);
    for (int k = 0; k < N; k++) if (m->sh[k].status && !err) {
        err = m->sh[k].status;
        snprintf(m->err, sizeof m->err, "shard %d of %d: %s (%s)", k, N, cg_strerror(err), cg_last_error(m->ctx[k]));
    }
    if (err) goto fail;
    /* ---- gather: a halo record that was still open at the previous cut turns final in the first shard whose own cut it does not
     * reach: its bytes sit in that shard's side buffer.  Events in shard (= position) order, counters summed. ---- */
    {
        int64_t ne = 0;
        memset(out->counters, 0, sizeof out->counters);
        m->last_ms = 0; m->last_h2d = 0;
        for (int k = 0; k < N; k++) {
            cgm_shard *s = &m->sh[k];
            if (k > 0 && s->needs_left && out->qual_out) {
                const cgm_shard *l = &m->sh[k - 1];
                const int64_t base = in->off[s->h0];
                for (int64_t i = s->h0; i < s->r0; i++) {
                    if (in->l_qseq[i] <= 0 || !open_at(in, i, l->win.hi_tid, l->win.hi_pos)) continue;   /* was final in an earlier shard */
                    if (open_at(in, i, s->win.hi_tid, s->win.hi_pos)) continue;     /* still open: a later shard has it in its halo too */
                    /* open at every cut since its own shard, closed here: but only the FIRST shard after its last open cut holds the final bytes, and
                     * that is this one, because it was still open at the cut just before */
                    memcpy(out->qual_out + in->off[i], s->head + (in->off[i] - base), (size_t)in->l_qseq[i]);
                }
            }
            if (ne + s->res.n_events > m->cap_ev) {
                const int64_t nc = (ne + s->res.n_events) * 2 + 1024;
                cg_bed_event *nv = (cg_bed_event *)realloc(m->ev, sizeof(cg_bed_event) * (size_t)nc);
                if (!nv) { err = CG_ERR_NOMEM; goto fail; }
                m->ev = nv; m->cap_ev = nc;
            }
            for (int64_t j = 0; j < s->res.n_events; j++, ne++) { m->ev[ne] = s->res.events[j]; if (out->events && ne < out->events_cap) out->events[ne] = s->res.events[j]; }
            for (int c = 0; c < CG_N_COUNTERS; c++) out->counters[c] += s->res.counters[c];
            if (s->ms_total > m->last_ms) m->last_ms = s->ms_total;
            m->last_h2d += cg_last_h2d_bytes(m->ctx[k]);
        }
        out->n_events = ne; out->n_columns = 0; m->n_ev = ne;
        cgm_shard *lastS = &m->sh[N - 1];
        m->have_carry = lastS->has_right;
        if (lastS->has_right) memcpy(m->carry, lastS->carry_out, CG_CARRY_BYTES);
    }
fail:
    for (int k = 0; k < m->n; k++) shard_free(&m->sh[k]);
    free(own_pmax);
    return err;
}

int cgm_process(cg_multi *m, const cg_batch *in, cg_result *out) { return cgm_process_window(m, in, NULL, out); }

/* the BED events of the last call again (a caller whose event buffer was too small): returns how many there are */
int64_t cgm_events(const cg_multi *m, cg_bed_event *buf, int64_t cap) {
    for (int64_t i = 0; i < m->n_ev && i < cap; i++) buf[i] = m->ev[i];
    return m->n_ev;
}
