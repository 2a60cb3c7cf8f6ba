/*
 * TEST INFRASTRUCTURE ONLY — never linked into libcrumble_gpu.so.
 *
 * libcg_emu_stream.so (tests/emu/stream.mk): the emulation of cg_emu_device.cpp plus the stream entry cg_stream_device of
 * include/crumble_gpu.h, with the plan / cut / keep / retain / ingest / emit bodies of cg_device.cu's kernels (cg_pipeline.h) in plain
 * loops around the emulated window chain.  The CPU suite (tests/test_device_stream.py) calls it through ctypes.
 *
 * The entries that must refuse to run while a stream is open (CG_ERR_STATE) are the emulation's own, renamed on inclusion and wrapped
 * below; the state of an open stream lives in a table keyed by context, which cg_destroy clears.
 */
#define cg_destroy        cg_emu_base_destroy
#define cg_process        cg_emu_base_process
#define cg_process_window cg_emu_base_process_window
#define cg_process_device cg_emu_base_process_device
#define cg_shard_begin    cg_emu_base_shard_begin
#define cg_shard_carry    cg_emu_base_shard_carry
#define cg_shard_end      cg_emu_base_shard_end
#include "cg_emu_device.cpp"
#undef cg_destroy
#undef cg_process
#undef cg_process_window
#undef cg_process_device
#undef cg_shard_begin
#undef cg_shard_carry
#undef cg_shard_end
#include <unordered_map>

/* an open stream: the held store in the padded working layout, and the state of the next call */
struct EmuStream {
    int open = 0, has_key = 0, unplaced = 0; uint64_t kmax = 0; int64_t e0 = 0, qual_len = 0, seq_len = 0;
    std::vector<int32_t> tid, pos, lq; std::vector<uint16_t> flag, nc; std::vector<uint8_t> mapq, qual, seq; std::vector<uint32_t> cig;
    cg_window win = { 1, -1, 0, 0, -1, 0, 0 };
};
static std::unordered_map<const cg_ctx *, EmuStream> g_streams;
static EmuStream &stream_of(const cg_ctx *ctx) { return g_streams[ctx]; }
static int stream_busy(cg_ctx *ctx) {
    const auto it = g_streams.find(ctx);
    if (it == g_streams.end() || !it->second.open) return 0;
    snprintf(ctx->err, sizeof ctx->err, "a stream is open on this context");
    return CG_ERR_STATE;
}

extern "C" void cg_destroy(cg_ctx *c) { g_streams.erase(c); cg_emu_base_destroy(c); }
extern "C" int cg_process(cg_ctx *ctx, const cg_batch *in, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    return cg_emu_base_process(ctx, in, out);
}
extern "C" int cg_process_window(cg_ctx *ctx, const cg_batch *in, const cg_window *win, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    return cg_emu_base_process_window(ctx, in, win, out);
}
extern "C" int cg_process_device(cg_ctx *ctx, const cg_dev_batch *in, uint8_t *qual_out, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    return cg_emu_base_process_device(ctx, in, qual_out, out);
}
extern "C" int cg_shard_begin(cg_ctx *ctx, const cg_batch *in, const cg_window *win, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    return cg_emu_base_shard_begin(ctx, in, win, out);
}
extern "C" int cg_shard_carry(cg_ctx *ctx, const void *carry_in, void *carry_out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    return cg_emu_base_shard_carry(ctx, carry_in, carry_out);
}
extern "C" int cg_shard_end(cg_ctx *ctx, cg_result *out) {
    if (stream_busy(ctx)) return CG_ERR_STATE;
    return cg_emu_base_shard_end(ctx, out);
}

/* ---- cg_device.cu's cg_stream_device, step for step ---------------------------------------------------------------------------------- */
static int emu_stream_call(cg_ctx *ctx, const cg_dev_batch *in, int last, uint8_t *qual_out, cg_result *out, cg_stream_out *so) {
    EmuStream &S = stream_of(ctx);
    const int64_t nh = (int64_t)S.tid.size(), ni = in->n_reads, n = nh + ni, e0 = S.e0;
    const int64_t hcig = (int64_t)S.cig.size(), hpad = (int64_t)S.qual.size();
    std::vector<int32_t> tid(S.tid), pos(S.pos), lq(S.lq); std::vector<uint16_t> flag(S.flag), nc(S.nc); std::vector<uint8_t> mapq(S.mapq);
    std::vector<uint32_t> cig(S.cig);
    tid.insert(tid.end(), in->tid, in->tid + ni); pos.insert(pos.end(), in->pos, in->pos + ni); lq.insert(lq.end(), in->l_qseq, in->l_qseq + ni);
    flag.insert(flag.end(), in->flag, in->flag + ni); nc.insert(nc.end(), in->n_cigar, in->n_cigar + ni); mapq.insert(mapq.end(), in->mapq, in->mapq + ni);
    cig.insert(cig.end(), in->cigar, in->cigar + in->n_cigar_total);
    std::vector<int64_t> off(n + 1), qsrc(n + 1), ssrc(n + 1); std::vector<int32_t> coff(n + 1), rspan(n + 1);
    int64_t padded = 0, ncig = 0, nq = 0, ns = 0, neg = 0;
    for (int64_t r = 0; r < n; r++) {
        const int64_t l = lq[r];
        off[r] = padded; coff[r] = (int32_t)ncig; qsrc[r] = nq; ssrc[r] = ns;
        padded += (l + 7) & ~(int64_t)7; ncig += nc[r]; nq += l; ns += (l + 1) >> 1; neg += l < 0;
    }
    if (neg || nq - S.qual_len != in->qual_len || ns - S.seq_len != in->seq_len || ncig - hcig != in->n_cigar_total) {
        snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: sums disagree"); return CG_ERR_BAD_ARG;
    }
    memset(so, 0, sizeof *so); memset(out->counters, 0, sizeof out->counters); out->n_events = 0; out->n_columns = 0;
    if (n == 0) return 0;
    std::vector<uint8_t> qual((size_t)padded + 8, 0xee), seq((size_t)padded / 2 + 8, 0xee), qo((size_t)padded + 8, 0);
    memcpy(qual.data(), S.qual.data(), (size_t)hpad); memcpy(seq.data(), S.seq.data(), (size_t)hpad / 2);
    const CgIngest I = { lq.data() + nh, off.data() + nh, qsrc.data() + nh, ssrc.data() + nh, in->qual, in->seq, qual.data(), seq.data(), S.qual_len, S.seq_len };
    for (int64_t r = 0; r < ni; r++) for (int k = 0; k < (in->l_qseq[r] + 7) >> 3; k++) cg_ingest_group(&I, r, k);
    /* plan and cut */
    CgDev D; memset(&D, 0, sizeof D);
    int32_t err = 0;
    D.n_reads = n; D.n_cigar_total = ncig; D.tid = tid.data(); D.pos = pos.data(); D.flag = flag.data(); D.mapq = mapq.data(); D.l_qseq = lq.data();
    D.n_cigar = nc.data(); D.off = off.data(); D.cigar_off = coff.data(); D.cigar = cig.data(); D.rspan = rspan.data(); D.err = &err;
    for (int64_t r = 0; r < n; r++) cg_prep_read(&D, r);
    CgStreamRed red; cg_stream_red_init(&red);
    for (int64_t r = 0; r < n; r++) { const CgStreamRed c = cg_stream_plan_item(&D, r, n, nh, e0); cg_stream_red_merge(&red, &c); }
    const CgStreamCut c = cg_stream_cut(&D, &red, n, e0, last, qsrc.data(), nq);
    if (red.kmin <= red.kmax && ((S.has_key && red.kmin < S.kmax) || S.unplaced)) { snprintf(ctx->err, sizeof ctx->err, "unsorted across chunks"); return CG_ERR_UNSORTED; }
    /* the held set, through the retain bodies */
    std::vector<uint8_t> keep(n);
    std::vector<int32_t> didx(n + 1), dcig(n + 1); std::vector<int64_t> doff(n + 1);
    int64_t hn = 0, hp = 0, hc = 0, hq = 0, hs = 0;
    for (int64_t r = 0; r < n; r++) {
        keep[r] = (uint8_t)cg_stream_keep(&D, r, &c);
        didx[r] = (int32_t)hn; doff[r] = hp; dcig[r] = (int32_t)hc;
        if (keep[r]) { hn++; hp += ((int64_t)lq[r] + 7) & ~(int64_t)7; hc += nc[r]; hq += lq[r]; hs += ((int64_t)lq[r] + 1) >> 1; }
    }
    EmuStream N;
    N.tid.resize(hn); N.pos.resize(hn); N.lq.resize(hn); N.flag.resize(hn); N.nc.resize(hn); N.mapq.resize(hn); N.cig.resize(hc);
    N.qual.resize(hp); N.seq.resize(hp / 2);
    const CgRetain K = { tid.data(), pos.data(), lq.data(), flag.data(), nc.data(), mapq.data(), off.data(), coff.data(), cig.data(), qual.data(), seq.data(),
                         didx.data(), dcig.data(), doff.data(), N.tid.data(), N.pos.data(), N.lq.data(), N.flag.data(), N.nc.data(), N.mapq.data(),
                         N.cig.data(), N.qual.data(), N.seq.data() };
    for (int64_t r = 0; r < n; r++) if (keep[r]) for (int j = 0, nj = cg_retain_items(&K, r); j < nj; j++) cg_retain_item(&K, r, j);
    N.open = 1; N.win = S.win; N.e0 = hn - (n - c.f); N.qual_len = hq; N.seq_len = hs;
    N.has_key = S.has_key; N.kmax = S.kmax; N.unplaced = S.unplaced | red.unplaced;
    if (red.kmin <= red.kmax) { N.has_key = 1; N.kmax = red.kmax; }
    int64_t n_emit = 0;
    if (!c.skip) {
        cg_window w = S.win; w.hi_tid = c.hi_tid; w.hi_pos = c.hi_pos; w.next_lo_pos = c.S;
        cg_batch b; memset(&b, 0, sizeof b);
        b.n_reads = c.m; b.tid = tid.data(); b.pos = pos.data(); b.flag = flag.data(); b.mapq = mapq.data(); b.l_qseq = lq.data(); b.n_cigar = nc.data();
        b.off = off.data(); b.cigar_off = coff.data(); b.cigar = cig.data(); b.n_cigar_total = ncig;
        b.seq = seq.data(); b.seq_bytes = padded / 2; b.qual = qual.data(); b.qual_bytes = padded; b.packed = 1;
        cg_result r = *out; r.qual_out = qo.data();
        const int e = emu_process(ctx, &b, &w, &r);
        if (e) return e;
        out->n_events = r.n_events; memcpy(out->counters, r.counters, sizeof out->counters);
        const CgEmit E = { lq.data() + e0, off.data() + e0, qsrc.data() + e0, qo.data(), qual_out, c.q_e0 };
        for (int64_t i = 0; i < c.f - e0; i++) for (int j = 0, nw = cg_emit_words(&E, i); j < nw; j++) cg_emit_word(&E, i, j);
        n_emit = c.f - e0;
        if (c.hi_tid >= 0) { N.win.first = 0; N.win.lo_tid = c.hi_tid; N.win.lo_pos = c.S; N.win.cnt_pos = c.hi_pos; }
        else { N.win.first = 1; N.win.lo_tid = -1; N.win.lo_pos = N.win.cnt_pos = 0; }
    }
    S = N;
    so->n_records = n_emit; so->qual_len = n_emit ? c.q_f - c.q_e0 : 0;
    return 0;
}

extern "C" int cg_stream_device(cg_ctx *ctx, const cg_dev_batch *in, int last, uint8_t *qual_out, int64_t qual_cap, cg_result *out, cg_stream_out *so) {
    cg_dev_batch none; memset(&none, 0, sizeof none);
    if (!in) in = &none;
    if (!out || !so || out->columns || out->qual_out || out->qual_head || ctx->p.region_tid >= 0) { snprintf(ctx->err, sizeof ctx->err, "cg_stream_device: bad arguments"); return CG_ERR_BAD_ARG; }
    EmuStream &S = stream_of(ctx);
    if (qual_cap < S.qual_len + in->qual_len) { snprintf(ctx->err, sizeof ctx->err, "cg_stream_device: qual_cap too small"); return CG_ERR_BAD_ARG; }
    const int64_t n = in->n_reads;
    if (n < 0 || in->n_cigar_total < 0 || in->seq_len < 0 || in->qual_len < 0) { snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: negative count"); return CG_ERR_BAD_ARG; }
    if ((n && (!in->tid || !in->pos || !in->flag || !in->mapq || !in->l_qseq || !in->n_cigar)) || (in->n_cigar_total && !in->cigar) ||
        (in->seq_len && !in->seq) || (in->qual_len && !in->qual) || (qual_cap && !qual_out)) { snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: missing array"); return CG_ERR_BAD_ARG; }
    S.open = 1;
    if (n == 0 && !last) {
        memset(so, 0, sizeof *so); memset(out->counters, 0, sizeof out->counters); out->n_events = 0; out->n_columns = 0;
        so->held_records = (int64_t)S.tid.size(); so->held_qual_len = S.qual_len;
        return 0;
    }
    const int e = emu_stream_call(ctx, in, last, qual_out, out, so);
    if (e || last) S = EmuStream();
    if (e) return e;
    so->held_records = (int64_t)S.tid.size(); so->held_qual_len = S.qual_len;
    return 0;
}

/* the cut of one working batch alone (no held records): m, f, hi_tid, hi_pos, S, skip, for the CPU tests' model of it */
extern "C" void cg_emu_stream_cut(const cg_dev_batch *in, int64_t e0, int last, int32_t *res) {
    const int64_t n = in->n_reads;
    std::vector<int32_t> coff(n + 1), rspan(n + 1); std::vector<int64_t> qsrc(n + 1);
    int64_t nc = 0, nq = 0;
    for (int64_t r = 0; r < n; r++) { coff[r] = (int32_t)nc; qsrc[r] = nq; nc += in->n_cigar[r]; nq += in->l_qseq[r]; }
    CgDev D; memset(&D, 0, sizeof D);
    int32_t err = 0;
    D.n_reads = n; D.n_cigar_total = nc; D.tid = in->tid; D.pos = in->pos; D.flag = in->flag; D.l_qseq = in->l_qseq; D.n_cigar = in->n_cigar;
    D.cigar_off = coff.data(); D.cigar = in->cigar; D.rspan = rspan.data(); D.err = &err;
    for (int64_t r = 0; r < n; r++) cg_prep_read(&D, r);
    CgStreamRed red; cg_stream_red_init(&red);
    for (int64_t r = 0; r < n; r++) { const CgStreamRed c = cg_stream_plan_item(&D, r, n, 0, e0); cg_stream_red_merge(&red, &c); }
    const CgStreamCut c = cg_stream_cut(&D, &red, n, e0, last, qsrc.data(), nq);
    res[0] = c.m; res[1] = c.f; res[2] = c.hi_tid; res[3] = c.hi_pos; res[4] = c.S; res[5] = c.skip;
}
