/*
 * TEST INFRASTRUCTURE ONLY — never linked into libcrumble_gpu.so.
 *
 * The host emulation of cg_emu.cpp as a shared library (libcg_emu.so, tests/emu/device.mk), plus the device-resident entry
 * cg_process_device of include/crumble_gpu.h: "device" pointers are host memory here, and the ingest / emit bodies of cg_device.cu's
 * k_ingest / k_emit (cg_pipeline.h) run in plain loops around the emulated chain.  The CPU suite (tests/test_device_batch.py) calls it
 * through ctypes.
 */
#include "cg_emu.cpp"

/* records in "device" memory (host memory here): the running sums the device scans build, the same checks, then the ingest bodies,
 * the emulated chain on the padded layout and the emit bodies of cg_device.cu's k_ingest / k_emit */
extern "C" int cg_process_device(cg_ctx *ctx, const cg_dev_batch *in, uint8_t *qual_out, cg_result *out) {
    const int64_t n = in->n_reads;
    if (n < 0 || in->n_cigar_total < 0 || in->seq_len < 0 || in->qual_len < 0) { snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: negative count"); return CG_ERR_BAD_ARG; }
    if (out->qual_out || out->qual_head) { snprintf(ctx->err, sizeof ctx->err, "out->qual_out and out->qual_head must be NULL"); return CG_ERR_BAD_ARG; }
    if ((n && (!in->tid || !in->pos || !in->flag || !in->mapq || !in->l_qseq || !in->n_cigar)) || (in->n_cigar_total && !in->cigar) ||
        (in->seq_len && !in->seq) || (in->qual_len && (!in->qual || !qual_out))) { snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: missing array"); return CG_ERR_BAD_ARG; }
    std::vector<int64_t> off(n + 1), qsrc(n + 1), ssrc(n + 1); std::vector<int32_t> coff(n + 1);
    int64_t padded = 0, ncig = 0, nq = 0, ns = 0, neg = 0;
    for (int64_t r = 0; r < n; r++) {
        const int64_t l = in->l_qseq[r];
        off[r] = padded; coff[r] = (int32_t)ncig; qsrc[r] = nq; ssrc[r] = ns;
        padded += (l + 7) & ~(int64_t)7; ncig += in->n_cigar[r]; nq += l; ns += (l + 1) >> 1; neg += l < 0;
    }
    if (neg || nq != in->qual_len || ns != in->seq_len || ncig != in->n_cigar_total) {
        snprintf(ctx->err, sizeof ctx->err, "cg_dev_batch: sums disagree (%lld negative l_qseq; %lld/%lld quality bytes, %lld/%lld sequence bytes, %lld/%lld CIGAR operations)",
                 (long long)neg, (long long)nq, (long long)in->qual_len, (long long)ns, (long long)in->seq_len, (long long)ncig, (long long)in->n_cigar_total);
        return CG_ERR_BAD_ARG;
    }
    std::vector<uint8_t> qual((size_t)padded + 8, 0xee), seq((size_t)padded / 2 + 8, 0xee), qo((size_t)padded + 8, 0);
    const CgIngest I = { in->l_qseq, off.data(), qsrc.data(), ssrc.data(), in->qual, in->seq, qual.data(), seq.data() };
    for (int64_t r = 0; r < n; r++) for (int k = 0; k < (in->l_qseq[r] + 7) >> 3; k++) cg_ingest_group(&I, r, k);
    cg_batch b; memset(&b, 0, sizeof b);
    b.n_reads = n; b.tid = in->tid; b.pos = in->pos; b.flag = in->flag; b.mapq = in->mapq; b.l_qseq = in->l_qseq; b.n_cigar = in->n_cigar;
    b.off = off.data(); b.cigar_off = coff.data(); b.cigar = in->cigar; b.n_cigar_total = in->n_cigar_total;
    b.seq = seq.data(); b.seq_bytes = padded / 2; b.qual = qual.data(); b.qual_bytes = padded; b.packed = 1;
    cg_result r = *out; r.qual_out = qo.data();
    const int e = emu_process(ctx, &b, NULL, &r);
    if (e) return e;
    out->n_events = r.n_events; out->n_columns = r.n_columns;
    memcpy(out->counters, r.counters, sizeof out->counters);
    const CgEmit E = { in->l_qseq, off.data(), qsrc.data(), qo.data(), qual_out };
    for (int64_t i = 0; i < n; i++) for (int j = 0, nw = cg_emit_words(&E, i); j < nw; j++) cg_emit_word(&E, i, j);
    return 0;
}
/* the padded working layout k_ingest builds, for the CPU tests: qual[padded], seq[padded / 2] */
extern "C" int64_t cg_emu_ingest(const cg_dev_batch *in, uint8_t *qual, uint8_t *seq) {
    std::vector<int64_t> off(in->n_reads + 1), qsrc(in->n_reads + 1), ssrc(in->n_reads + 1);
    int64_t padded = 0, nq = 0, ns = 0;
    for (int64_t r = 0; r < in->n_reads; r++) {
        const int64_t l = in->l_qseq[r];
        off[r] = padded; qsrc[r] = nq; ssrc[r] = ns; padded += (l + 7) & ~(int64_t)7; nq += l; ns += (l + 1) >> 1;
    }
    if (!qual) return padded;
    const CgIngest I = { in->l_qseq, off.data(), qsrc.data(), ssrc.data(), in->qual, in->seq, qual, seq };
    for (int64_t r = 0; r < in->n_reads; r++) for (int k = 0; k < (in->l_qseq[r] + 7) >> 3; k++) cg_ingest_group(&I, r, k);
    return padded;
}

