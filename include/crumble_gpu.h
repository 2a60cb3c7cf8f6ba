/*
 * crumble_gpu.h — C ABI of the B200-native consensus + quality-rewrite hot path.
 *
 * This is the drop-in boundary for ONE path of jkbonfield/crumble: everything that
 * `int transcode(cram_lossy_params *p, samFile *in, samFile *out, bam_hdr_t *header,
 * hts_itr_t *h_iter)` (reference snp_score.c:1336-2029) does between reading a
 * record and writing it back: pileup construction, calculate_consensus_pileup
 * (snp_score.c:533-797), the column heuristics (1658-1819), STR keep windows
 * (mask_LC_regions 1230-1290, find_STR str_finder.c:135-189), the per-base quality
 * rewrite (1822-1920), the tail/keep handling (1926-1975) and flush_bam_list's
 * strip + P-block (1090-1100, pblock 803-834).
 *
 * Plain C, plain pointers and sizes; no CUDA, C++ or torch types cross this line.
 * All compute entry points fail with CG_ERR_NO_DEVICE when no CUDA device is usable:
 * there is no CPU fallback behind this ABI.
 */
#ifndef CRUMBLE_GPU_H
#define CRUMBLE_GPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CG_ABI_VERSION 3

/* ---- error codes (negative; 0 = ok).  transcode_gpu() maps any of these to -1, the
 * value transcode() returns on failure (snp_score.c:1480-1481,1979-1980). ------------- */
enum {
    CG_OK               =  0,
    CG_ERR_NO_DEVICE    = -1,   /* no CUDA device / driver: the GPU path is mandatory */
    CG_ERR_CUDA         = -2,   /* a CUDA runtime call or kernel failed (see cg_last_error) */
    CG_ERR_NOMEM        = -3,
    CG_ERR_BAD_ARG      = -4,
    CG_ERR_UNSORTED     = -5,   /* input not coordinate sorted (htslib's pileup aborts too) */
    CG_ERR_UNSUPPORTED  = -6,   /* option combination not implemented on the device yet */
    CG_ERR_OVERFLOW     = -7,   /* an internal fixed-size device list overflowed */
    CG_ERR_STATE        = -8    /* calls made out of order */
};

/* ---- parameters: POD mirror of cram_lossy_params (snp_score.c:185-226) -------------- */
typedef struct { int32_t tid, start, end; } cg_bed_reg;      /* bed.h:4-6 */

typedef struct cg_params {
    int32_t reduce_qual, binary_qual;            /* -L, -B */
    int32_t iSTR_add, sSTR_add;                  /* -i, -s */
    double  iSTR_mul, sSTR_mul;
    int32_t qlow, qcutoff, qhigh, qcap;          /* -l -c -u -U */
    int32_t min_mqual;                           /* -m */
    double  indel_fract;                         /* -Y */
    int32_t min_qual_A, min_indel_A;             /* -q -d */
    double  min_discrep_A;                       /* -x */
    int32_t min_qual_B, min_indel_B;             /* -Q -D */
    double  min_discrep_B;                       /* -X */
    double  low_mqual_perc, clip_perc, ins_len_perc, over_depth, indel_ov_perc;   /* -M -C -Z -P -V */
    int32_t pblock;                              /* -p */
    int32_t softclip;                            /* -S */
    int32_t perfect_col;                         /* -N */
    int32_t verbose;                             /* -v */
    int32_t noPG;                                /* -z */
    /* -r region (hts_itr_t beg/end, snp_score.c:1513-1518); region_tid < 0 = whole file */
    int32_t region_tid, region_beg, region_end;
    /* -k / -K: 0 none, 1 keep if diffs, 2 always keep (snp_score.c:232,2362-2375) */
    uint8_t preserve_qual[256];
    /* -R keep.bed, sorted + merged as bed.c:20-40 leaves them; borrowed pointer */
    const cg_bed_reg *bed;
    int32_t nbed;
    /* BD/BI binarisation and tag lists are host-side only (purge_tags) and not part of this ABI */
} cg_params;

/* defaults = reference main() initialiser (snp_score.c:2152-2192) */
void cg_params_default(cg_params *p);
/* level presets -1,-3,-5,-7,-8,-9 (snp_score.c:2380-2482); returns 0 or CG_ERR_BAD_ARG */
int  cg_params_level(cg_params *p, int level);

/* ---- a batch of decoded alignment records, structure-of-arrays, host memory ----------
 * Records are in input (coordinate-sorted) order.  Byte layout:
 *   qual : per read l_qseq bytes at qual[off[i]], off[i] a multiple of 8
 *   seq  : 4-bit codes =ACMGRSVTWYHKDBN, high nibble first, at seq[off[i] / 2]
 *   cigar: BAM encoding len<<4|op at cigar[cigar_off[i]], n_cigar[i] entries
 * Build one with the cgb_* functions below (they also pin the memory).               */
typedef struct cg_batch {
    int64_t  n_reads;
    const int32_t  *tid;        /* -1 for unplaced */
    const int32_t  *pos;        /* 0-based leftmost reference coordinate */
    const uint16_t *flag;
    const uint8_t  *mapq;
    const int32_t  *l_qseq;
    const uint16_t *n_cigar;
    const int64_t  *off;        /* qual byte offset; seq byte offset is off/2 */
    const int32_t  *cigar_off;
    const uint32_t *cigar;  int64_t n_cigar_total;
    const uint8_t  *seq;    int64_t seq_bytes;
    const uint8_t  *qual;   int64_t qual_bytes;
    int32_t  packed;            /* 1: off[] and cigar_off[] are the running sums of ((l_qseq + 7) & ~7) and n_cigar starting at 0 (what the
                                   cgb_* batcher builds): the device rebuilds them with two scans instead of receiving 12 bytes per record */
    /* Optional COMPACT PLANES of the two big arrays (cgb_pack builds them next to seq / qual).  When present the upload moves these
     * instead and the device expands them into its 4-bit / 8-bit working arrays: 0.25 + 0.25..0.5 bytes per base cross PCIe in place
     * of 1.5.  Both are indexed like qual[] (position = byte offset in the quality buffer, padding included).
     *   seq2     2-bit bases A0 C1 G2 T3, four per byte, position i at bits 2*(i&3) of byte i>>2; every other nt16 code is an
     *            exception: seq_exc[] = (position << 4 | code), ascending (padding positions are A and never listed);
     *   qualp    dictionary codes of the qualities, qual_bits (2 or 4) per position, low bits first; qual_dict[code] = value
     *            (padding positions carry code 0).  qual_bits = 0: no such plane (more than 16 distinct values), qual[] travels. */
    const uint8_t  *seq2;     int64_t seq2_bytes;
    const uint64_t *seq_exc;  int64_t n_seq_exc;
    const uint8_t  *qualp;    int64_t qualp_bytes;
    int32_t  qual_bits;
    uint8_t  qual_dict[16];
    /* optional: running maximum of pos + reference span inside each contig (the batcher keeps it): lets cgm_process place region
     * shard cuts and halos by binary search instead of walking every CIGAR */
    const int32_t *pmax_end;
    /* Optional COMPACT PLANES of the per-record arrays (cgb_pack builds them for a packed batch; meta_planes = 1 says they are all
     * there).  The upload then moves about 6 bytes per record instead of 21 and the device rebuilds tid / pos / l_qseq / n_cigar /
     * cigar from them, so the first slice of a streamed call starts (and its results start to travel back) that much earlier.
     *   tid_runs  (first record index << 32 | (uint32_t)tid), one entry per run of equal tid, ascending;
     *   pos_d8    pos - pos of the previous record, 0..254; 255: the record is listed in pos_abs (first of a contig, large gaps,
     *             unsorted stretches): pos_abs[] = (record index << 32 | (uint32_t)pos), ascending;
     *   lq8       l_qseq = lq_dict[lq8[i]] (at most 256 distinct read lengths);
     *   nc8       n_cigar (0..254); 255: the CIGAR is one M operation of l_qseq bases and is not listed;
     *   cigar_x   the CIGAR operations of the other records, back to back in record order.
     * flag[] and mapq[] travel as they are. */
    int32_t  meta_planes;
    const uint64_t *tid_runs; int64_t n_tid_runs;
    const uint8_t  *pos_d8;
    const uint64_t *pos_abs;  int64_t n_pos_abs;
    const uint8_t  *lq8;      int32_t lq_dict[256];
    const uint8_t  *nc8;
    const uint32_t *cigar_x;  int64_t n_cigar_x;
} cg_batch;

/* BED_DIST-expanded suspicious-region events (snp_score.c:1496-1498,1676-1678,
 * 1768-1770,1802-1804,1810-1812), in the order the reference prints them. */
enum { CG_BED_VDEEP = 0, CG_BED_DEEP = 1, CG_BED_CLIP = 2, CG_BED_INDEL_LEN = 3, CG_BED_INDEL_COVERAGE = 4 };
typedef struct { int32_t tid, pos, tag; } cg_bed_event;    /* pos = column; line is max(pos-50,0), pos+50 */

/* the reference's -v counters (snp_score.c:1292-1311), same order as printed (2652-2665) */
enum {
    CG_CNT_DIFF = 0, CG_CNT_INDEL_QUAL, CG_CNT_INDEL,
    CG_CNT_HET_QUAL_A, CG_CNT_HET_A, CG_CNT_HOM_QUAL_A, CG_CNT_HOM_A, CG_CNT_DISCREP_A,
    CG_CNT_HET_QUAL_B, CG_CNT_HET_B, CG_CNT_HOM_QUAL_B, CG_CNT_HOM_B, CG_CNT_DISCREP_B,
    CG_CNT_COLUMNS, CG_CNT_LOW_MQUAL_PERC, CG_CNT_CLIP_PERC, CG_CNT_INS_LEN_PERC,
    CG_CNT_INDEL_OV_PERC, CG_CNT_OVER_DEPTH,
    CG_N_COUNTERS
};

/* optional per-column dump for parity checks (consensus_t, snp_score.c:257-281) */
typedef struct {
    int32_t tid, pos, n_plp;
    int32_t call, het_call, het_phred, phred;     /* mode B if enabled else mode A */
    float   discrep;
    uint32_t flags;       /* bit0 preserve, bit1 keep_qual, bit2 window active, bit3 processed,
                             bit4 trigger, bit5 had_indel; bits 8-12 BED tags (1<<(8+tag)) */
} cg_column;

typedef struct cg_result {
    uint8_t      *qual_out;        /* caller buffer, >= batch.qual_bytes; same layout as batch.qual */
    cg_bed_event *events;          /* caller buffer or NULL */
    int64_t       events_cap, n_events;
    int64_t       counters[CG_N_COUNTERS];
    cg_column    *columns;         /* caller buffer or NULL (NULL = no dump) */
    int64_t       columns_cap, n_columns;
    /* optional: bytes [0, head_bytes) of the quality layout go to qual_head[] instead of qual_out[] (a region shard's read halo,
     * which lies before the shard's own byte range of a shared output buffer: see cgm_process) */
    uint8_t      *qual_head;
    int64_t       head_bytes;
} cg_result;

typedef struct cg_ctx cg_ctx;

/* ---- life cycle ---------------------------------------------------------------------- */
int         cg_abi_version(void);
int         cg_device_count(void);                                 /* 0 when no usable GPU */
cg_ctx     *cg_create(const cg_params *p, int device, int *err);   /* NULL + *err on failure */
void        cg_destroy(cg_ctx *ctx);
int         cg_set_params(cg_ctx *ctx, const cg_params *p);
const char *cg_strerror(int code);
const char *cg_last_error(const cg_ctx *ctx);                      /* detail of the last failure */
/* run on a caller-owned stream (cudaStream_t as void*), e.g. torch's current stream */
int         cg_set_stream(cg_ctx *ctx, void *cuda_stream);

/* ---- the hot path ---------------------------------------------------------------------
 * cg_process  = upload + run + download: host buffers in, host buffers out (end to end).
 * The split form lets a caller keep a batch resident and time the kernel chain alone.   */
int cg_process(cg_ctx *ctx, const cg_batch *in, cg_result *out);
int cg_upload(cg_ctx *ctx, const cg_batch *in);
int cg_run(cg_ctx *ctx);
int cg_download(cg_ctx *ctx, cg_result *out);
int cg_sync(cg_ctx *ctx);
/* cg_process streams the batch in upload chunks of about this many quality bytes (default 96 MiB, at most 32 chunks);
 * slice i of the kernel chain starts when chunk i has landed.  Results do not depend on it. */
int cg_set_chunk_bytes(cg_ctx *ctx, int64_t bytes);

/* ---- records already in GPU memory: "concatenated BAM fields" ----------------------------
 * What a GPU BAM decoder or a torch pipeline naturally holds; no offset arrays.  Every pointer is device memory of the
 * context's device (NULL is allowed where its count is 0).  Records in input (coordinate-sorted) order, types as cg_batch. */
typedef struct cg_dev_batch {
    int64_t n_reads;
    const int32_t  *tid, *pos;  const uint16_t *flag;  const uint8_t *mapq;
    const int32_t  *l_qseq;     const uint16_t *n_cigar;
    const uint32_t *cigar;  int64_t n_cigar_total;  /* records' CIGARs back to back */
    const uint8_t  *seq;    int64_t seq_len;        /* record i: (l_qseq[i]+1)/2 bytes, BAM nibble order, back to back, each record starts on a byte */
    const uint8_t  *qual;   int64_t qual_len;       /* record i: l_qseq[i] bytes, back to back; qual_len = sum of l_qseq */
} cg_dev_batch;

/* qual_out: device, qual_len bytes, same concatenated layout; may equal in->qual (rewrite in place).
 * out: events, counters and the optional column dump, exactly as for cg_process; out->qual_out and out->qual_head must be NULL.
 * Runs on the context's stream (cg_set_stream).  The three sums (qual_len, seq_len, n_cigar_total) are checked on the device
 * before anything uses them: CG_ERR_BAD_ARG when they disagree, when a count is negative or when a pointer is not device memory
 * of the context's device.  On return the counters and events are on the host; qual_out is written in stream order, so work
 * queued later on the same stream sees it.  The caller's input buffers are free once the stream has passed the call.
 * Afterwards the batch is resident as after cg_upload + cg_run: cg_run may time the chain on it again, and cg_download
 * (qual_out = NULL) re-fetches a longer event list.  cg_last_ms(CG_T_H2D / CG_T_D2H) time the ingest and emit kernels,
 * and cg_last_h2d_bytes reads 0. */
int cg_process_device(cg_ctx *ctx, const cg_dev_batch *in, uint8_t *qual_out, cg_result *out);

/* ---- a stream of records in GPU memory, pushed in chunks of any size (DESIGN.md §3.6) ---------------------------------------------
 * The first call opens a stream on the context; each call appends `in` (the next records of one coordinate-sorted stream; NULL or
 * n_reads 0 allowed) and writes to qual_out (device) the rewritten qualities of the FINAL PREFIX of the stream, back to back in the
 * concatenated layout of cg_process_device: every record not emitted yet, up to the first one that is not final yet.  Records come out
 * in exactly the order they went in, so a producer that keeps names and aux data on its side pairs them up as a FIFO.  last = 1 ends
 * the stream: everything held is flushed and the stream closes.  out gets the BED events and counters of the columns this call owns:
 * the events of all calls concatenated and the counters summed equal one cg_process_device on the whole stream, as do the qualities.
 * out->qual_out, out->qual_head and out->columns must be NULL; a longer event list comes again through cg_download (qual_out = NULL).
 * in's buffers are free once the stream has passed the call, and qual_out may alias in->qual.
 * CG_ERR_BAD_ARG before anything is enqueued, with the context and the open stream unchanged: whatever cg_process_device rejects,
 * qual_cap < held_qual_len + in->qual_len, out->columns set, a -r region in the parameters.  Any later error (sums that disagree, a
 * chunk that breaks the sort order: CG_ERR_UNSORTED, CUDA errors) closes the stream and drops what it held; the context stays usable.
 * While a stream is open, cg_process, cg_process_device, cg_process_window, cg_upload, cg_run, cg_shard_*, cg_set_params and
 * cg_set_stream return CG_ERR_STATE. */
typedef struct cg_stream_out {
    int64_t n_records;        /* records whose final qualities this call wrote: the next n_records of the stream, in stream order */
    int64_t qual_len;         /* bytes written to qual_out = sum of their l_qseq */
    int64_t held_records;     /* records the context now holds for later calls (read halo + not yet final + held-back tail) */
    int64_t held_qual_len;    /* their quality bytes: the next call needs qual_cap >= held_qual_len + its in->qual_len */
} cg_stream_out;
int cg_stream_device(cg_ctx *ctx, const cg_dev_batch *in, int last, uint8_t *qual_out, int64_t qual_cap, cg_result *out, cg_stream_out *so);

/* ---- chained calls: a coordinate-sorted stream of any length in bounded memory ------------
 * (region shards with a read halo, SURVEY.md §8(e): the reference keeps its state in a streaming loop, snp_score.c:1437-1975)
 * The caller cuts the stream wherever it likes.  Let X be the position of the first record AFTER call k (same contig),
 * S <= X the smallest start of a record of call k that reaches column X or beyond (S = X if none).  Then
 *   call k   owns the columns below X:    hi_tid/hi_pos = X, next_lo_pos = S; records ending at or below X are final,
 *   call k+1 = every pileup record seen so far that reaches beyond column S (the read halo, original order and
 *              original qualities) followed by the new records, with lo_pos = S and cnt_pos = X: columns [S,X) are
 *              processed again for the reads still open but neither counted nor reported twice.
 * The two pieces of cross-column state (keep-window chain, depth average) are kept inside the context between calls,
 * as they stand before column S.  Results are bit-identical to one call on the whole stream.                           */
typedef struct cg_window {
    int32_t first;                 /* 1: no earlier call to continue (also after a contig change): state is reset and lo/cnt are
                                      ignored; 2: state is reset but lo/cnt apply (a region shard started on its own, see below) */
    int32_t lo_tid, lo_pos;        /* columns of lo_tid below lo_pos belong to earlier calls (ignored when first) */
    int32_t cnt_pos;               /* columns of lo_tid in [lo_pos, cnt_pos) were counted by the previous call */
    int32_t hi_tid, hi_pos;        /* columns at/after (hi_tid, hi_pos) are left to the next call; hi_tid < 0: none */
    int32_t next_lo_pos;           /* the next call's lo_pos (contig hi_tid); ignored when hi_tid < 0 */
} cg_window;
/* cg_process restricted to the window's columns; the records the caller treats as final are its own business */
int cg_process_window(cg_ctx *ctx, const cg_batch *in, const cg_window *win, cg_result *out);

/* Region shards of ONE contig on several contexts / GPUs at once.  The column stage (2/3 of the time) never depends on the
 * carried state and the sparse passes only do where a keep window is still open at the shard's first column or the -P
 * over-depth test can fire, so shards may start on their own (first = 2: reset state, halo and lo/cnt as usual) and be
 * checked afterwards, in position order: shard r exports the state it saved at shard r+1's lo_pos; if that state is neutral for
 * shard r+1 (no open window reaching lo_pos; depth average out of play) shard r+1's results stand, otherwise shard r+1 imports
 * it and runs again with first = 0 (and its own exported state is then the one to hand on).  Bit-identical to one call. */
#define CG_CARRY_BYTES 128
int cg_carry_export(cg_ctx *ctx, void *buf);                       /* CG_ERR_STATE unless the last window call had hi_tid >= 0 */
int cg_carry_import(cg_ctx *ctx, const void *buf);                 /* what the next cg_process_window(first = 0) resumes from */
/* Would the last window call of ctx (run with first = 2 at (tid, lo_pos)) have given the same results resuming from buf?
 * 1 yes; 0 no: a keep window is still open there (run it again from buf); -1 no: the depth average is in play (-P can fire) —
 * then only a chain run in position order from the contig's first shard hands on exact depth sums */
int cg_carry_is_neutral(const cg_ctx *ctx, const void *buf, int32_t tid, int32_t lo_pos);
/* pos + reference span of every record (pos itself for records outside the pileup): what a host needs to plan shards and halos */
void cg_batch_ends(const cg_batch *in, int32_t *end_out);

/* The same shards without speculation: every shard gets the TRUE state of its left neighbour, yet only a sliver of the work is serial.
 * A shard's work is split in three (cg_device.cu, slice_A / slice_B):
 *   cg_shard_begin   upload, pileup, consensus, column decisions, STR searches: nothing here depends on carried state.  All shards
 *                    run it at the same time (window as for cg_process_window; first = 2 is read as 0);
 *   cg_shard_carry   state in (NULL for a shard that starts a contig) -> depth prefix sums + epochs and the keep-window chain over the
 *                    shard's columns below its right neighbour's first column -> state out.  Shard after shard, but tiny;
 *   cg_shard_end     over-depth test, window painting, per-read rewrite, downloads: all shards at the same time again.
 * Results are bit-identical to one call on the whole batch at every option level, -1/-3/-5 (depth average) included.
 * `in` must stay valid until cg_shard_end returns. */
int cg_shard_begin(cg_ctx *ctx, const cg_batch *in, const cg_window *win, cg_result *out);
int cg_shard_carry(cg_ctx *ctx, const void *carry_in, void *carry_out);     /* CG_CARRY_BYTES each; carry_out may be NULL */
int cg_shard_end(cg_ctx *ctx, cg_result *out);

/* ---- one batch over several GPUs (crumble_b200/csrc/cg_multi.c) -------------------------------------------------------------------
 * As many region shards as devices, of about equal size, cut at record boundaries; one host thread and one context per device; the three
 * cg_shard_* phases above; every device downloads its own byte range of out->qual_out.  Same results as cg_process / cg_process_window,
 * in the same buffers (the per-column dump is not available).  cgm_process_window keeps the state between the calls of a chain inside
 * the cg_multi object, as a context does for cg_process_window. */
typedef struct cg_multi cg_multi;
cg_multi   *cgm_create(const cg_params *p, int n_devices, const int *devices /* NULL: 0 .. n_devices-1 */, int *err);
void        cgm_destroy(cg_multi *m);
int         cgm_n_devices(const cg_multi *m);
int         cgm_process(cg_multi *m, const cg_batch *in, cg_result *out);
int         cgm_process_window(cg_multi *m, const cg_batch *in, const cg_window *win, cg_result *out);
const char *cgm_last_error(const cg_multi *m);
float       cgm_last_ms(const cg_multi *m);                 /* slowest shard's device time of the last call */
int64_t     cgm_last_h2d_bytes(const cg_multi *m);
cg_ctx     *cgm_context(cg_multi *m, int i);                /* borrowed */
int64_t     cgm_events(const cg_multi *m, cg_bed_event *buf, int64_t cap);   /* the last call's BED events again; returns their number */

/* measurement helpers */
enum { CG_T_TOTAL = 0, CG_T_TILES, CG_T_COLUMNS, CG_T_FLAGGED, CG_T_DEPTH, CG_T_CHAIN, CG_T_REWRITE, CG_T_CELLS, CG_T_EVENTS, CG_T_H2D, CG_T_D2H, CG_N_TIMERS };
float   cg_last_ms(const cg_ctx *ctx, int which);        /* CUDA-event time of the last cg_run / copies */
int64_t cg_last_launches(const cg_ctx *ctx);             /* kernels launched by the last cg_run */
int64_t cg_last_h2d_bytes(const cg_ctx *ctx);            /* bytes the last cg_upload / cg_process / cg_process_window copied to the device */
int64_t cg_algorithmic_bytes(const cg_batch *in);        /* SURVEY §8(d): sum ceil(l/2)+2l+4*n_cigar+16 over pileup reads */
int64_t cg_aligned_bases(const cg_batch *in);            /* sum l_qseq over records entering the pileup */
int64_t cg_n_columns(const cg_ctx *ctx);                 /* covered reference columns in the resident batch */

/* ---- host batcher: decoded records -> pinned SoA (replaces pileup_callback's bam_dup1
 * into RB-trees, snp_score.c:1113-1153) ------------------------------------------------ */
/* Host memory for buffers that cross PCIe (cg_result.qual_out, batches laid out by the caller): page-locked when a device exists, so that
 * cg_process can overlap its copies with the kernels; plain malloc otherwise.  Free with cg_host_free. */
void *cg_host_alloc(size_t bytes);
void  cg_host_free(void *p);

typedef struct cg_batch_builder cg_batch_builder;
cg_batch_builder *cgb_create(int pinned);
void  cgb_destroy(cg_batch_builder *b);
void  cgb_reset(cg_batch_builder *b);
/* optional: capacity for this many records / quality bytes / CIGAR operations up front (pinned memory is costly to grow) */
int   cgb_reserve(cg_batch_builder *b, int64_t n_reads, int64_t qual_bytes, int64_t n_cigar);
/* one record; the pointers are BAM-layout fields (bam1_t core + data) */
int   cgb_add(cg_batch_builder *b, int32_t tid, int32_t pos, uint16_t flag, uint8_t mapq,
              int32_t l_qseq, uint32_t n_cigar, const uint32_t *cigar, const uint8_t *seq4, const uint8_t *qual);
/* every record of an uncompressed BAM stream (BAM\1 magic + header + records) */
int   cgb_add_bam_stream(cg_batch_builder *b, const uint8_t *buf, size_t len);
int   cgb_finish(cg_batch_builder *b, cg_batch *out);    /* out points into the builder */
/* build the compact planes (cg_batch.seq2 / seq_exc / qualp) of everything added so far, with `threads` workers (0 = all cores);
 * the next cgb_finish hands them out.  Optional: costs one pass over the base data on the host, saves two thirds of the upload. */
int   cgb_pack(cg_batch_builder *b, int threads);
int64_t cgb_bytes(const cg_batch_builder *b);

#ifdef __cplusplus
}
#endif
#endif
