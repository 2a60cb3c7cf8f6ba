/*
 * crumble_host.h — host-side option block and driver entry points of the crumble CLI
 * built on the GPU path.  crumble_opts = the device-relevant cg_params plus the
 * options that only the host uses (reference cram_lossy_params, snp_score.c:185-226).
 */
#ifndef CRUMBLE_HOST_H
#define CRUMBLE_HOST_H
#include <stdio.h>
#include <stdint.h>
#include "htslib/sam.h"
#include "../../include/crumble_gpu.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct crumble_opts {
    cg_params p;
    char *region;                 /* -r */
    char *bed_fn;                 /* -R */
    FILE *bed_fp;                 /* -b */
    uint8_t *aux_whitelist;       /* -t: 8192-byte bitmap over 2-char tags, or NULL */
    uint8_t *aux_blacklist;       /* -T */
    int BD_low, BD_mid, BD_high;  /* -e -f -g */
    int BI_low, BI_mid, BI_high;  /* -E -F -G */
    int device;                   /* CUDA device ordinal */
    int64_t counters[CG_N_COUNTERS];
    float last_device_ms;
} crumble_opts;

void crumble_opts_default(crumble_opts *o);
/* getopt loop of the reference main() (snp_score.c:2199-2504). Returns 0, or 1 = print
 * usage(stderr) and exit 1, or 2 = -h given.  *optind_out = index of first non-option. */
int  crumble_parse_args(crumble_opts *o, int argc, char **argv, htsFormat *in_fmt, htsFormat *out_fmt, int *optind_out);
void crumble_usage(FILE *fp);
void crumble_print_params(const crumble_opts *o);          /* -v block, snp_score.c:2506-2540 */
void crumble_print_counters(const crumble_opts *o);        /* -v block, snp_score.c:2650-2666 */
void crumble_purge_tags(const crumble_opts *o, bam1_t *b); /* snp_score.c:989-1054 */
cg_bed_reg *crumble_bed_load(const char *fn, bam_hdr_t *header, int *nreg);   /* bed.c:42-103 */
int  transcode_gpu(crumble_opts *o, samFile *in, samFile *out, bam_hdr_t *header, hts_itr_t *h_iter);
/* pos + cg_pileup_span (cg_core.h): a pileup record's end (exclusive), pos itself for any other record (cg_host.cpp) */
int32_t cg_record_end(int32_t tid, int32_t pos, uint16_t flag, const uint32_t *cigar, int n_cigar);
int  crumble_main(int argc, char **argv);

#ifdef __cplusplus
}
#endif
#endif
