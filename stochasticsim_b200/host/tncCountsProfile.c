/*
 * tncCountsProfile -- drop-in replacement for the reference program of the same name.
 *
 *   tncCountsProfile <target fasta>            (same argv, stdout and exit codes as the reference)
 *   tncCountsProfile <genome fasta> <bed>      (extension, BASELINE config 3: the counts the reference gives on the FASTA that
 *                                               `bedtools getfasta -fi <genome> -bed <bed>` would write, without writing it)
 *   tncCountsProfile <genome fasta> <bed> --per-interval
 *                                              (extension: one row per BED interval, in BED order -- "chrom start end" and the 32
 *                                               counts the reference gives on the FASTA getfasta writes for that interval alone,
 *                                               after a "#chrom start end ACA ... TTT" header line; tab separated)
 *
 * Replaces main() of tncCountsProfile.c:366-485.  This file stays in C and only does what a host
 * has to do -- open/map the file, hand byte ranges to the GPU(s), print the 32 lines.  All
 * counting happens in libssb200.so (CUDA, sm_100a); there is no CPU fallback: without a B200
 * the program fails with exit status 3.
 *
 * Environment (the reference reads none; these only select hardware):
 *   SSB_GPUS=N      spread the file over the first N GPUs by byte range (default 1); the per-GPU
 *                   count vectors are combined with ONE NCCL all-reduce of 64 int64.  With a BED the
 *                   intervals are split into N ranges instead; per interval each GPU writes its own rows.
 *   SSB_DEVICE=i    first device ordinal (default 0).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>
#include <fcntl.h>
#include <unistd.h>
#include <pthread.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include "ssb200.h"

int ssb_nccl_init_all(ssb_ctx **ctxs, int n, void **comms_out);
int ssb_tnc_allreduce_group(ssb_ctx **ctxs, void **comms, int64_t **d_counts64, int n);
void ssb_nccl_destroy_all(void **comms, int n);

typedef struct {
    ssb_ctx *ctx;
    const uint8_t *base;
    size_t off, len;
    ssb_tnc_carry carry_in;
    int64_t counts[64];
    int rc;
    /* BED mode: the whole genome text goes to every GPU, the intervals [first, last) are this GPU's share */
    const ssb_fasta_contig *contigs; size_t n_contigs; const ssb_bed_interval *iv; size_t n_iv, first, last; size_t n_all;
    int64_t *rows;     /* --per-interval: 64 counters per interval of [first, last) (host), instead of `counts` */
} shard_t;

static void *shard_main(void *arg)
{
    shard_t *s = (shard_t *)arg;
    if (!s->iv) { s->rc = ssb_tnc_count_host(s->ctx, s->base + s->off, s->len, &s->carry_in, NULL, s->counts); return NULL; }
    void *d_fa = NULL, *d_cnt = NULL;
    const size_t cnt_bytes = s->rows ? (s->last - s->first) * 64 * sizeof(int64_t) : sizeof s->counts;
    s->rc = ssb_dev_alloc(s->ctx, s->n_all + 64, &d_fa);
    if (!s->rc) s->rc = ssb_dev_alloc(s->ctx, cnt_bytes, &d_cnt);
    if (!s->rc) s->rc = ssb_memcpy_h2d(s->ctx, d_fa, s->base, s->n_all);
    if (!s->rc) s->rc = ssb_memset_dev(s->ctx, d_cnt, 0, cnt_bytes);
    if (!s->rc && s->rows) s->rc = ssb_tnc_count_intervals_device(s->ctx, (const uint8_t *)d_fa, s->n_all, s->contigs, s->n_contigs, s->iv, s->n_iv, s->first, s->last, (int64_t *)d_cnt);
    else if (!s->rc) s->rc = ssb_tnc_count_bed_device(s->ctx, (const uint8_t *)d_fa, s->n_all, s->contigs, s->n_contigs, s->iv, s->n_iv, s->first, s->last, (int64_t *)d_cnt);
    if (!s->rc) s->rc = ssb_memcpy_d2h(s->ctx, s->rows ? (void *)s->rows : (void *)s->counts, d_cnt, cnt_bytes);
    if (!s->rc) s->rc = ssb_sync(s->ctx);
    if (d_fa) ssb_dev_free(s->ctx, d_fa);
    if (d_cnt) ssb_dev_free(s->ctx, d_cnt);
    return NULL;
}

/* BED rows "chrom<TAB>start<TAB>end[...]" -> intervals, chrom looked up in the FASTA index; lines starting with '#', "track" or
 * "browser" are skipped, unknown contigs are an error */
static ssb_bed_interval *load_bed(const char *fn, const char **names, const uint32_t *name_lens, size_t n_contigs, size_t *n_out)
{
    FILE *f = fopen(fn, "r");
    if (!f) return NULL;
    size_t n = 0, cap = 1024; ssb_bed_interval *v = malloc(cap * sizeof *v);
    char *line = NULL; size_t lcap = 0;
    while (getline(&line, &lcap, f) != -1) {
        if (line[0] == '#' || line[0] == '\n' || !strncmp(line, "track", 5) || !strncmp(line, "browser", 7)) continue;
        char *t1 = strchr(line, '\t'); if (!t1) continue;
        const size_t nl = (size_t)(t1 - line);
        long long a = 0, b = 0;
        if (sscanf(t1 + 1, "%lld\t%lld", &a, &b) != 2) continue;
        int c = -1;
        for (size_t i = 0; i < n_contigs; i++) if (name_lens[i] == nl && !memcmp(names[i], line, nl)) { c = (int)i; break; }
        if (c < 0) { fprintf(stderr, "tncCountsProfile: BED contig %.*s is not in the FASTA\n", (int)nl, line); free(v); fclose(f); *n_out = 0; return NULL; }
        if (n == cap) { cap *= 2; v = realloc(v, cap * sizeof *v); }
        v[n].contig = c; v[n].reserved = 0; v[n].start = a; v[n].end = b; n++;
    }
    free(line); fclose(f);
    *n_out = n;
    return v;
}

int main(int argc, char **argv)
{
    /* tncCountsProfile.c:380-382: fopen failure (or no argument) -> silent exit(EXIT_FAILURE) */
    int fd = argv[1] ? open(argv[1], O_RDONLY) : -1;
    if (fd < 0) exit(EXIT_FAILURE);
    struct stat sb;
    if (fstat(fd, &sb) != 0) exit(EXIT_FAILURE);
    size_t n = (size_t)sb.st_size;
    const uint8_t *data = (const uint8_t *)"";
    if (n) {
        data = mmap(NULL, n, PROT_READ, MAP_PRIVATE, fd, 0);
        if (data == MAP_FAILED) {
            /* not mappable (pipe, /dev/stdin): slurp it */
            size_t cap = 1 << 20, len = 0; uint8_t *buf = malloc(cap); ssize_t r;
            while ((r = read(fd, buf + len, cap - len)) > 0) { len += (size_t)r; if (len == cap) { cap *= 2; buf = realloc(buf, cap); } }
            data = buf; n = len;
        } else madvise((void *)data, n, MADV_SEQUENTIAL);
    } else {
        /* st_size 0 may still be a pipe */
        size_t cap = 1 << 20, len = 0; uint8_t *buf = malloc(cap); ssize_t r;
        while ((r = read(fd, buf + len, cap - len)) > 0) { len += (size_t)r; if (len == cap) { cap *= 2; buf = realloc(buf, cap); } }
        data = buf; n = len;
    }
    if (n && memchr(data, 0, n)) {
        fprintf(stderr, "tncCountsProfile: NUL byte in input is not supported (see DESIGN.md)\n");
        return 2;
    }

    int ngpu = getenv("SSB_GPUS") ? atoi(getenv("SSB_GPUS")) : 1;
    int dev0 = getenv("SSB_DEVICE") ? atoi(getenv("SSB_DEVICE")) : 0;
    if (ngpu < 1) ngpu = 1;
    if (ngpu > 64) ngpu = 64;
    if ((size_t)ngpu > n / 4096 + 1) ngpu = (int)(n / 4096 + 1);
    /* BED mode (second argument) */
    ssb_fasta_contig *contigs = NULL; ssb_bed_interval *iv = NULL; size_t n_contigs = 0, n_iv = 0;
    const char **names = NULL; uint32_t *nlens = NULL;
    int64_t *rows = NULL;                                     /* --per-interval: 64 counters per interval */
    if (argc > 2 && argv[2]) {
        int rc = ssb_fasta_index(data, n, NULL, NULL, NULL, 0, &n_contigs);
        if (rc) { fprintf(stderr, "tncCountsProfile: %s: a record's lines are not all as wide as its first one (%s)\n", argv[1], ssb_strerror(rc)); return 3; }
        contigs = malloc((n_contigs + 1) * sizeof *contigs);
        names = malloc((n_contigs + 1) * sizeof *names); nlens = malloc((n_contigs + 1) * sizeof *nlens);
        ssb_fasta_index(data, n, contigs, names, nlens, n_contigs, &n_contigs);
        iv = load_bed(argv[2], names, nlens, n_contigs, &n_iv);
        if (!iv) exit(EXIT_FAILURE);
        if ((size_t)ngpu > n_iv / 64 + 1) ngpu = (int)(n_iv / 64 + 1);
        if (argc > 3 && argv[3] && !strcmp(argv[3], "--per-interval")) {
            rows = malloc((n_iv + 1) * 64 * sizeof *rows);
            if (!rows) { fprintf(stderr, "tncCountsProfile: out of host memory for %zu rows\n", n_iv); return 3; }
        }
    }

    shard_t sh[64]; ssb_ctx *ctxs[64];
    memset(sh, 0, sizeof sh);
    for (int g = 0; g < ngpu; g++) {
        int rc = ssb_ctx_create(dev0 + g, &ctxs[g]);
        if (rc) { fprintf(stderr, "tncCountsProfile: device %d: %s\n", dev0 + g, ssb_strerror(rc)); return 3; }
        sh[g].ctx = ctxs[g]; sh[g].base = data;
        sh[g].off = (n / (size_t)ngpu * (size_t)g) & ~(size_t)31;
        if (iv) { sh[g].iv = iv; sh[g].n_iv = n_iv; sh[g].contigs = contigs; sh[g].n_contigs = n_contigs; sh[g].n_all = n;
                  sh[g].first = n_iv * (size_t)g / (size_t)ngpu; sh[g].last = n_iv * (size_t)(g + 1) / (size_t)ngpu;
                  if (rows) sh[g].rows = rows + sh[g].first * 64; }
    }
    for (int g = 0; g < ngpu; g++) {
        sh[g].len = (g + 1 < ngpu ? sh[g + 1].off : n) - sh[g].off;
        /* scanner state at the shard start, from the bytes before it (no counting) */
        if (g && !iv) ssb_tnc_carry_after(data, sh[g].off, NULL, &sh[g].carry_in);
    }
    pthread_t th[64];
    for (int g = 1; g < ngpu; g++) pthread_create(&th[g], NULL, shard_main, &sh[g]);
    shard_main(&sh[0]);
    for (int g = 1; g < ngpu; g++) pthread_join(th[g], NULL);
    for (int g = 0; g < ngpu; g++)
        if (sh[g].rc) { fprintf(stderr, "tncCountsProfile: %s (%s)\n", ssb_strerror(sh[g].rc), ssb_last_error(ctxs[g])); return 3; }
    if (rows) {
        /* header: the 32 names in the order of the reference's output lines (as ssb_tnc_format prints them) */
        char names32[4096]; int64_t zero[64] = {0};
        const int nw = ssb_tnc_format(zero, names32, sizeof names32);
        if (nw < 0) return 3;
        printf("#chrom\tstart\tend");
        for (char *p = names32; p < names32 + nw; p = strchr(p, '\n') + 1) printf("\t%.*s", (int)(strchr(p, '\t') - p), p);
        printf("\n");
        /* the GPUs wrote their ranges of rows side by side: print them in BED order */
        for (size_t i = 0; i < n_iv; i++) {
            int64_t o[32];
            ssb_tnc_fold32(rows + i * 64, o);
            printf("%.*s\t%lld\t%lld", (int)nlens[iv[i].contig], names[iv[i].contig], (long long)iv[i].start, (long long)iv[i].end);
            for (int k = 0; k < 32; k++) printf("\t%lld", (long long)o[k]);
            printf("\n");
        }
        for (int g = 0; g < ngpu; g++) ssb_ctx_destroy(ctxs[g]);
        return 0;
    }

    int64_t total[64];
    if (ngpu == 1) memcpy(total, sh[0].counts, sizeof total);
    else {
        /* the path's only collective: all-reduce the 64 counters over NVLink */
        void *comms[64]; int64_t *dc[64];
        int rc = ssb_nccl_init_all(ctxs, ngpu, comms);
        if (rc) { fprintf(stderr, "tncCountsProfile: %s (%s)\n", ssb_strerror(rc), ssb_last_error(ctxs[0])); return 3; }
        for (int g = 0; g < ngpu; g++) {
            if (ssb_dev_alloc(ctxs[g], sizeof total, (void **)&dc[g]) || ssb_memcpy_h2d(ctxs[g], dc[g], sh[g].counts, sizeof total)) return 3;
        }
        rc = ssb_tnc_allreduce_group(ctxs, comms, dc, ngpu);
        if (rc) { fprintf(stderr, "tncCountsProfile: %s (%s)\n", ssb_strerror(rc), ssb_last_error(ctxs[0])); return 3; }
        if (ssb_memcpy_d2h(ctxs[0], total, dc[0], sizeof total) || ssb_sync(ctxs[0])) return 3;
        for (int g = 0; g < ngpu; g++) { ssb_sync(ctxs[g]); ssb_dev_free(ctxs[g], dc[g]); }
        ssb_nccl_destroy_all(comms, ngpu);
    }
    char out[4096];
    int w = ssb_tnc_format(total, out, sizeof out);           /* tncCountsProfile.c:452-483 */
    if (w < 0) return 3;
    fwrite(out, 1, (size_t)w, stdout);
    for (int g = 0; g < ngpu; g++) ssb_ctx_destroy(ctxs[g]);
    return 0;
}
