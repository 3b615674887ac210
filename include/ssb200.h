/*
 * ssb200.h -- C ABI of libssb200.so: the B200 (sm_100a) implementation of the two
 * data-parallel hot paths of stochasticSim.
 *
 * The reference has no library/FFI boundary: its two hot paths are standalone C
 * programs whose interface is argv + files (SURVEY.md 8b).  The drop-in boundary is
 * therefore the pair of executables built from stochasticsim_b200/host/ (same argv,
 * same outputs, same exit codes); those mains stay in C and reach the GPU only
 * through the entry points below.  Each entry point names the reference code it
 * replaces.
 *
 * Conventions: plain pointers and sizes, caller-owned buffers, one ssb_ctx per
 * device, no global state, return 0 on success or a negative SSB_E_* code
 * (ssb_strerror() gives the text).  There is NO CPU fallback anywhere behind this
 * header: without a usable CUDA device ssb_ctx_create() fails.
 */
#ifndef SSB200_H
#define SSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSB_ABI_VERSION 2

enum {
    SSB_OK            =  0,
    SSB_E_CUDA        = -1,   /* CUDA runtime error (text kept in the ctx)              */
    SSB_E_NODEVICE    = -2,   /* no CUDA device / wrong architecture                    */
    SSB_E_ARG         = -3,   /* bad argument                                           */
    SSB_E_NOMEM       = -4,
    SSB_E_FORMAT      = -5,   /* input violates a documented precondition (see DESIGN.md) */
    SSB_E_UNSORTED    = -6,   /* SAM input not coordinate sorted                        */
    SSB_E_DEPTH       = -7,   /* pileup deeper than MAX_PILEUP_SIZE (stochasticSpike.c:38) */
    SSB_E_REF         = -8,   /* contig missing from / longer than the reference FASTA  */
    SSB_E_STATE       = -9,   /* call order violated                                    */
    SSB_E_NCCL        = -10,
    SSB_E_SHARD       = -11,  /* a shard's alignment lines do not match its coordinate range / halo too small */
    SSB_E_PEER        = -12   /* another shard of the cooperative run failed                                  */
};

typedef struct ssb_ctx ssb_ctx;

int         ssb_abi_version(void);
const char *ssb_strerror(int code);
/* Last CUDA/NCCL error text recorded in this context ("" if none). */
const char *ssb_last_error(const ssb_ctx *ctx);

/* Binds to CUDA device `device`; fails with SSB_E_NODEVICE unless it is compute capability 10.x. */
int  ssb_ctx_create(int device, ssb_ctx **out);
void ssb_ctx_destroy(ssb_ctx *ctx);
/* Name, SM count, memory of the bound device (any pointer may be NULL). */
int  ssb_ctx_device_info(const ssb_ctx *ctx, char *name, size_t name_cap, int *sm_count, size_t *total_mem);

/* Plumbing shared by the C mains, tests and bench (pinned host / device buffers, copies on the
 * context's stream, device timing).  Nothing here computes anything. */
int  ssb_host_alloc(ssb_ctx *ctx, size_t bytes, void **out);      /* pinned */
void ssb_host_free(ssb_ctx *ctx, void *p);
int  ssb_dev_alloc(ssb_ctx *ctx, size_t bytes, void **out);
void ssb_dev_free(ssb_ctx *ctx, void *p);
int  ssb_memcpy_h2d(ssb_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);   /* async on ctx stream */
int  ssb_memcpy_d2h(ssb_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);   /* async on ctx stream */
int  ssb_memset_dev(ssb_ctx *ctx, void *dst_dev, int value, size_t bytes);
int  ssb_sync(ssb_ctx *ctx);
/* CUDA-event stopwatch on the context's stream: start, stop -> elapsed device milliseconds. */
int  ssb_timer_start(ssb_ctx *ctx);
int  ssb_timer_stop(ssb_ctx *ctx, float *ms);
/* Number of kernels this library launched through this context since creation. */
uint64_t ssb_kernel_launches(const ssb_ctx *ctx);
/* Optional per-kernel device timing: when enabled every launch of the kernels below is bracketed by
 * CUDA events on its own stream; ssb_profile_read() synchronises and returns the summed duration
 * and the number of launches of one kernel slot (and optionally resets them). */
enum { SSB_PROF_TNC_SCAN = 0, SSB_PROF_TNC_FIXUP = 1, SSB_PROF_SPIKE_PARSE = 2, SSB_PROF_SPIKE_EMIT = 3,
       SSB_PROF_SPIKE_CHAIN = 4, SSB_PROF_SPIKE_OTHER = 5, SSB_PROF_SPIKE_TALLY = 6, SSB_PROF_TNC_INTERVALS = 7 };
int  ssb_profile_enable(ssb_ctx *ctx, int on);
int  ssb_profile_read(ssb_ctx *ctx, int slot, double *total_ms, uint64_t *launches, int reset);

/* ------------------------------------------------------------------------------------------
 * Hot path 2: trinucleotide-context scan.
 * Replaces: tncCountsProfile.c:391-447 (the getline/3-byte-window loop) and incCtx
 * (tncCountsProfile.c:105-363).  counts64[] is indexed 16*a+4*b+c with A<C<G<T
 * (tncCountsProfile.c:14-77), exactly the reference's `long ctxCnt[64]`.
 * ------------------------------------------------------------------------------------------ */

/* Scanner state carried from one piece of a FASTA to the next, so a file can be cut anywhere
 * (host chunks, or one shard per GPU).  A zeroed struct means "start of file". */
typedef struct ssb_tnc_carry {
    uint8_t started;        /* 0 = start of file (the other fields are ignored)                    */
    uint8_t prev[3];        /* the 3 bytes preceding this piece                                     */
    uint8_t carry;          /* last byte of the nearest kept, newline-terminated line; 0 = none    */
    uint8_t frag_nonempty;  /* the piece starts inside a line that already has >= 1 byte            */
    uint8_t frag_first;     /* first byte of that line                                              */
    uint8_t frag_has_base;  /* that line already holds an upper-case A/C/G/T                        */
} ssb_tnc_carry;

/* Device-resident piece: d_fasta[0..n) (n < 2^32) in HBM.  Adds this piece's windows to the 64
 * device counters d_counts64 (int64, caller zeroes them once).  carry_in may be NULL (= start of
 * file); carry_out may be NULL.  Asynchronous on the context's stream except for carry_out,
 * which synchronises.  This is the call bench.py times for `value`. */
int ssb_tnc_count_device(ssb_ctx *ctx, const uint8_t *d_fasta, size_t n,
                         const ssb_tnc_carry *carry_in, ssb_tnc_carry *carry_out,
                         int64_t *d_counts64);

/* Host-resident FASTA of any size: streams it through double-buffered pinned chunks on two
 * copy/compute streams and returns the 64 totals in counts64 (host, overwritten).  `fasta` may be
 * pageable or pinned.  This is what the tncCountsProfile main calls, and bench.py's `e2e`. */
int ssb_tnc_count_host(ssb_ctx *ctx, const uint8_t *fasta, size_t n,
                       const ssb_tnc_carry *carry_in, ssb_tnc_carry *carry_out,
                       int64_t counts64[64]);

/* The state a scanner is in after consuming fasta[0..n) from `carry_in`, computed on the host
 * WITHOUT counting anything: used to cut a FASTA into independent shards (one per GPU). */
int ssb_tnc_carry_after(const uint8_t *fasta, size_t n, const ssb_tnc_carry *carry_in, ssb_tnc_carry *carry_out);

/* Sum the 64 device counters across ranks (the path's only collective).  `nccl_comm` is an
 * ncclComm_t created by the caller; the reduction runs on the context's stream. */
int ssb_tnc_allreduce(ssb_ctx *ctx, void *nccl_comm, int64_t *d_counts64);

/* BED-restricted scan (BASELINE.json configs[2]: "tncCountsProfile over whole GRCh38 FASTA restricted to a synthetic exome BED").
 * The reference has no BED input: the result is DEFINED as what tncCountsProfile.c:391-447 counts on the FASTA that holds, per
 * interval in BED order, one header line and the interval's bases on one line (the shape `bedtools getfasta` writes); that
 * FASTA is built on the device and scanned by the same exact kernels.  contigs[] is a .fai-style index of the genome text
 * (ssb_fasta_index makes it); interval.contig indexes it.  Counts the windows of intervals [first, last) -- including the one
 * straddling window the reference sees between the nearest kept earlier interval and the first of this range -- so that the
 * counts of a partition of [0, n_intervals) add up to the whole (one range per GPU, then ssb_tnc_allreduce). */
typedef struct ssb_fasta_contig { uint64_t seq_off; int64_t len; uint32_t line_bases, line_bytes; } ssb_fasta_contig;
typedef struct ssb_bed_interval { int32_t contig, reserved; int64_t start, end; } ssb_bed_interval;      /* 0-based, half open */
/* SSB_E_FORMAT when a record's sequence lines are not all as wide as its first one (only the last may be shorter). */
int ssb_fasta_index(const uint8_t *fasta, size_t n, ssb_fasta_contig *out, const char **names, uint32_t *name_lens, size_t cap, size_t *n_out);
int ssb_tnc_count_bed_device(ssb_ctx *ctx, const uint8_t *d_fasta, size_t n, const ssb_fasta_contig *contigs, size_t n_contigs,
                             const ssb_bed_interval *intervals, size_t n_intervals, size_t first, size_t last, int64_t *d_counts64);

/* Per-interval counts: adds the windows of each interval [first, last), on its own, to row (i - first) of d_rows
 * (int64[(last - first) * 64], device, caller zeroes it; counts64 layout per row).  Row i is DEFINED as what
 * tncCountsProfile.c:391-447 counts on the FASTA `bedtools getfasta` writes for interval i alone: one header line, then the
 * interval's bases on one line.  That reduces to: a window counts at every position p in [start, end-2) where bases p, p+1
 * and p+2 are all upper-case A/C/G/T; line terminators of the genome text are skipped through the index.  So rows do not
 * depend on BED order, duplicates or overlaps, and they do NOT add up to ssb_tnc_count_bed_device's total: that one also
 * counts the one straddling window the reference sees between consecutive kept intervals.  The genome text is read in
 * place (no extracted FASTA).  d_fasta is 16-byte aligned, of any size (64-bit offsets throughout); contigs[] is its index
 * (ssb_fasta_index).  Refusals as in ssb_tnc_count_bed_device: end < start -> SSB_E_ARG; an interval outside its contig, or
 * an index that does not describe the file -> SSB_E_FORMAT.  Asynchronous except for the error check. */
int ssb_tnc_count_intervals_device(ssb_ctx *ctx, const uint8_t *d_fasta, size_t n, const ssb_fasta_contig *contigs, size_t n_contigs,
                                   const ssb_bed_interval *intervals, size_t n_intervals, size_t first, size_t last, int64_t *d_rows);

/* The reference's fold of the 64 contexts into its 32 output lines (tncCountsProfile.c:452-483): context + reverse
 * complement, in the order of its printf block. */
void ssb_tnc_fold32(const int64_t counts64[64], int64_t out32[32]);

/* The reference's 32-line stdout (tncCountsProfile.c:452-483): "CTX\t%ld\n", the 32 values of ssb_tnc_fold32, fixed
 * order.  Returns bytes written (excluding NUL) or SSB_E_ARG if cap is short. */
int ssb_tnc_format(const int64_t counts64[64], char *dst, size_t cap);

/* ------------------------------------------------------------------------------------------
 * Hot path 1: stochastic spike-in.
 * Replaces the pileup loop of stochasticSpike.c:1129-1623 (read filter read_bam :243-268, RNG
 * helpers :283-360, overlap handling :363-432, attemptToMutateBase :526-904, write-out
 * :1272-1285/:1362-1371, target advance :1578-1619) for SAM TEXT input.  The host main keeps the
 * reference's argv/file handling (stochasticsim_b200/host/stochasticSpike.c) and calls in here.
 *
 * One ssb_spike object = one reference genome on one device.  A run takes the alignment lines of
 * a coordinate-sorted SAM (header removed), the `.spike` targets in FILE order and the seed, and
 * produces: the output alignment lines (kept reads ordered by end position, bases substituted,
 * QUAL untouched), one result per target (everything a truth.vcf target / NO_COVERAGE line needs),
 * the SEQ_ERROR records and the five counters of the stats block (stochasticSpike.c:1668).
 * ------------------------------------------------------------------------------------------ */
typedef struct ssb_spike ssb_spike;

typedef struct ssb_contig {
    const char    *name;      /* @SQ SN, in header order: index = tid (sam_hdr_name2tid)            */
    int64_t        len;       /* bases available in `seq`                                            */
    const uint8_t *seq;       /* host pointer: the contig as faidx_fetch_seq64 returns it (newlines
                                 stripped, CASE PRESERVED), or NULL when the FASTA lacks the contig */
} ssb_contig;

/* One valid `.spike` record as getNextTarget() parses it (stochasticSpike.c:98-158, struct :88-94). */
typedef struct ssb_target {
    int32_t c_tid;            /* sam_hdr_name2tid(contig), -1 when unknown                           */
    int32_t reserved;
    int64_t locus;            /* atol(POS) - 1                                                       */
    uint8_t base;             /* first byte of the ALT field                                         */
    uint8_t pad[3];
    float   af;               /* (float)atof(AF)                                                     */
} ssb_target;

enum { SSB_T_HIT = 0, SSB_T_NOCOV = 1, SSB_T_NOCOV_SILENT = 2, SSB_T_TAIL = 3,
       SSB_T_ELSEWHERE = 4 /* sharded runs: the target is consumed at a locus another shard owns */ };
enum { SSB_F_NONE = 0, SSB_F_PASS = 1, SSB_F_MASKED = 2, SSB_F_MASKED_OVL = 3, SSB_F_UNDETECTED = 4 };

typedef struct ssb_target_result {
    int32_t status;           /* SSB_T_*: HIT = spiked at a covered locus; NOCOV = passed over, line
                                 printed; NOCOV_SILENT = passed over but stochasticSpike.c:1603 suppresses
                                 the line; TAIL = left over after the last covered locus (:1630-1646) */
    int32_t at_tid;           /* covered locus where the target was consumed (HIT: the target)       */
    int64_t at_pos;
    int64_t locus_index;      /* ordinal of that covered locus (orders lines inside truth.vcf)       */
    uint8_t ref_base, mutant_allele, filter, pad;
    int32_t ref_cnt, mut_cnt;
    int32_t err_cnt[4];       /* G, C, A, T (the reference's errorAlleleDepths order, :1207)         */
    int64_t rng_offset;       /* rand() calls consumed before this locus (diagnostic)                */
} ssb_target_result;

typedef struct ssb_spike_stats {
    int64_t alignmentCount, numberOfLociCovered, totalFoldCoverage, maxDepth;   /* :1668            */
    int64_t n_lines, n_kept, in_bytes, out_bytes, n_runs, n_hits, rng_draws;
    int64_t chain_mode;       /* chunks the RNG chain ran as: 1 = serial, P > 1 = P parallel chunk maps      */
    float   ms_parse, ms_sort, ms_emit, ms_cover, ms_gather, ms_rng, ms_chain, ms_patch, ms_total;
    /* sharded runs (ssb_spike_run_shard_*): where this shard sits in the one rand() stream and what the hand-off cost */
    int64_t rng_k_in, rng_k_out;      /* rand() calls consumed before the shard's first / after its last covered locus */
    int64_t locus_base;               /* covered loci owned by the shards before this one (added to locus_index)       */
    int64_t n_forwarded;              /* spiked bases handed to the next shard (reads that end in its range)           */
    float   ms_handoff_wait;          /* host time blocked on the predecessor's 8-byte offset                          */
    float   ms_phase1, ms_tally, ms_exchange;
    int32_t n_window_retries;         /* groups of the RNG chain that were walked again because the exact offset left their window */
    int32_t reserved2;
} ssb_spike_stats;

int  ssb_spike_create(ssb_ctx *ctx, const ssb_contig *contigs, int n_contigs, ssb_spike **out);
void ssb_spike_destroy(ssb_spike *sp);

/* Run on alignment lines already in HBM (d_sam 16-byte aligned; the allocation behind it must extend at
 * least 32 bytes past n -- the copy kernel reads whole 16-byte words, their contents past n are ignored;
 * ssb_spike_run_host pads its own staging buffer).  The output lines are written to
 * d_out (capacity out_cap >= n + 1 is always enough); *out_bytes gets their size.  results[] has
 * n_targets entries.  Device work is asynchronous internally but the call returns synchronised.
 * This is the call bench.py times for `value`. */
int ssb_spike_run_device(ssb_spike *sp, const uint8_t *d_sam, size_t n, uint8_t *d_out, size_t out_cap,
                         const ssb_target *targets, size_t n_targets, unsigned seed,
                         ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes);

/* Same, host buffers: copies `sam` in, runs, copies the output lines back into `out`.  This is
 * what the stochasticSpike main calls, and bench.py's `e2e`. */
int ssb_spike_run_host(ssb_spike *sp, const uint8_t *sam, size_t n, uint8_t *out, size_t out_cap,
                       const ssb_target *targets, size_t n_targets, unsigned seed,
                       ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes);

/* The reference's random stream: rand() #k0 .. #k0+n-1 after srand(seed) (stochasticSpike.c:948,297,334;
 * glibc TYPE_3 generator), produced on the device by polynomial skip-ahead.  Test / diagnostic hook. */
int ssb_spike_rand(ssb_spike *sp, unsigned seed, uint64_t k0, size_t n, int32_t *out_host);

/* SEQ_ERROR records of the last run (truth.vcf lines :1494-1557): loci, in covered order, where no
 * target was spiked and at least one non-reference allele was tallied. */
typedef struct ssb_seq_error {
    int32_t tid; int32_t ref_cnt;
    int64_t pos;
    int64_t locus_index;
    int32_t err_cnt[4];       /* G, C, A, T */
    uint8_t ref_base, pad[7];
} ssb_seq_error;
int ssb_spike_seq_error_count(ssb_spike *sp, size_t *count);
int ssb_spike_seq_errors(ssb_spike *sp, ssb_seq_error *dst, size_t cap);

/* ------------------------------------------------------------------------------------------
 * Hot path 1 on several GPUs: ONE coordinate-sorted input cut into coordinate ranges, one range
 * ("shard") per ssb_spike object / GPU / process.  The reference has one rand() stream and one
 * pileup (stochasticSpike.c:948, :1129, :1197), so the shards cooperate:
 *   - a read belongs to the input of the shard its START lies in; the shard's body is preceded by
 *     `halo_bytes` of the previous shard's last lines (every read that can reach into this range:
 *     start within the largest reference span before `lo`);
 *   - a covered locus, its pileup, its truth.vcf line and its draws belong to the shard whose range
 *     holds the locus; a read is WRITTEN by the shard whose range holds its last base, so that the
 *     outputs of the shards, concatenated in shard order, are the reference's output (:1272-1285);
 *   - the rand() offset at the start of a shard is handed over exactly: every shard simulates the
 *     window of offsets it can be entered with while its predecessors are still working (phase 1 of
 *     the chain), the 8-byte exact offset then travels shard 0 -> 1 -> ... as a table lookup each,
 *     and the targets are applied (phase 3) once it is known;
 *   - bases spiked into a read that a LATER shard writes are forwarded to that shard.
 * What travels between shards is: 5 scalars per shard (all-gather), one max-reduction over an
 * int64 per .spike record (the target stream's skip logic, :1578-1619, is one global scan), the
 * 8-byte offset (+ a flag word) and the forwarded bases -- never alignment text.
 * ------------------------------------------------------------------------------------------ */
typedef struct ssb_exchange ssb_exchange;      /* how cooperating shards talk */

/* n handles for n shards driven by n threads of ONE process (any mix of devices): out[i] belongs to shard i. */
int  ssb_exchange_local_create(int n_shards, ssb_exchange **out);
/* One handle per process over an NCCL communicator (rank = shard index).  ctx supplies the device staging. */
int  ssb_exchange_nccl_create(ssb_ctx *ctx, void *nccl_comm, int rank, int n_ranks, ssb_exchange **out);
void ssb_exchange_destroy(ssb_exchange *xc);
/* NCCL plumbing for callers that have no communicator of their own (bench.py under torchrun, the C mains):
 * rank 0 makes the id, ships the 128 bytes to the others by any means, every rank then joins. */
int  ssb_nccl_unique_id(uint8_t id128[128]);
int  ssb_nccl_comm_init_rank(ssb_ctx *ctx, int n_ranks, int rank, const uint8_t id128[128], void **comm_out);
void ssb_nccl_comm_destroy(void *nccl_comm);

typedef struct ssb_spike_shard {
    int32_t  index, count;        /* this is shard `index` of `count`, in coordinate order                       */
    int32_t  lo_tid, hi_tid;      /* owned loci: (lo_tid, lo_pos) <= (tid, pos) < (hi_tid, hi_pos), @SQ order;   */
    int64_t  lo_pos, hi_pos;      /* first shard: lo = (0, 0); last shard: hi_tid = INT32_MAX                    */
    uint64_t halo_bytes;          /* leading bytes of the body that repeat the predecessor's last lines          */
} ssb_spike_shard;

/* One shard of a cooperative run; every shard of the group must make the same call (same targets, seed).
 * Body, output and results as in ssb_spike_run_device / _host; results[t].status == SSB_T_ELSEWHERE for the
 * targets other shards consume (SSB_T_TAIL is reported by the last shard only), locus_index is global.
 * stats are this shard's share: the stats block of stochasticSpike.c:1668 is the sum over shards
 * (maxDepth: the maximum).  xc == NULL is allowed for count == 1. */
int ssb_spike_run_shard_device(ssb_spike *sp, const ssb_spike_shard *shard, ssb_exchange *xc,
                               const uint8_t *d_sam, size_t n, uint8_t *d_out, size_t out_cap,
                               const ssb_target *targets, size_t n_targets, unsigned seed,
                               ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes);
int ssb_spike_run_shard_host(ssb_spike *sp, const ssb_spike_shard *shard, ssb_exchange *xc,
                             const uint8_t *sam, size_t n, uint8_t *out, size_t out_cap,
                             const ssb_target *targets, size_t n_targets, unsigned seed,
                             ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes);

/* Host helper: cuts a coordinate-sorted SAM body into `count` shards of about equal bytes.  contig_names are the
 * @SQ names (index = tid).  halo_bases = the largest reference span a read can have (reads that start less than
 * this before a cut are repeated in front of the next shard).  Fills shards[i] and the byte range
 * [body_off[i], body_off[i] + body_len[i]) of shard i's body inside `sam` (halo included, so ranges overlap).
 * Fewer than `count` shards are made when the body is too small; returns the number made (>= 1) or < 0. */
int ssb_spike_plan_shards(const uint8_t *sam, size_t n, const char *const *contig_names, int n_contigs,
                          int count, int64_t halo_bases, ssb_spike_shard *shards, size_t *body_off, size_t *body_len);

#ifdef __cplusplus
}
#endif
#endif /* SSB200_H */
