// spike.cu -- stochastic spike-in on B200 (hot path 1).
//
// Replaces the per-locus pileup loop of stochasticSpike.c:1129-1623 for SAM text input, as a
// per-read / per-target pipeline (legal because of the facts listed in DESIGN.md section 3):
//
//   parse      one streaming pass over the SAM text -> 64-byte SamRec per line (sam_parse.cuh)
//   keep/sort  read_bam filter flags -> kept ordinals (scan), coordinate-sortedness check
//   mates      per kept read: the next kept read with the same QNAME inside its reference span
//   cover      union of [pos,end) over kept reads -> covered runs, covered-locus ordinals, stats
//   order      stable order of kept reads by (tid,end) = the reference's write order (:1272-1285,:1362-1371)
//   emit       copy every kept line to its output slot
//   targets    which .spike records hit a covered locus / are passed over (max-plus scan of :1578-1619)
//   gather     pileup entries (qpos, base, BQ, mate) of the hit targets, in pileup order
//   rng        glibc rand() stream, generated in parallel by polynomial skip-ahead (rng_glibc.cuh)
//   chain      the inherently serial part: walk the covered loci consuming selectMutantAllele draws
//              (:1197), and at each hit target run attemptToMutateBase (:526-904) over its entries
//   patch      substitute the spiked bases in the emitted text (SEQ only, QUAL untouched)
//
// No CPU fallback: every stage above is a CUDA kernel (CUB device scans/sorts are used for plumbing).
#include "common.cuh"
#include "spike_types.cuh"
#include "rng_glibc.cuh"
#include "sam_parse.cuh"
#include <cub/cub.cuh>
#include <math.h>
#include <stdlib.h>
#include <vector>
#include <time.h>

namespace {

constexpr int MAX_PILEUP = 10000;                 // stochasticSpike.c:38
constexpr int RNG_SEG    = 1024;                  // rand() outputs generated per thread
constexpr int RNG_TPB    = 256;                   // threads per block of the generator
constexpr uint64_t RNG_BLOCK = (uint64_t)RNG_SEG * RNG_TPB;

struct DevErr { int code; int pad; unsigned long long where; };

__device__ __forceinline__ void set_err(DevErr *e, int code, unsigned long long where)
{
    if (atomicCAS(&e->code, 0, code) == 0) e->where = where;
}

// ------------------------------------------------------------------------------------------
// shard range.  Keys are (tid << 32) | pos.  A shard owns the loci lo <= (tid, pos) < hi; a single-shard run has
// lo = 0, hi = ~0.  Reads are clipped to the range wherever loci are counted; a read is written by the shard that owns
// its LAST base (the reference writes a read when the pileup reaches that base, stochasticSpike.c:1272,:1362).
// ------------------------------------------------------------------------------------------
struct Range { unsigned long long lo, hi; };
__host__ __device__ __forceinline__ unsigned long long clip_s(unsigned long long skey, const Range &r) { return skey < r.lo ? r.lo : skey; }
__host__ __device__ __forceinline__ unsigned long long clip_e(unsigned long long ekey, const Range &r) { return ekey > r.hi ? r.hi : ekey; }
// ekey = (tid << 32) | end, end exclusive and >= 1 for a kept read: the key of the last base is ekey - 1
__host__ __device__ __forceinline__ bool owns_last(unsigned long long ekey, const Range &r) { return ekey - 1 >= r.lo && ekey - 1 < r.hi; }
// owned positions of contig `tid`: [x_lo, x_hi)
__device__ __forceinline__ void owned_span(const Range &r, int tid, int64_t &x_lo, int64_t &x_hi)
{
    const unsigned long long t = (unsigned long long)(uint32_t)tid << 32;
    x_lo = (r.lo >> 32) == (uint32_t)tid ? (int64_t)(uint32_t)r.lo : (r.lo > t ? 0x7fffffffffffll : 0);
    x_hi = (r.hi >> 32) == (uint32_t)tid ? (int64_t)(uint32_t)r.hi : (r.hi > t ? 0x7fffffffffffll : 0);
}

// ------------------------------------------------------------------------------------------
// compaction of the kept lines (keep flags and sortedness keys come from the tokeniser, sam_parse.cuh:line_keys)
// ------------------------------------------------------------------------------------------
// per output line: where it comes from (one 16-byte load in the emit kernel instead of a chain of dependent loads)
struct __align__(16) EmitDesc { unsigned long long src_off; uint32_t len; uint32_t add_nl; };

struct MaxOp { template <typename T> __device__ __forceinline__ T operator()(const T &a, const T &b) const { return a > b ? a : b; } };

__global__ void compact_kernel(const SamRec *__restrict__ recs, size_t n, const uint32_t *__restrict__ keep, const uint32_t *__restrict__ kord,
                               const unsigned long long *__restrict__ pkey, const unsigned long long *__restrict__ pmax,
                               uint32_t *__restrict__ k_rec, unsigned long long *__restrict__ k_start, unsigned long long *__restrict__ k_end,
                               EmitDesc *__restrict__ k_desc, unsigned long long *__restrict__ k_hash, uint32_t *__restrict__ k_hash32, uint8_t *__restrict__ k_bits,
                               unsigned long long *__restrict__ fold, unsigned int *__restrict__ maxspan, DevErr *err,
                               Range rg, unsigned long long halo_bytes)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long span = 0, fullspan = 0;
    if (i < n) {
        if (pkey[i] && pkey[i] < pmax[i]) set_err(err, SSB_E_UNSORTED, recs[i].line_off);
        if (pkey[i]) {
            // the shard's lines must be the ones its range says: halo lines start before lo, own lines inside [lo, hi)
            const unsigned long long sk = pkey[i] - (1ull << 32);
            const bool in_halo = recs[i].line_off < halo_bytes;
            if (in_halo ? sk >= rg.lo : (sk < rg.lo || sk >= rg.hi)) set_err(err, SSB_E_SHARD, recs[i].line_off);
            fullspan = (unsigned long long)(recs[i].end - recs[i].pos);
        }
        if (keep[i]) {
            const SamRec r = recs[i];
            const uint32_t o = kord[i];
            k_rec[o] = (uint32_t)i;
            const unsigned long long ks = ((unsigned long long)(uint32_t)r.tid << 32) | (uint32_t)r.pos, ke = ((unsigned long long)(uint32_t)r.tid << 32) | (uint32_t)r.end;
            k_start[o] = ks;
            k_end[o] = ke;
            { EmitDesc d; d.src_off = r.line_off; d.len = r.line_len; d.add_nl = (r.bits & REC_NO_NL) ? 1u : 0u; k_desc[o] = d; }   // a body without a final newline gets one
            k_hash[o] = r.qhash; k_hash32[o] = (uint32_t)r.qhash ^ (uint32_t)(r.qhash >> 32); k_bits[o] = r.bits;
            span = clip_e(ke, rg) - clip_s(ks, rg);            // the part of the read inside the shard's range
        }
    }
    // totalFoldCoverage = sum of reference spans of kept reads (stochasticSpike.c:1259): one atomic per block
    __shared__ unsigned long long s_sum[8]; __shared__ unsigned int s_max[8];
    unsigned long long s = span;
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    unsigned int m = (unsigned int)fullspan;                   // largest span of a pushed read: what the next shard's halo must cover
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_sum[w] = s; s_max[w] = m; }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        for (int k = 1; k < nw; k++) { s += s_sum[k]; m = max(m, s_max[k]); }
        if (s) atomicAdd(fold, s);
        if (m) atomicMax(maxspan, m);
    }
}

// ------------------------------------------------------------------------------------------
// mates: nxt[o] = first kept read after o (file order) with the same QNAME whose start lies inside
// o's reference span, NO_MATE if none; bit 31 flags "a second such read exists" (then users rescan).
// ------------------------------------------------------------------------------------------
constexpr uint32_t NO_MATE = 0x7fffffffu, MATE_MORE = 0x80000000u, PRV_NONE = 0xffffffffu;

__device__ bool same_qname(const uint8_t *sam, const SamRec &a, const SamRec &b)
{
    if (a.qhash != b.qhash || a.qname_len != b.qname_len) return false;
    const uint8_t *x = sam + a.line_off, *y = sam + b.line_off;
    for (int i = 0; i < a.qname_len; i++) if (x[i] != y[i]) return false;
    return true;
}

constexpr int MATES_TPB = 512, MATES_TILE = 1024, MATES_SLOTS = 4096;     // reads per block; its own reads + 512 ahead are staged and hashed per block
constexpr uint32_t MATES_NIL = 0xffffffffu;

__global__ void __launch_bounds__(MATES_TPB)
mates_kernel(const uint8_t *__restrict__ sam, const SamRec *__restrict__ recs, const uint32_t *__restrict__ k_rec,
             const unsigned long long *__restrict__ k_start, const unsigned long long *__restrict__ k_end,
             const uint32_t *__restrict__ k_hash32, size_t K, uint32_t *__restrict__ nxt, uint32_t *__restrict__ prv,
             uint8_t *__restrict__ cplx)
{
    // The reads that start inside a read's span follow it directly (start order): at 100x a hundred or so.  The block stages the
    // 32-bit hash folds and the start keys of its own reads and of the 512 behind them, and chains them into a small hash table
    // (push-front with an atomic exchange): a read then meets only the few entries of its own bucket instead of every read under its
    // span.  Only a read whose span reaches beyond the staged reads (very deep input) goes back to global memory for the rest.
    __shared__ uint32_t s_hash[MATES_TILE];
    __shared__ unsigned long long s_start[MATES_TILE];
    __shared__ uint32_t s_head[MATES_SLOTS];
    __shared__ uint16_t s_next[MATES_TILE];
    const size_t b0 = (size_t)blockIdx.x * MATES_TPB;
    for (int i = threadIdx.x; i < MATES_SLOTS; i += MATES_TPB) s_head[i] = MATES_NIL;
    __syncthreads();
    for (int i = threadIdx.x; i < MATES_TILE; i += MATES_TPB) {
        const size_t g = b0 + i;
        const uint32_t hh = g < K ? k_hash32[g] : 0u;
        s_hash[i] = hh;
        s_start[i] = g < K ? k_start[g] : ~0ull;
        if (g < K) s_next[i] = (uint16_t)atomicExch(&s_head[(hh * 0x9E3779B1u) >> 20], (uint32_t)i);       // NIL -> 0xffff
    }
    __syncthreads();
    const size_t o = b0 + threadIdx.x;
    if (o >= K) return;
    const unsigned long long lim = k_end[o];       // same tid, pos < end  <=>  start key < end key
    const uint32_t h = s_hash[threadIdx.x];        // candidates by a 32-bit fold of the QNAME hash; same_qname() decides
    uint32_t first = NO_MATE; bool more = false;
    auto candidate = [&](size_t b) {               // (the bucket is met in no particular order: `first` is the lowest so far)
        if (!same_qname(sam, recs[k_rec[o]], recs[k_rec[b]])) return;
        if (first == NO_MATE) first = (uint32_t)b;
        else {
            // three or more same-name reads overlap: every member takes the exact brute-force path
            more = true; cplx[o] = 1; cplx[first] = 1; cplx[b] = 1;
            if ((uint32_t)b < first) first = (uint32_t)b;
        }
    };
    for (uint32_t t = s_head[(h * 0x9E3779B1u) >> 20]; t < (uint32_t)MATES_TILE; t = s_next[t])
        if (t > threadIdx.x && s_hash[t] == h && s_start[t] < lim) candidate(b0 + t);
    if (s_start[MATES_TILE - 1] < lim && b0 + MATES_TILE < K) {
        // the span reaches beyond the staged reads: the rest from global memory (galloping bound, then four hashes per step)
        size_t g_hi;
        {
            size_t step = 64, l = b0 + MATES_TILE;
            g_hi = l;
            while (g_hi < K && k_start[g_hi] < lim) { l = g_hi + 1; g_hi += step; step <<= 1; }
            if (g_hi > K) g_hi = K;
            while (l < g_hi) { const size_t mid = (l + g_hi) >> 1; if (k_start[mid] < lim) l = mid + 1; else g_hi = mid; }
        }
        for (size_t c0 = b0 + MATES_TILE; c0 < g_hi; c0 += 4) {
            uint32_t hb[4];
#pragma unroll
            for (int u = 0; u < 4; u++) hb[u] = (c0 + u < g_hi) ? k_hash32[c0 + u] : ~h;
            if (hb[0] != h && hb[1] != h && hb[2] != h && hb[3] != h) continue;
#pragma unroll
            for (int u = 0; u < 4; u++) if (hb[u] == h && c0 + u < g_hi) candidate(c0 + u);
        }
    }
    if (first != NO_MATE) prv[first] = (uint32_t)o;                         // injective: see DESIGN.md (mate links)
    nxt[o] = first | (more ? MATE_MORE : 0u);
}

// ------------------------------------------------------------------------------------------
// coverage runs
// ------------------------------------------------------------------------------------------
// Clipped end keys (input of the prefix maximum that finds the gaps in the coverage)
__global__ void clipend_kernel(const unsigned long long *__restrict__ k_end, size_t K, Range rg, unsigned long long *__restrict__ ce)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o < K) ce[o] = clip_e(k_end[o], rg);
}

// Per kept read (start order): does it open a new covered run, and how many loci does it cover that no earlier read covered
// (pm = maximum clipped end key of the reads before it).  The exclusive sum of `newcov` is the covered ordinal at which the
// read's new part begins -- for the first read of a run, the ordinal of the run's first locus.
__global__ void newcov_kernel(const unsigned long long *__restrict__ k_start, const unsigned long long *__restrict__ ce,
                              const unsigned long long *__restrict__ pm, size_t K, Range rg, uint32_t *__restrict__ flag, unsigned long long *__restrict__ newcov)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= K) return;
    const unsigned long long cs = clip_s(k_start[o], rg), e = ce[o], m = (o == 0) ? 0ull : pm[o];
    flag[o] = (o == 0 || cs > m) ? 1u : 0u;                     // new run: other contig, or a gap before this read
    const unsigned long long from = cs > m ? cs : m;
    newcov[o] = e > from ? e - from : 0ull;
}

__global__ void runs_kernel(const unsigned long long *__restrict__ k_start, const unsigned long long *__restrict__ ce,
                            const unsigned long long *__restrict__ pm, const uint32_t *__restrict__ flag, const uint32_t *__restrict__ rid_incl,
                            const unsigned long long *__restrict__ cbase, size_t K, Range rg, CovRun *__restrict__ runs)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= K) return;
    if (flag[o]) {
        const uint32_t r = rid_incl[o] - 1;
        const unsigned long long cs = clip_s(k_start[o], rg);
        runs[r].tid = (int32_t)(cs >> 32);
        runs[r].start = (int32_t)(uint32_t)cs;
        runs[r].base = (int64_t)cbase[o]; runs[r].pad = 0;
        if (o > 0) runs[r - 1].end = (int32_t)(uint32_t)pm[o];
    }
    if (o == K - 1) {
        // lexicographic max of the clipped (tid,end) over all kept reads = (last contig, end of its last run)
        const unsigned long long m = (o > 0 && pm[o] > ce[o]) ? pm[o] : ce[o];
        runs[rid_incl[o] - 1].end = (int32_t)(uint32_t)m;
    }
}

// R and n_cov of the run, for the host
__global__ void cover_totals_kernel(const uint32_t *__restrict__ rid_incl, const unsigned long long *__restrict__ cbase, const unsigned long long *__restrict__ newcov,
                                    size_t K, unsigned int *__restrict__ n_runs, unsigned long long *__restrict__ n_cov)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) { *n_runs = rid_incl[K - 1]; *n_cov = cbase[K - 1] + newcov[K - 1]; }
}

// run index containing covered ordinal g (runs sorted by base)
__device__ __forceinline__ size_t run_of_ordinal(const CovRun *runs, size_t R, int64_t g)
{
    size_t lo = 0, hi = R;              // last run with base <= g
    while (hi - lo > 1) { size_t mid = (lo + hi) >> 1; if (runs[mid].base <= g) lo = mid; else hi = mid; }
    return lo;
}

__device__ __forceinline__ int gcat_index(uint8_t b) { return b == 'G' ? 0 : b == 'C' ? 1 : b == 'A' ? 2 : b == 'T' ? 3 : 4; }

// reference class per covered locus: index into "GCAT" (stochasticSpike.c:340), 4 = anything else
__device__ __forceinline__ uint8_t ref_class(uint8_t c) { return c == 'G' ? 0 : c == 'C' ? 1 : c == 'A' ? 2 : c == 'T' ? 3 : 4; }

__global__ void cls_kernel(const CovRun *__restrict__ runs, size_t R, int64_t n_cov, const uint8_t *const *__restrict__ contig_seq,
                           const int64_t *__restrict__ contig_len, uint8_t *__restrict__ cls, DevErr *err)
{
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_cov) return;
    size_t r = run_of_ordinal(runs, R, g);
    int tid = runs[r].tid; int64_t x = runs[r].start + (g - runs[r].base);
    const uint8_t *seq = contig_seq[tid];
    if (!seq || x >= contig_len[tid]) { set_err(err, SSB_E_REF, (unsigned long long)g); cls[g] = 4; return; }
    cls[g] = ref_class(seq[x]);
}

// ------------------------------------------------------------------------------------------
// output order and emit
// ------------------------------------------------------------------------------------------
__global__ void iota_kernel(uint32_t *p, size_t n) { size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = (uint32_t)i; }

__global__ void outlen_kernel(const uint32_t *__restrict__ perm, const unsigned long long *__restrict__ s_end, const EmitDesc *__restrict__ k_desc,
                              size_t K, Range rg, unsigned long long *__restrict__ len, EmitDesc *__restrict__ desc, unsigned long long *__restrict__ n_owned)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool mine = false;
    if (o < K) {
        mine = owns_last(s_end[o], rg);                 // a read whose last base lies beyond the range is written by the next shard
        EmitDesc d = k_desc[perm[o]];                   // (one 16-byte gather; the order is nearly the start order)
        if (!mine) { d.len = 0u; d.add_nl = 0u; }
        len[o] = (unsigned long long)d.len + d.add_nl;
        desc[o] = d;
    }
    const int cnt = __syncthreads_count(mine);          // one atomic per block: a million per-warp atomics on one address cost more than the gather
    if (threadIdx.x == 0 && cnt) atomicAdd(n_owned, (unsigned long long)cnt);
}

__global__ void ordoff_kernel(const uint32_t *__restrict__ perm, const unsigned long long *__restrict__ out_off, size_t K, unsigned long long *__restrict__ ord_off)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o < K) ord_off[perm[o]] = out_off[o];
}

// One warp per output line, 16 bytes per lane: destination-aligned 16-byte stores; the source bytes of a chunk lie in two
// aligned 16-byte source words, shifted into place.  The shift is the same for the whole line (= for the whole warp), so the
// word part of it is a four-way switch over statically indexed registers.  Two lines are in flight per warp.
struct EmitJob { const uint8_t *src; uint8_t *dst; uint32_t len, head, nvec, mis, add_nl;
                 __device__ __forceinline__ const uint4 *S() const { return reinterpret_cast<const uint4 *>(src + head - mis); }
                 __device__ __forceinline__ uint4 *D() const { return reinterpret_cast<uint4 *>(dst + head); } };

__device__ __forceinline__ EmitJob emit_job(const uint8_t *__restrict__ sam, const EmitDesc r, unsigned long long off, uint8_t *__restrict__ out)
{
    EmitJob j;
    j.src = sam + r.src_off; j.dst = out + off; j.len = r.len; j.add_nl = r.add_nl;
    uint32_t head = (uint32_t)((16 - ((uintptr_t)j.dst & 15)) & 15);
    if (head > j.len) head = j.len;
    j.head = head;
    j.nvec = (j.len - head) >> 4;
    const uint8_t *s0 = j.src + head;
    j.mis = (uint32_t)((uintptr_t)s0 & 15);
    return j;
}
template <int WQ>
__device__ __forceinline__ uint4 emit_shift(const uint4 A, const uint4 B, uint32_t sh)
{
    const uint32_t W[8] = {A.x, A.y, A.z, A.w, B.x, B.y, B.z, B.w};
    uint4 o;
    o.x = __funnelshift_r(W[WQ], W[WQ + 1], sh); o.y = __funnelshift_r(W[WQ + 1], W[WQ + 2], sh);
    o.z = __funnelshift_r(W[WQ + 2], W[WQ + 3], sh); o.w = __funnelshift_r(W[WQ + 3], W[WQ + 4], sh);
    return o;
}
__device__ __forceinline__ void emit_load(const EmitJob &j, uint32_t i, const uint8_t *sam_end, uint4 &A, uint4 &B)
{
    const uint4 *S = j.S();
    A = __ldg(S + i);
    B = make_uint4(0, 0, 0, 0);
    if (j.mis && reinterpret_cast<const uint8_t *>(S + i + 1) < sam_end) B = __ldg(S + i + 1);
}
__device__ __forceinline__ void emit_store(const EmitJob &j, uint32_t i, const uint4 A, const uint4 B)
{
    const uint32_t sh = (j.mis & 3u) * 8u;
    uint4 o;
    switch (j.mis >> 2) {
    case 0: o = emit_shift<0>(A, B, sh); break;
    case 1: o = emit_shift<1>(A, B, sh); break;
    case 2: o = emit_shift<2>(A, B, sh); break;
    default: o = emit_shift<3>(A, B, sh); break;
    }
    j.D()[i] = o;
}
__device__ __forceinline__ void emit_edges(const EmitJob &j, int lane)
{
    // < 16 bytes up to the first aligned destination address (lanes 0..15) and < 16 tail bytes (lanes 16..31) in one pass
    const uint32_t done = j.head + (j.nvec << 4);
    const uint32_t off = lane < 16 ? (uint32_t)lane : done + (uint32_t)lane - 16u;
    const bool on = lane < 16 ? (uint32_t)lane < j.head : off < j.len;
    if (on) j.dst[off] = j.src[off];
    if (lane == 0 && j.add_nl) j.dst[j.len] = '\n';
}

// one output line per warp
__global__ void __launch_bounds__(256, 8)
emit_kernel(const uint8_t *__restrict__ sam, size_t n_sam, const EmitDesc *__restrict__ desc, const unsigned long long *__restrict__ out_off, size_t K,
            uint8_t *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const uint8_t *sam_end = sam + n_sam;
    for (size_t o = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); o < K; o += warps) {
        const EmitJob j = emit_job(sam, desc[o], out_off[o], out);
        uint4 A, B;
        if ((uint32_t)lane < j.nvec) { emit_load(j, lane, sam_end, A, B); emit_store(j, lane, A, B); }
        for (uint32_t i = lane + 32; i < j.nvec; i += 32) { emit_load(j, i, sam_end, A, B); emit_store(j, i, A, B); }
        emit_edges(j, lane);
    }
}

__global__ void patch_kernel(const Patch *__restrict__ patches, const unsigned int *__restrict__ n_patches, const SamRec *__restrict__ recs,
                             const uint32_t *__restrict__ k_rec, const unsigned long long *__restrict__ k_end, const unsigned long long *__restrict__ ord_off, Range rg,
                             uint8_t *__restrict__ out)
{
    unsigned int n = *n_patches;
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const Patch p = patches[i];
        if (owns_last(k_end[p.ord], rg)) out[ord_off[p.ord] + recs[k_rec[p.ord]].seq_off + p.qpos] = (uint8_t)p.base;
    }
}

// spiked bases of reads that the NEXT shard writes (their last base lies beyond this shard's range): handed over, the read
// named by its line index counted from the end of this body
__global__ void fwd_collect_kernel(const Patch *__restrict__ patches, const unsigned int *__restrict__ n_patches, const uint32_t *__restrict__ k_rec,
                                   const unsigned long long *__restrict__ k_end, Range rg, unsigned long long n_lines,
                                   FwdPatch *__restrict__ fwd, unsigned int *__restrict__ n_fwd, unsigned int fwd_cap, DevErr *err)
{
    unsigned int n = *n_patches;
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const Patch p = patches[i];
        if (owns_last(k_end[p.ord], rg)) continue;
        const unsigned int slot = atomicAdd(n_fwd, 1u);
        if (slot < fwd_cap) { FwdPatch f; f.from_end = (uint32_t)(n_lines - k_rec[p.ord]); f.qpos = p.qpos; f.base = p.base; f.order = p.pad; fwd[slot] = f; }
        else set_err(err, SSB_E_NOMEM, i);
    }
}

// bases spiked by the previous shard into reads this shard writes (they are the first lines of this body: the halo)
__global__ void fwd_apply_kernel(const FwdPatch *__restrict__ fwd, unsigned int n, unsigned long long halo_lines, const uint32_t *__restrict__ keep, const uint32_t *__restrict__ kord,
                                 const SamRec *__restrict__ recs, const unsigned long long *__restrict__ k_end, const unsigned long long *__restrict__ ord_off, Range rg,
                                 uint8_t *__restrict__ out, DevErr *err)
{
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const FwdPatch f = fwd[i];
        if (f.from_end == 0 || f.from_end > halo_lines) { set_err(err, SSB_E_SHARD, i); continue; }
        const unsigned long long line = halo_lines - f.from_end;
        if (!keep[line]) { set_err(err, SSB_E_SHARD, i); continue; }
        const uint32_t ord = kord[line];
        if (!owns_last(k_end[ord], rg)) { set_err(err, SSB_E_SHARD, i); continue; }      // a read spanning three shards: the halo was cut too short
        out[ord_off[ord] + recs[line].seq_off + f.qpos] = (uint8_t)f.base;
    }
}

// Where an odd patch shares its byte with other patches, the one made at the latest locus must win
// (the reference applies them in locus order); patch_kernel wrote them in no particular order.
struct OddPatch;
__global__ void odd_fix_kernel(const OddPatch *odd_, const unsigned int *n_odd, unsigned int odd_cap, const Patch *__restrict__ patches,
                               const unsigned int *__restrict__ n_patches, const SamRec *__restrict__ recs, const uint32_t *__restrict__ k_rec,
                               const unsigned long long *__restrict__ k_end, const unsigned long long *__restrict__ ord_off, Range rg, uint8_t *__restrict__ out);

// ------------------------------------------------------------------------------------------
// depth
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ size_t upper_bound_u64(const unsigned long long *a, size_t n, unsigned long long key)
{
    size_t lo = 0, hi = n;                            // first index with a[i] > key
    while (lo < hi) { size_t mid = (lo + hi) >> 1; if (a[mid] <= key) lo = mid + 1; else hi = mid; }
    return lo;
}
__device__ __forceinline__ size_t lower_bound_u64(const unsigned long long *a, size_t n, unsigned long long key)
{
    size_t lo = 0, hi = n;                            // first index with a[i] >= key
    while (lo < hi) { size_t mid = (lo + hi) >> 1; if (a[mid] < key) lo = mid + 1; else hi = mid; }
    return lo;
}

// ------------------------------------------------------------------------------------------
// targets (stochasticSpike.c:1234-1245, :1578-1619, :1630-1646)
// ------------------------------------------------------------------------------------------
struct DevTarget { int32_t c_tid; uint32_t thresh; int64_t locus; uint8_t base; uint8_t pad[7]; };

// first covered ordinal whose (tid,pos) >= (c_tid, locus); n_cov if none
__device__ int64_t lb_ordinal(const CovRun *runs, size_t R, int64_t n_cov, int32_t c_tid, int64_t locus)
{
    if (c_tid < 0) return 0;
    size_t lo = 0, hi = R;                            // first run with (tid, end-1) >= (c_tid, locus)
    while (lo < hi) {
        size_t mid = (lo + hi) >> 1;
        bool before = runs[mid].tid < c_tid || (runs[mid].tid == c_tid && (int64_t)runs[mid].end - 1 < locus);
        if (before) lo = mid + 1; else hi = mid;
    }
    if (lo == R) return n_cov;
    const CovRun r = runs[lo];
    if (r.tid == c_tid && locus > r.start) return r.base + (locus - r.start);
    return r.base;
}

// Per covered locus g: cs[g] = kept reads that start at or before it, ce[g] = kept reads that end at or before it (end exclusive),
// so that the pileup depth is cs[g] - ce[g] without a search.  One pass over the reads in start order and one in end order: the
// last read of a group of equal keys fills the loci up to the next key (never more than one read span).
__global__ void cum_fill_kernel(const unsigned long long *__restrict__ keys, size_t K, const CovRun *__restrict__ runs, size_t R, int64_t n_cov,
                                uint32_t *__restrict__ out)
{
    const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= K) return;
    const unsigned long long key = keys[o];
    if (o + 1 < K && keys[o + 1] == key) return;
    const int64_t g0 = lb_ordinal(runs, R, n_cov, (int32_t)(key >> 32), (int64_t)(uint32_t)key);
    int64_t g1 = n_cov;
    if (o + 1 < K) { const unsigned long long nk = keys[o + 1]; g1 = lb_ordinal(runs, R, n_cov, (int32_t)(nk >> 32), (int64_t)(uint32_t)nk); }
    for (int64_t g = g0; g < g1; g++) out[g] = (uint32_t)(o + 1);
}

// maxDepth (stochasticSpike.c:1216)
__global__ void maxdepth_kernel(const uint32_t *__restrict__ cs, const uint32_t *__restrict__ ce, int64_t n_cov, unsigned int *__restrict__ max_depth)
{
    unsigned int d = 0;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_cov; g += (int64_t)gridDim.x * blockDim.x) d = max(d, cs[g] - ce[g]);
    for (int s = 16; s; s >>= 1) d = max(d, __shfl_xor_sync(0xffffffffu, d, s));
    if ((threadIdx.x & 31) == 0 && d) atomicMax(max_depth, d);
}

// v[t] = lb_t - t, lb_t = covered ordinal (global: ord_base + local) of the first covered locus at or after target t.
// mode 0 (cooperating shards): only the shard whose range holds the target's key knows it; the others write "minus infinity"
//   and a max-reduction over the shards assembles the array (targets on unknown contigs have lb = 0: shard 0 writes them).
// mode 1 (shards processed one after the other): targets before carry_t were consumed by earlier shards; the last ordinal
//   they used is folded into v[carry_t - 1], every later target is clamped into this shard (before the range -> its first
//   locus, after the range -> one past its last locus).
constexpr long long V_NONE = -(1ll << 62);
__global__ void target_lb_kernel(const DevTarget *__restrict__ tg, size_t T, const CovRun *__restrict__ runs, size_t R, int64_t n_cov, Range rg, long long ord_base,
                                 int mode, int shard_index, long long carry_t, long long carry_h, long long *__restrict__ v)
{
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const DevTarget x = tg[t];
    long long out;
    if (mode == 0) {
        const unsigned long long key = ((unsigned long long)(uint32_t)x.c_tid << 32) | (uint32_t)(x.locus < 0 ? 0 : x.locus);
        bool mine;
        if (x.c_tid < 0) mine = shard_index == 0;
        else if (x.locus < 0) mine = rg.lo <= ((unsigned long long)(uint32_t)x.c_tid << 32) && ((unsigned long long)(uint32_t)x.c_tid << 32) < rg.hi;   // before the contig's first base
        else if (x.locus > 0xfffffffell) mine = false;          // beyond any coordinate (handled below)
        else mine = key >= rg.lo && key < rg.hi;
        if (x.c_tid >= 0 && x.locus > 0xfffffffell) {            // past every position of its contig: first locus of the next contig
            const unsigned long long nk = ((unsigned long long)(uint32_t)(x.c_tid + 1)) << 32;
            mine = nk - 1 >= rg.lo && nk - 1 < rg.hi;
        }
        out = mine ? ord_base + (long long)(R ? lb_ordinal(runs, R, n_cov, x.c_tid, x.locus) : 0) - (long long)t : V_NONE;
    } else {
        if ((long long)t < carry_t) out = ((long long)t == carry_t - 1) ? carry_h - (long long)t : V_NONE;
        else out = ord_base + (long long)(R ? lb_ordinal(runs, R, n_cov, x.c_tid, x.locus) : (x.c_tid < 0 ? 0 : 0)) - (long long)t;
    }
    v[t] = out;
}

// h_t = t + max_{u<=t} (lb_u - u): every target consumes exactly one covered locus (the if-not-while of :1596-1599).
// The shard reports the targets whose h_t falls on one of its own loci [ord_base, ord_base + n_cov).
__global__ void target_status_kernel(const DevTarget *__restrict__ tg, size_t T, const long long *__restrict__ vmax, const CovRun *__restrict__ runs, size_t R,
                                     int64_t n_cov, long long ord_base, long long total_cov /* < 0: unknown */, int is_last,
                                     ssb_target_result *__restrict__ res, uint32_t *__restrict__ hitflag)
{
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    ssb_target_result r;
    memset(&r, 0, sizeof r);
    const long long h = vmax[t] + (long long)t;
    r.locus_index = h;
    r.rng_offset = -1;
    uint32_t hit = 0;
    if (h < ord_base || h >= ord_base + n_cov) {
        const bool tail = total_cov >= 0 ? h >= total_cov : false;
        r.status = (tail && is_last) ? SSB_T_TAIL : SSB_T_ELSEWHERE; r.at_tid = -1; r.at_pos = -1;
        if (tail) r.locus_index = total_cov;
    } else {
        const long long hl = h - ord_base;
        size_t ri = run_of_ordinal(runs, R, hl);
        int tid = runs[ri].tid; int64_t pos = runs[ri].start + (hl - runs[ri].base);
        r.at_tid = tid; r.at_pos = pos;
        if (tid == tg[t].c_tid && pos == tg[t].locus) { r.status = SSB_T_HIT; hit = 1; r.filter = SSB_F_UNDETECTED; }
        else r.status = (pos == tg[t].locus) ? SSB_T_NOCOV_SILENT : SSB_T_NOCOV;       // :1603
    }
    res[t] = r;
    hitflag[t] = hit;
}

__global__ void hits_kernel(const DevTarget *__restrict__ tg, size_t T, const uint32_t *__restrict__ hitflag, const uint32_t *__restrict__ hidx,
                            const ssb_target_result *__restrict__ res, long long ord_base, HitTarget *__restrict__ hits)
{
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T || !hitflag[t]) return;
    HitTarget h;
    memset(&h, 0, sizeof h);
    h.locus_index = res[t].locus_index - ord_base; h.tid = res[t].at_tid; h.pos = (int32_t)res[t].at_pos;     // local ordinal
    h.target = (uint32_t)t; h.thresh = tg[t].thresh; h.base = tg[t].base;
    hits[hidx[t]] = h;
}

// ------------------------------------------------------------------------------------------
// pileup gather at the hit targets
// ------------------------------------------------------------------------------------------
// column geometry of one read at reference position x (htslib resolve_cigar semantics, SURVEY App. D)
__device__ void column_of(const uint8_t *cig, int cig_len, int32_t rpos, int32_t x, uint32_t &qpos, uint8_t &skip)
{
    int64_t ref = rpos; uint32_t y = 0;
    qpos = 0; skip = 0;
    uint32_t num = 0;
    for (int i = 0; i < cig_len; i++) {
        uint8_t c = cig[i];
        if (c >= '0' && c <= '9') { num = num * 10 + (c - '0'); continue; }
        uint32_t l = num; num = 0;
        if (c == 'M' || c == '=' || c == 'X') { if (x < ref + l) { qpos = y + (uint32_t)(x - ref); return; } ref += l; y += l; }
        else if (c == 'D' || c == 'N') { if (x < ref + l) { skip = 1; qpos = y; return; } ref += l; }
        else if (c == 'I' || c == 'S') y += l;
    }
}

// candidates of a locus: kept reads [lo, hi) by start; an entry is a candidate whose end lies beyond the locus
__device__ __forceinline__ void cand_range(const unsigned long long *k_start, size_t K, int32_t tid, int32_t pos, unsigned int maxspan, size_t &lo, size_t &hi)
{
    const unsigned long long key = ((unsigned long long)(uint32_t)tid << 32) | (uint32_t)pos;
    int64_t first = (int64_t)pos - (int64_t)maxspan + 1; if (first < 0) first = 0;
    lo = lower_bound_u64(k_start, K, ((unsigned long long)(uint32_t)tid << 32) | (uint32_t)first);
    hi = upper_bound_u64(k_start, K, key);
}

__global__ void gather_count_kernel(const HitTarget *__restrict__ hits, size_t H, const unsigned long long *__restrict__ k_start,
                                    const unsigned long long *__restrict__ k_end, size_t K, const unsigned int *__restrict__ maxspan,
                                    unsigned long long *__restrict__ cnt, DevErr *err)
{
    const int lane = threadIdx.x & 31;
    size_t h = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (h >= H || hits[h].tid < 0) return;              // slots past the last hit are marked tid < 0
    size_t lo, hi; cand_range(k_start, K, hits[h].tid, hits[h].pos, *maxspan, lo, hi);
    const unsigned long long lim = ((unsigned long long)(uint32_t)hits[h].tid << 32) | (uint32_t)hits[h].pos;
    unsigned int c = 0;
    for (size_t i = lo + lane; i < hi; i += 32) c += (k_end[i] > lim) ? 1u : 0u;
    for (int s = 16; s; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
    if (lane == 0) { cnt[h] = c; if (c > MAX_PILEUP) set_err(err, SSB_E_DEPTH, (unsigned long long)h); }
}

__global__ void gather_fill_kernel(const uint8_t *__restrict__ sam, const SamRec *__restrict__ recs, const uint32_t *__restrict__ k_rec,
                                   const HitTarget *__restrict__ hits, size_t H, const unsigned long long *__restrict__ k_start,
                                   const unsigned long long *__restrict__ k_end, size_t K, const unsigned int *__restrict__ maxspan,
                                   const unsigned long long *__restrict__ eoff, PlpEntry *__restrict__ ent)
{
    const int lane = threadIdx.x & 31;
    size_t h = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (h >= H) return;
    const int32_t x = hits[h].pos;
    size_t lo, hi; cand_range(k_start, K, hits[h].tid, x, *maxspan, lo, hi);
    const unsigned long long lim = ((unsigned long long)(uint32_t)hits[h].tid << 32) | (uint32_t)x;
    unsigned long long w = eoff[h];
    for (size_t base = lo; base < hi; base += 32) {
        size_t i = base + lane;
        bool in = i < hi && k_end[i] > lim;
        unsigned m = __ballot_sync(0xffffffffu, in);
        if (in) {
            const SamRec &r = recs[k_rec[i]];
            PlpEntry e;
            e.ord = (uint32_t)i; e.mate = -1; e.pad = 0;
            const uint8_t *line = sam + r.line_off;
            column_of(line + r.cigar_off, r.cigar_len, r.pos, x, e.qpos, e.skip);
            e.base = line[r.seq_off + e.qpos];
            e.bq = (r.bits & REC_QUALSTAR) ? (uint8_t)0xff : (uint8_t)(line[r.qual_off + e.qpos] - 33);
            ent[w + __popc(m & ((1u << lane) - 1u))] = e;
        }
        w += __popc(m);
    }
}

// mate = index, inside the same pileup, of the first later entry with the same QNAME (findOverlappingMate, :363-383)
__global__ void gather_mate_kernel(const uint8_t *__restrict__ sam, const SamRec *__restrict__ recs, const uint32_t *__restrict__ k_rec,
                                   const unsigned long long *__restrict__ k_start, const unsigned long long *__restrict__ k_end,
                                   const unsigned long long *__restrict__ k_hash, size_t K, const uint32_t *__restrict__ nxt,
                                   const HitTarget *__restrict__ hits, size_t H, const unsigned long long *__restrict__ eoff, PlpEntry *__restrict__ ent)
{
    const int lane = threadIdx.x & 31;
    size_t h = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (h >= H) return;
    const unsigned long long e0 = eoff[h], e1 = eoff[h + 1];
    const unsigned long long lim = ((unsigned long long)(uint32_t)hits[h].tid << 32) | (uint32_t)hits[h].pos;
    for (unsigned long long j = e0 + lane; j < e1; j += 32) {
        const uint32_t a = ent[j].ord;
        uint32_t n1 = nxt[a];
        uint32_t mate_ord = NO_MATE;
        if ((n1 & ~MATE_MORE) != NO_MATE) {
            uint32_t b = n1 & ~MATE_MORE;
            if (k_start[b] <= lim && k_end[b] > lim) mate_ord = b;          // the first same-name read covers the locus
            else if ((n1 & MATE_MORE) && k_start[b] <= lim) {
                // rare: several same-name reads start inside a's span; take the first one that covers the locus
                for (size_t c = b + 1; c < K && k_start[c] <= lim; c++)
                    if (k_hash[c] == k_hash[a] && k_end[c] > lim && same_qname(sam, recs[k_rec[a]], recs[k_rec[c]])) { mate_ord = (uint32_t)c; break; }
            }
        }
        if (mate_ord != NO_MATE) {
            // entries are sorted by ord: binary search inside (j, e1)
            unsigned long long lo = j + 1, hi = e1;
            while (lo < hi) { unsigned long long mid = (lo + hi) >> 1; if (ent[mid].ord < mate_ord) lo = mid + 1; else hi = mid; }
            if (lo < e1 && ent[lo].ord == mate_ord) ent[j].mate = (int32_t)(lo - e0);
        }
    }
}

// ------------------------------------------------------------------------------------------
// "odd" patches.  getBaseWithRPOcheck (:387-432) takes the mate's base at the mate's qpos without
// looking at is_del / is_refskip, and for a deleted/skipped column htslib's qpos is the NEXT
// aligned base.  attemptToMutateBase cases 3-6 can therefore overwrite a base that belongs to a
// LATER locus, and because the reference edits reads in place every later locus sees it.  Such
// patches are rare (a mate inside a D/N at a target that tosses heads); they are kept in a small
// list that the chain and the tally consult so that the result stays bit-exact.
// ------------------------------------------------------------------------------------------
struct OddPatch { uint32_t ord, qpos, base, h; int32_t tid, pos; };

__device__ __forceinline__ unsigned long long odd_bit(uint32_t ord) { return 1ull << ((ord * 2654435761u) >> 26); }

// value of (ord,qpos) as seen at locus (tid,pos): the last odd patch made at an earlier locus wins
__device__ uint8_t odd_view(const OddPatch *odd, unsigned int n_odd, uint32_t ord, uint32_t qpos, int32_t tid, int64_t pos, uint8_t base)
{
    for (unsigned int i = 0; i < n_odd; i++)          // list is in target (= locus) order
        if (odd[i].ord == ord && odd[i].qpos == qpos && (odd[i].tid < tid || (odd[i].tid == tid && odd[i].pos < pos))) base = (uint8_t)odd[i].base;
    return base;
}

__global__ void odd_fix_kernel(const OddPatch *odd, const unsigned int *n_odd, unsigned int odd_cap, const Patch *__restrict__ patches,
                               const unsigned int *__restrict__ n_patches, const SamRec *__restrict__ recs, const uint32_t *__restrict__ k_rec,
                               const unsigned long long *__restrict__ k_end, const unsigned long long *__restrict__ ord_off, Range rg, uint8_t *__restrict__ out)
{
    const unsigned int no = min(*n_odd, odd_cap), np = *n_patches;
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < no; i += gridDim.x * blockDim.x) {
        const OddPatch q = odd[i];
        uint32_t best_h = 0, best_base = q.base; bool any = false;
        for (unsigned int p = 0; p < np; p++)
            if (patches[p].ord == q.ord && patches[p].qpos == q.qpos && (!any || patches[p].pad >= best_h)) { any = true; best_h = patches[p].pad; best_base = patches[p].base; }
        if (owns_last(k_end[q.ord], rg)) out[ord_off[q.ord] + recs[k_rec[q.ord]].seq_off + q.qpos] = (uint8_t)best_base;
    }
}

// ------------------------------------------------------------------------------------------
// per-locus allele tallies at the loci that are not spike targets (stochasticSpike.c:1296-1357), for
// the SEQ_ERROR lines of truth.vcf (:1494-1557).
//
// ref(x) = depth(x) - minus(x): depth comes from the sorted start/end arrays, minus(x) counts the
// pileup entries at x that do NOT add to refAlleleCnt (deleted/skipped bases, BQ 0, N, mismatches,
// second mates already handled).  Only those exceptional bases cost an atomic.
// err64[x] packs the four error-allele counters (G,C,A,T, 16 bits each; depth <= 10000).
// ------------------------------------------------------------------------------------------
struct ReadView {
    const uint8_t *line; const uint8_t *cig; int cig_len; int32_t pos, end; uint32_t seq_off, qual_off, l_seq; bool qual_star;
    uint32_t ord; int32_t tid; const OddPatch *odd; unsigned int n_odd;      // odd != NULL only for the few reads an odd patch touched
    bool simple;                                                             // CIGAR of M/=/X only: qpos = x - pos
};
__device__ __forceinline__ ReadView view_of(const uint8_t *sam, const SamRec &r, uint32_t ord, const OddPatch *odd, unsigned int n_odd, unsigned long long bloom)
{
    ReadView v; v.line = sam + r.line_off; v.ord = ord; v.tid = r.tid; v.odd = NULL; v.n_odd = 0; v.simple = (r.bits & REC_SIMPLE) != 0;
    if (n_odd && (bloom & odd_bit(ord))) { v.odd = odd; v.n_odd = n_odd; } v.cig = v.line + r.cigar_off; v.cig_len = r.cigar_len; v.pos = r.pos; v.end = r.end;
    v.seq_off = r.seq_off; v.qual_off = r.qual_off; v.l_seq = r.l_seq; v.qual_star = (r.bits & REC_QUALSTAR) != 0;
    return v;
}
__device__ __forceinline__ void base_at(const ReadView &v, int32_t x, uint8_t &base, int &bq, bool &skip)
{
    uint32_t qpos; uint8_t sk;
    if (v.simple) { qpos = (uint32_t)(x - v.pos); sk = 0; }
    else column_of(v.cig, v.cig_len, v.pos, x, qpos, sk);
    if (qpos >= v.l_seq) qpos = v.l_seq - 1;        // malformed CIGAR tail (the reference would read out of bounds)
    base = v.line[v.seq_off + qpos];
    if (v.odd) base = odd_view(v.odd, v.n_odd, v.ord, qpos, v.tid, x, base);
    bq = v.qual_star ? 255 : (int)v.line[v.qual_off + qpos] - 33;
    skip = sk != 0;
}

struct TallyArgs {
    const uint8_t *sam; const SamRec *recs; const uint32_t *k_rec; const unsigned long long *k_start, *k_end, *k_hash; const uint8_t *k_bits; size_t K;
    const uint32_t *nxt, *prv; const uint8_t *cplx; unsigned int maxspan;
    const CovRun *runs; size_t R; const uint8_t *const *contig_seq; const int64_t *contig_len;
    unsigned long long *err64; unsigned int *minus; DevErr *err;
    const OddPatch *odd; const unsigned int *n_odd; const unsigned long long *odd_bloom;
    int listed_only;          // 1: the tokeniser's exception list is in use; fast reads it did not cover take the generic kernel
    Range rg;                 // loci outside the shard's range belong to another shard's tallies
};

// what entry `self` (index into members) adds at locus x, given the same-name reads that cover x in file order:
// 0 nothing, 1 ref, 2..5 error allele G,C,A,T   (the j-loop of :1255-1357 restricted to one QNAME)
__device__ int chain_contribution(const ReadView *mem, int n, int self, int32_t x, uint8_t F)
{
    bool handled[8];
    for (int i = 0; i < n; i++) handled[i] = false;
    for (int m = 0; m <= self; m++) {
        uint8_t Rb; int rbq; bool sk;
        base_at(mem[m], x, Rb, rbq, sk);
        int contrib = 0;
        if (!(sk || rbq == 0 || handled[m])) {
            uint8_t Mb = 0; int mbq = 0;
            const int mate = m + 1 < n ? m + 1 : -1;                    // first later entry with the same QNAME
            if (mate >= 0 && !handled[mate]) { bool msk; base_at(mem[mate], x, Mb, mbq, msk); }
            if (Mb == 'N') mbq = 0;
            if (Rb == 'N') rbq = 0;
            uint8_t base = Rb;
            if (Mb && Mb != Rb && mbq > rbq) base = Mb;
            if (base == 'N') { handled[m] = true; if (Mb) handled[mate] = true; }
            else if (base == F) contrib = 1;
            else { int gi = gcat_index(base); contrib = gi < 4 ? 2 + gi : 0; handled[m] = true; if (Mb) handled[mate] = true; }
        }
        if (m == self) return contrib;
    }
    return 0;
}

__device__ __forceinline__ void tally_add(const TallyArgs &A, int64_t g, int contrib)
{
    if (contrib == 1) return;
    atomicAdd(&A.minus[g], 1u);
    if (contrib >= 2) atomicAdd(&A.err64[g], 1ull << (16 * (contrib - 2)));
}

// A read takes the fast tally when every query base aligns 1:1 to the reference (CIGAR of M/=/X only), the only reads
// that share its QNAME inside its span are its direct neighbours in the mate chain and are just as simple, and no odd
// patch touched any of them.
__device__ __forceinline__ bool tally_simple_read(const TallyArgs &A, size_t o, unsigned int n_odd, unsigned long long bloom)
{
    if (!(A.k_bits[o] & REC_SIMPLE) || A.cplx[o]) return false;
    if (n_odd && (bloom & odd_bit((uint32_t)o))) return false;
    return true;
}
__device__ __forceinline__ bool tally_is_fast(const TallyArgs &A, size_t o, const SamRec &r, unsigned int n_odd, unsigned long long bloom)
{
    if (!tally_simple_read(A, o, n_odd, bloom)) return false;
    const uint32_t p = A.prv[o], q = A.nxt[o] & ~MATE_MORE;
    if (p != PRV_NONE && !tally_simple_read(A, p, n_odd, bloom)) return false;
    if (q != NO_MATE && !tally_simple_read(A, q, n_odd, bloom)) return false;
    (void)r;
    return true;
}

// List mode: a read is settled from the tokeniser's exception list iff it is fast-eligible, the tokeniser listed its own
// exceptional bases, and it listed those of its mate-chain neighbours too (a plain base only changes its contribution when a
// neighbour's base over the same position is exceptional, and that entry is what triggers the re-evaluation).  Every other
// read is self-contained work of tally_kernel.
__device__ __forceinline__ bool tally_is_listed(const TallyArgs &A, size_t o, const SamRec &r, unsigned int n_odd, unsigned long long bloom)
{
    if (!(A.k_bits[o] & REC_EXC_DONE) || !tally_is_fast(A, o, r, n_odd, bloom)) return false;
    const uint32_t p = A.prv[o], q = A.nxt[o] & ~MATE_MORE;
    if (p != PRV_NONE && !(A.k_bits[p] & REC_EXC_DONE)) return false;
    if (q != NO_MATE && !(A.k_bits[q] & REC_EXC_DONE)) return false;
    return true;
}

__device__ __forceinline__ uint32_t ldg_u32_unaligned(const uint8_t *p)
{
    const uint32_t a = (uint32_t)((uintptr_t)p & 3u);
    const uint32_t *q = reinterpret_cast<const uint32_t *>(p - a);
    return __funnelshift_r(__ldg(q), __ldg(q + 1), a * 8);
}

// 0x80 flags of the bytes of a simple read that are not plain "reference base with BQ > 0" at query offset w..w+3
__device__ __forceinline__ uint32_t exc_word(const uint8_t *seq, const uint8_t *qual, bool qstar, uint32_t w, uint32_t refw)
{
    const uint32_t sq = ldg_u32_unaligned(seq + w);
    const uint32_t ql = qstar ? 0x7e7e7e7eu : ldg_u32_unaligned(qual + w);
    // a read N counts nothing, also where it equals a reference N (reads through the N runs of a real reference)
    return (~samparse::zero_bytes(sq ^ refw) | samparse::zero_bytes(sq ^ 0x4E4E4E4Eu) | samparse::zero_bytes(ql ^ 0x21212121u)) & 0x80808080u;
}

// the rare path of the fast tally: one exceptional base of read o at reference position x, evaluated exactly
__device__ __noinline__ void tally_exceptional_base(const TallyArgs &A, uint32_t o, int32_t x, int64_t g)
{
    const SamRec &r = A.recs[A.k_rec[o]];
    ReadView mem[3]; int n = 0, self = 0;
    const uint32_t p = A.prv[o], q = A.nxt[o] & ~MATE_MORE;
    if (p != PRV_NONE && (uint32_t)A.k_end[p] > (uint32_t)r.pos) mem[n++] = view_of(A.sam, A.recs[A.k_rec[p]], p, NULL, 0, 0);
    self = n; mem[n++] = view_of(A.sam, r, o, NULL, 0, 0);
    if (q != NO_MATE) mem[n++] = view_of(A.sam, A.recs[A.k_rec[q]], q, NULL, 0, 0);
    ReadView cov[3]; int nc = 0, sc = 0;
    for (int m = 0; m < n; m++) if (mem[m].pos <= x && x < mem[m].end) { if (m == self) sc = nc; cov[nc++] = mem[m]; }
    const uint8_t F = A.contig_seq[r.tid][x];
    tally_add(A, g, chain_contribution(cov, nc, sc, x, F));
}

// Compact per-read metadata for the fast tally (one 32-byte load instead of a chain of dependent loads)
struct __align__(16) KMeta { unsigned long long line_off; uint32_t seq_off, qual_off, l_seq; int32_t pos, end; uint32_t tid_bits; };
static_assert(sizeof(KMeta) == 32, "KMeta layout");

__global__ void kmeta_kernel(const SamRec *__restrict__ recs, const uint32_t *__restrict__ k_rec, size_t K, KMeta *__restrict__ km)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= K) return;
    const SamRec &r = recs[k_rec[o]];
    KMeta m; m.line_off = r.line_off; m.seq_off = r.seq_off; m.qual_off = r.qual_off; m.l_seq = r.l_seq; m.pos = r.pos; m.end = r.end;
    m.tid_bits = ((uint32_t)r.tid << 8) | r.bits;
    km[o] = m;
}

// One warp per read: SEQ, QUAL and the reference compared four bytes per lane; only bytes that differ from the
// reference or have BQ 0 -- in this read or in an overlapping mate -- are evaluated one by one.
__global__ void __launch_bounds__(128, 8)
tally_fast_kernel(TallyArgs A, const KMeta *__restrict__ km)
{
    const int lane = threadIdx.x & 31;
    const size_t o = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (o >= A.K) return;
    const unsigned int n_odd = *A.n_odd; const unsigned long long bloom = *A.odd_bloom;
    const KMeta me = km[o];
    const uint32_t p = A.prv[o], q = A.nxt[o] & ~MATE_MORE;
    auto simple_ok = [&](uint32_t idx, uint32_t tid_bits) {
        return (tid_bits & REC_SIMPLE) && !A.cplx[idx] && !(n_odd && (bloom & odd_bit(idx)));
    };
    if (!simple_ok((uint32_t)o, me.tid_bits)) return;
    KMeta mp, mq; mp.pos = 0; mp.end = 0; mq.pos = 0; mq.end = 0;
    bool hp = false, hq = false;
    if (p != PRV_NONE) { mp = km[p]; if (!simple_ok(p, mp.tid_bits)) return; hp = mp.end > me.pos; }
    if (q != NO_MATE) { mq = km[q]; if (!simple_ok(q, mq.tid_bits)) return; hq = true; }
    const int tid = (int)(me.tid_bits >> 8);
    const uint8_t *ref = A.contig_seq[tid];
    if (!ref || (int64_t)me.end > A.contig_len[tid]) { if (lane == 0) set_err(A.err, SSB_E_REF, me.line_off); return; }
    size_t ri; { size_t lo = 0, hi = A.R; while (hi - lo > 1) { size_t mid = (lo + hi) >> 1;
                   bool le = A.runs[mid].tid < tid || (A.runs[mid].tid == tid && A.runs[mid].start <= me.pos); if (le) lo = mid; else hi = mid; } ri = lo; }
    const int64_t gbase = A.runs[ri].base - A.runs[ri].start + me.pos;    // covered ordinal of query offset 0
    int64_t xl, xh; owned_span(A.rg, tid, xl, xh);
    const uint8_t *seq = A.sam + me.line_off + me.seq_off, *qual = A.sam + me.line_off + me.qual_off, *rf = ref + me.pos;
    const bool qstar = (me.tid_bits & REC_QUALSTAR) != 0;
    const uint32_t L = me.l_seq;
    for (uint32_t w = lane * 4; w < L; w += 128) {
        const uint32_t rw = ldg_u32_unaligned(rf + w);
        uint32_t exc = exc_word(seq, qual, qstar, w, rw);
        const int32_t x0 = me.pos + (int32_t)w;
        if (hp && !(x0 + 3 < mp.pos || x0 >= mp.end)) {
            if (x0 >= mp.pos && x0 + 4 <= mp.end)
                exc |= exc_word(A.sam + mp.line_off + mp.seq_off, A.sam + mp.line_off + mp.qual_off, (mp.tid_bits & REC_QUALSTAR) != 0, (uint32_t)(x0 - mp.pos), rw);
            else exc = 0x80808080u;                                    // the mate starts or ends inside this word: look at every byte
        }
        if (hq && !(x0 + 3 < mq.pos || x0 >= mq.end)) {
            if (x0 >= mq.pos && x0 + 4 <= mq.end)
                exc |= exc_word(A.sam + mq.line_off + mq.seq_off, A.sam + mq.line_off + mq.qual_off, (mq.tid_bits & REC_QUALSTAR) != 0, (uint32_t)(x0 - mq.pos), rw);
            else exc = 0x80808080u;
        }
        const uint32_t rem = L - w;
        if (rem < 4) exc &= (1u << (8 * rem)) - 1u;
        while (exc) {
            const int k = (__ffs(exc) - 1) >> 3; exc &= exc - 1;
            if (x0 + k >= xl && x0 + k < xh) tally_exceptional_base(A, (uint32_t)o, x0 + k, gbase + w + k);
        }
    }
}

// One thread per exceptional base listed by the tokeniser: the base itself, and any mate lying over the same position
// whose own base is plain (so it has no entry of its own) but which this base may have marked handled.
__global__ void __launch_bounds__(128)
tally_resolve_kernel(TallyArgs A, const unsigned long long *__restrict__ list, unsigned long long n_list, const uint32_t *__restrict__ keep,
                     const uint32_t *__restrict__ kord)
{
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_list) return;
    const unsigned long long e = list[i];
    const size_t line = (size_t)(e >> 16);
    if (!keep[line]) return;
    const uint32_t o = kord[line];
    const SamRec &r = A.recs[A.k_rec[o]];
    const unsigned int n_odd = *A.n_odd; const unsigned long long bloom = *A.odd_bloom;
    const bool own = tally_is_listed(A, o, r, n_odd, bloom);           // else the read itself is tally_kernel's work
    const int32_t x = r.pos + (int32_t)(e & 0xffff);
    { int64_t xl, xh; owned_span(A.rg, r.tid, xl, xh); if (x < xl || x >= xh) return; }
    size_t ri; { size_t lo = 0, hi = A.R; while (hi - lo > 1) { size_t mid = (lo + hi) >> 1;
                   bool le = A.runs[mid].tid < r.tid || (A.runs[mid].tid == r.tid && A.runs[mid].start <= r.pos); if (le) lo = mid; else hi = mid; } ri = lo; }
    const int64_t g = A.runs[ri].base + (x - A.runs[ri].start);
    if (A.cplx[o]) return;                                             // three or more same-name reads overlap: all of them are tally_kernel's
    ReadView mem[3]; uint32_t ords[3]; int n = 0, self = 0;
    const uint32_t p = A.prv[o], q = A.nxt[o] & ~MATE_MORE;
    if (p != PRV_NONE && (uint32_t)A.k_end[p] > (uint32_t)r.pos) { ords[n] = p; mem[n++] = view_of(A.sam, A.recs[A.k_rec[p]], p, NULL, 0, 0); }
    self = n; ords[n] = o; mem[n++] = view_of(A.sam, r, o, NULL, 0, 0);
    if (q != NO_MATE) { ords[n] = q; mem[n++] = view_of(A.sam, A.recs[A.k_rec[q]], q, NULL, 0, 0); }
    ReadView cov[3]; uint32_t cord[3]; int nc = 0, sc = 0;
    for (int m = 0; m < n; m++) if (mem[m].pos <= x && x < mem[m].end) { if (m == self) sc = nc; cord[nc] = ords[m]; cov[nc++] = mem[m]; }
    const uint8_t F = A.contig_seq[r.tid][x];
    if (own) tally_add(A, g, chain_contribution(cov, nc, sc, x, F));
    for (int m = 0; m < nc; m++) {
        if (m == sc) continue;
        if (!(A.k_bits[cord[m]] & REC_SIMPLE)) continue;                 // a neighbour with indels is never list-settled
        uint8_t b; int bq; bool sk;
        base_at(cov[m], x, b, bq, sk);
        // a plain base of a list-settled neighbour has no entry of its own: it matters only if it was marked handled here
        if (b == F && b != 'N' && bq != 0 && tally_is_listed(A, cord[m], A.recs[A.k_rec[cord[m]]], n_odd, bloom)) tally_add(A, g, chain_contribution(cov, nc, m, x, F));
    }
}

__global__ void __launch_bounds__(128)
tally_kernel(TallyArgs A)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= A.K) return;
    const SamRec &r = A.recs[A.k_rec[o]];
    const unsigned int n_odd = *A.n_odd; const unsigned long long bloom = *A.odd_bloom;
    if (A.listed_only ? tally_is_listed(A, o, r, n_odd, bloom) : tally_is_fast(A, o, r, n_odd, bloom)) return;   // settled by tally_resolve_kernel / tally_fast_kernel
    const ReadView me = view_of(A.sam, r, (uint32_t)o, A.odd, n_odd, bloom);
    const int tid = r.tid;
    const uint8_t *ref = A.contig_seq[tid];
    if (!ref || (int64_t)r.end > A.contig_len[tid]) { set_err(A.err, SSB_E_REF, r.line_off); return; }   // :1181 mplp_get_ref / read past the contig
    // same-name reads that overlap this one, in file order
    ReadView mem[8]; int n = 0, self = 0; bool use_chain = false;
    if (A.cplx[o]) {
        // exact brute force: every kept read of this contig that can overlap [pos,end) and carries the same QNAME
        const unsigned long long h = A.k_hash[o];
        int64_t first = (int64_t)r.pos - (int64_t)A.maxspan + 1; if (first < 0) first = 0;
        size_t lo = lower_bound_u64(A.k_start, A.K, ((unsigned long long)(uint32_t)tid << 32) | (uint32_t)first);
        const unsigned long long lim = A.k_end[o];
        for (size_t b = lo; b < A.K && A.k_start[b] < lim; b++) {
            if (b != o && (A.k_hash[b] != h || !same_qname(A.sam, r, A.recs[A.k_rec[b]]))) continue;
            if (b != o && (uint32_t)(A.k_end[b]) <= (uint32_t)r.pos) continue;
            if (n == 8) { set_err(A.err, SSB_E_FORMAT, r.line_off); return; }       // more than eight overlapping alignments of one QNAME: refused, never miscounted
            if (b == o) self = n;
            mem[n++] = view_of(A.sam, A.recs[A.k_rec[b]], (uint32_t)b, A.odd, n_odd, bloom);
        }
        use_chain = n > 1;
    } else {
        const uint32_t p = A.prv[o], q = A.nxt[o] & ~MATE_MORE;
        if (p != PRV_NONE && (uint32_t)A.k_end[p] > (uint32_t)r.pos) mem[n++] = view_of(A.sam, A.recs[A.k_rec[p]], p, A.odd, n_odd, bloom);
        self = n; mem[n++] = me;
        if (q != NO_MATE) mem[n++] = view_of(A.sam, A.recs[A.k_rec[q]], q, A.odd, n_odd, bloom);
        use_chain = n > 1;
    }
    // covered ordinal of this read's first base: reads never span two runs
    size_t ri; { size_t lo = 0, hi = A.R; while (hi - lo > 1) { size_t mid = (lo + hi) >> 1;
                   bool le = A.runs[mid].tid < tid || (A.runs[mid].tid == tid && A.runs[mid].start <= r.pos); if (le) lo = mid; else hi = mid; } ri = lo; }
    const int64_t gbase = A.runs[ri].base - A.runs[ri].start;           // g = gbase + x
    int64_t xl, xh; owned_span(A.rg, tid, xl, xh);
    // walk the CIGAR
    int64_t x = r.pos; uint32_t y = 0, num = 0;
    for (int ci = 0; ci < me.cig_len; ci++) {
        const uint8_t c = me.cig[ci];
        if (c >= '0' && c <= '9') { num = num * 10 + (c - '0'); continue; }
        const uint32_t l = num; num = 0;
        if (c == 'M' || c == '=' || c == 'X') {
            for (uint32_t t = 0; t < l; t++, x++, y++) {
                if (x < xl || x >= xh) continue;
                const uint8_t F = ref[x];
                int contrib;
                bool overlapped = false;
                if (use_chain) for (int m = 0; m < n; m++) if (m != self && mem[m].pos <= x && x < mem[m].end) { overlapped = true; break; }
                if (overlapped) {
                    ReadView cov[8]; int nc = 0, sc = 0;
                    for (int m = 0; m < n; m++) if (mem[m].pos <= x && x < mem[m].end) { if (m == self) sc = nc; cov[nc++] = mem[m]; }
                    contrib = chain_contribution(cov, nc, sc, (int32_t)x, F);
                } else {
                    uint8_t b = me.line[me.seq_off + y];
                    if (me.odd) b = odd_view(me.odd, me.n_odd, me.ord, y, tid, x, b);
                    const int bq = me.qual_star ? 255 : (int)me.line[me.qual_off + y] - 33;
                    if (bq == 0 || b == 'N') contrib = 0;
                    else if (b == F) contrib = 1;
                    else { int gi = gcat_index(b); contrib = gi < 4 ? 2 + gi : 0; }
                }
                tally_add(A, gbase + x, contrib);
            }
        } else if (c == 'D' || c == 'N') {
            for (uint32_t t = 0; t < l; t++, x++) if (x >= xl && x < xh) atomicAdd(&A.minus[gbase + x], 1u);      // in the pileup, adds to nothing
        } else if (c == 'I' || c == 'S') y += l;
    }
}

__global__ void tally_clear_hits_kernel(const HitTarget *__restrict__ hits, size_t H, unsigned long long *__restrict__ err64)
{
    size_t h = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (h < H) err64[hits[h].locus_index] = 0;          // a target locus prints its own line (:1406-1470), never SEQ_ERROR
}

__global__ void tally_flag_kernel(const unsigned long long *__restrict__ err64, int64_t n_cov, uint32_t *__restrict__ flag)
{
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < n_cov) flag[g] = err64[g] ? 1u : 0u;
}

__global__ void se_total_kernel(const uint32_t *__restrict__ idx, const uint32_t *__restrict__ flag, int64_t n_cov, unsigned long long *__restrict__ n_se)
{
    if (!blockIdx.x && !threadIdx.x) *n_se = (unsigned long long)idx[n_cov - 1] + flag[n_cov - 1];
}

__global__ void tally_emit_kernel(const unsigned long long *__restrict__ err64, const unsigned int *__restrict__ minus, const uint32_t *__restrict__ flag,
                                  const uint32_t *__restrict__ idx, int64_t n_cov, const CovRun *__restrict__ runs, size_t R,
                                  const uint32_t *__restrict__ cum_s, const uint32_t *__restrict__ cum_e,
                                  const uint8_t *const *__restrict__ contig_seq, long long ord_base, ssb_seq_error *__restrict__ out)
{
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_cov || !flag[g]) return;
    size_t ri = run_of_ordinal(runs, R, g);
    const int tid = runs[ri].tid; const int64_t x = runs[ri].start + (g - runs[ri].base);
    const long long depth = (long long)cum_s[g] - (long long)cum_e[g];
    ssb_seq_error e;
    memset(&e, 0, sizeof e);
    e.tid = tid; e.pos = x; e.locus_index = g + ord_base;
    e.ref_cnt = (int32_t)(depth - (long long)minus[g]);
    const unsigned long long v = err64[g];
    for (int i = 0; i < 4; i++) e.err_cnt[i] = (int32_t)((v >> (16 * i)) & 0xffff);
    e.ref_base = contig_seq[tid][x];
    out[idx[g]] = e;
}

#include "spike_chain.cuh"

} // namespace

#include "spike_run.cuh"
