// spike_chain.cuh -- the reference's random stream and everything that consumes it in order.
// (Included by spike.cu inside its anonymous namespace.)
//
// The reference draws from ONE glibc rand() stream: one selectMutantAllele(ref[pos]) per covered locus
// (stochasticSpike.c:1197; it redraws while the pick equals the reference base, :350-354) plus the coin tosses
// and extra picks of attemptToMutateBase at every target (:526-904).  The offset at which a target tosses is
// therefore the end of a data-dependent walk over every covered locus before it.
//
// B200 formulation:
//   rng_fill      the stream itself is generated in parallel by polynomial skip-ahead (rng_glibc.cuh); next to
//                 the raw values it writes three bit planes (class bit 0, class bit 1, rejected-by-randomNum).
//   cls_pack      the reference classes of the covered loci as three bit planes (bit 0, bit 1, "not GCAT").
//   walk_loci     lock step of draw k+i against locus g+i on 32-bit words: term = ((e0^c0)|(e1^c1)|cx) & ~ej says
//                 which draws end their locus; the run of trailing ones advances both cursors, a zero starts
//                 the "repeat draw" loop of that locus.  ~4 loci per iteration.
//   phase 1       the walk is a monotone map k_in -> k_out per stretch of loci, and walkers that meet stay
//                 together.  Chunks are taken in groups; for a group EVERY start offset of a +-4 sigma window
//                 around the expected offset (mean 4/3 draw per GCAT locus, variance 4/9) is simulated, and
//                 duplicates are dropped at geometrically spaced checkpoints: W walkers shrink like W/sqrt(loci),
//                 so a group of length L costs ~2 W sqrt(L) walker-loci instead of W L -- the longer the group the
//                 less work per locus.  The window is cut into slices (one block each; the host sizes groups and
//                 slices so that all blocks are resident at once), and the survivors at every chunk end inside the
//                 group are recorded.  A walker step resolves up to six "draw ends nothing" conflicts per set of
//                 loads (walk_seg).  Targets are dry-run per walker.
//   phase 2       one warp composes the group maps in order (a table lookup per group); then every chunk looks up
//                 its exact start offset in its group's recorded survivors.
//   phase 3       one warp per chunk repeats the walk from its exact offset and applies the targets for real
//                 (speculative 32-entry batches).  Exit offsets must equal the next chunk's start (checked).
//   fallback      a window miss, an inconsistent exit, a dry-run that was too complex, or any "odd patch"
//                 (which changes bases later targets see) reruns phase 3 as ONE chunk = the plain serial chain.
#pragma once

// ------------------------------------------------------------------------------------------
// glibc rand() stream
// ------------------------------------------------------------------------------------------
struct RngTables {
    uint32_t seg[RNG_TPB][GLIBC_DEG];     // x^(t * RNG_SEG) mod P
};

// out[i] = rand() #(k_base + i) for i in [0, M): thread (b, t) produces outputs [b*RNG_BLOCK + t*RNG_SEG, +RNG_SEG).
// e0/e1/ej (optional): bit planes of the same outputs, bit i of word w <-> output 32w + i.
__global__ void __launch_bounds__(RNG_TPB)
rng_fill_kernel(const uint32_t *__restrict__ block_poly /* [nblocks][31]: x^(310 + k_base + b*RNG_BLOCK) */, const RngTables *__restrict__ tab,
                const uint32_t *__restrict__ seedw /* 61 words */, int32_t *__restrict__ out, unsigned long long M,
                uint32_t *__restrict__ e0, uint32_t *__restrict__ e1, uint32_t *__restrict__ ej)
{
    __shared__ uint32_t s_w[61];
    __shared__ uint32_t s_bp[GLIBC_DEG];
    if (threadIdx.x < 61) s_w[threadIdx.x] = seedw[threadIdx.x];
    if (threadIdx.x < GLIBC_DEG) s_bp[threadIdx.x] = block_poly[(size_t)blockIdx.x * GLIBC_DEG + threadIdx.x];
    __syncthreads();
    const unsigned long long k0 = (unsigned long long)blockIdx.x * RNG_BLOCK + (unsigned long long)threadIdx.x * RNG_SEG;
    if (k0 >= M) return;
    uint32_t a[GLIBC_DEG], b[GLIBC_DEG], c[GLIBC_DEG], h[GLIBC_DEG];
    for (int i = 0; i < GLIBC_DEG; i++) { a[i] = s_bp[i]; b[i] = tab->seg[threadIdx.x][i]; }
    glibc_poly_mulmod(a, b, c);
    glibc_history(c, s_w, h);                        // h[t] = r[344 + k0 - 31 + t]
    unsigned long long k = k0;
    const unsigned long long kend = (k0 + RNG_SEG < M) ? k0 + RNG_SEG : M;
    uint32_t w0 = 0, w1 = 0, wj = 0;
    while (k < kend) {
#pragma unroll
        for (int i = 0; i < GLIBC_DEG; i++) {        // new word replaces r[n-31]; r[n-3] sits three slots back
            h[i] = h[i] + h[(i + 28) % GLIBC_DEG];
            if (k < kend) {
                const uint32_t r = h[i] >> 1;
                out[k] = (int32_t)r;
                const uint32_t bit = (uint32_t)(k & 31);
                w0 |= (r & 1u) << bit; w1 |= ((r >> 1) & 1u) << bit; wj |= (r >= GLIBC_CUT4 ? 1u : 0u) << bit;
                if (bit == 31 || k + 1 == kend) {
                    if (e0) { e0[k >> 5] = w0; e1[k >> 5] = w1; ej[k >> 5] = wj; }
                    w0 = w1 = wj = 0;
                }
            }
            k++;
        }
    }
}

// reference classes of covered loci [0, n) -> bit planes (bit 0, bit 1, "other")
__global__ void cls_pack_kernel(const uint8_t *__restrict__ cls, int64_t n, uint32_t *__restrict__ c0, uint32_t *__restrict__ c1, uint32_t *__restrict__ cx)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t c = g < n ? cls[g] : 4u;
    const uint32_t b0 = __ballot_sync(0xffffffffu, c & 1u), b1 = __ballot_sync(0xffffffffu, c & 2u), bx = __ballot_sync(0xffffffffu, c == 4u);
    if ((threadIdx.x & 31) == 0 && (g >> 5) <= ((n + 31) >> 5)) { c0[g >> 5] = b0; c1[g >> 5] = b1; cx[g >> 5] = bx; }
}

// ------------------------------------------------------------------------------------------
// shared state of the chain kernels
// ------------------------------------------------------------------------------------------
struct ChainArgs {
    const uint32_t *e0, *e1, *ej; const int32_t *R; unsigned long long M;      // draws [0, M), M a multiple of 32 (+2 words of padding)
    const uint32_t *c0, *c1, *cx; int64_t n_walk;                               // covered loci [0, n_walk)
    const HitTarget *hits; size_t H;
    const unsigned long long *eoff; PlpEntry *ent; uint8_t *hflag;
    ssb_target_result *res;
    Patch *patches; unsigned int *n_patches; unsigned int patch_cap;
    OddPatch *odd; unsigned int *n_odd; unsigned int odd_cap; unsigned long long *odd_bloom;
    const uint8_t *const *contig_seq;
    DevErr *err;
};

struct ChunkDesc { int64_t g0, g1; unsigned long long k_in, k_out; };            // k_out = ~0: unknown (stop after the last target, no check)
constexpr unsigned long long CHUNK_WALK_ONLY = ~0ull - 1;                        // k_out: walk to the end of the chunk, nothing to compare with
enum { CHAIN_OVERRUN = 1, CHAIN_MISS = 2, CHAIN_COMPLEX = 4, CHAIN_INCONSISTENT = 8 };

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Consumes the draws of covered loci [g, g_to): per locus, rand() until the pick differs from the reference base
// (selectMutantAllele / randomNum, stochasticSpike.c:283-302, 338-360).  false = the stream is too short.
// Cursors are kept as 32-bit offsets from word-aligned bases.  Instead of testing the end of the stream in the
// loop, word indices are clamped into the padding behind the planes, which holds all four classes in every nibble
// (e0 = 0xAAAAAAAA, e1 = 0xCCCCCCCC, ej = 0): a walker that runs off the end still terminates, and is caught by the
// single test at the end.
template <bool PF>
__device__ __forceinline__ bool walk_loci(const ChainArgs &A, int64_t &g, const int64_t g_to, unsigned long long &k)
{
    while (g < g_to) {
        if (k + 64 > A.M) return false;
        const unsigned long long kb = k & ~31ull; const int64_t gb = g & ~(int64_t)31;
        const uint32_t *__restrict__ E0 = A.e0 + (kb >> 5), *__restrict__ E1 = A.e1 + (kb >> 5), *__restrict__ EJ = A.ej + (kb >> 5);
        const uint32_t *__restrict__ C0 = A.c0 + (gb >> 5), *__restrict__ C1 = A.c1 + (gb >> 5), *__restrict__ CX = A.cx + (gb >> 5);
        uint32_t kr = (uint32_t)(k - kb), gr = (uint32_t)(g - gb);
        const uint32_t gto = (g_to - gb) > 0x40000000ll ? 0x40000000u : (uint32_t)(g_to - gb);
        const unsigned long long wleft = ((A.M - kb) >> 5) + 100ull;
        const uint32_t wmax = wleft > 0x02000000ull ? 0x02000000u : (uint32_t)wleft;       // last word index that may be read
        // the current word of every plane stays in registers; it is reloaded only when a cursor crosses a word boundary
        uint32_t cwe = 0xffffffffu, cwc = 0xffffffffu, E0w = 0, E1w = 0, EJw = 0, C0w = 0, C1w = 0, CXw = 0;
        while (gr < gto) {
            const uint32_t a = kr & 31u, b = gr & 31u;
            const uint32_t we = min(kr >> 5, wmax), wc = gr >> 5;
            if (we != cwe) {
                cwe = we; E0w = E0[we]; E1w = E1[we]; EJw = EJ[we];
                if (PF && (we & 31u) == 0) { prefetch_l2(E0 + we + 64); prefetch_l2(E1 + we + 64); prefetch_l2(EJ + we + 64); }
            }
            if (wc != cwc) {
                cwc = wc; C0w = C0[wc]; C1w = C1[wc]; CXw = CX[wc];
                if (PF && (wc & 31u) == 0) { prefetch_l2(C0 + wc + 64); prefetch_l2(C1 + wc + 64); prefetch_l2(CX + wc + 64); }
            }
            const uint32_t c0 = C0w >> b, c1 = C1w >> b, cx = CXw >> b;
            const uint32_t n = min(min(32u - a, 32u - b), gto - gr);
            const uint32_t term = ((((E0w >> a) ^ c0) | ((E1w >> a) ^ c1) | cx)) & ~(EJw >> a);       // bit i: draw k+i ends locus g+i
            const uint32_t t = (uint32_t)__ffs(~term) - 1u;                // trailing ones; 0xffffffff when term is all ones
            if (t >= n) { gr += n; kr += n; continue; }
            gr += t; kr += t;
            // draw k repeats the reference base of locus g (or was rejected): keep drawing for this locus
            const uint32_t m0 = 0u - ((c0 >> t) & 1u), m1 = 0u - ((c1 >> t) & 1u), mx = 0u - ((cx >> t) & 1u);
            for (;;) {
                const uint32_t w = min(kr >> 5, wmax);
                if (w != cwe) { cwe = w; E0w = E0[w]; E1w = E1[w]; EJw = EJ[w]; }
                const uint32_t ends = (((E0w ^ m0) | (E1w ^ m1) | mx) & ~EJw) >> (kr & 31u);
                if (ends == 0u) { kr = (kr | 31u) + 1u; continue; }
                kr += (uint32_t)__ffs(ends);                               // the ending draw is consumed too
                break;
            }
            gr += 1;
            if (kr > 0x7f000000u) break;                                   // re-base before the 32-bit cursor can wrap
        }
        k = kb + kr; g = gb + gr;
    }
    return k + 64 <= A.M;
}

__device__ __forceinline__ bool next_rand(const ChainArgs &A, unsigned long long &k, uint32_t &r)
{
    if (k + 64 > A.M) return false;
    r = (uint32_t)A.R[k++];
    return true;
}
// selectMutantAllele(wild) (:338-360): index into "GCAT" of the pick; wild_idx 4 = not one of GCAT
__device__ __forceinline__ bool select_allele(const ChainArgs &A, unsigned long long &k, uint32_t wild_idx, uint32_t &pick)
{
    for (;;) {
        uint32_t r;
        if (!next_rand(A, k, r)) return false;
        if (r >= GLIBC_CUT4) continue;
        if ((r & 3u) != wild_idx) { pick = r & 3u; return true; }
    }
}
__device__ __forceinline__ uint32_t locus_class(const ChainArgs &A, int64_t g)
{
    const size_t w = (size_t)(g >> 5); const uint32_t b = (uint32_t)(g & 31);
    if ((A.cx[w] >> b) & 1u) return 4u;
    return ((A.c0[w] >> b) & 1u) | (((A.c1[w] >> b) & 1u) << 1);
}

// Outcome of one pileup entry at a target locus, computed without side effects so that it can be evaluated
// speculatively (attemptToMutateBase, stochasticSpike.c:526-904; cases as in SURVEY App. A).
struct EntryOut {
    uint32_t draws;        // rand() values consumed
    uint8_t mark_self, mark_mate, filt /* 0 none, 1 P(ass), 2 K(masked), 3 O(vl) */, tally /* 0 none,1 ref,2 mut,3..6 err G,C,A,T */;
    uint8_t npatch; uint8_t pbase[2]; uint8_t pmate[2];   // patch i: base pbase[i] on (pmate[i] ? mate : self)
    bool ok;
};

// have_first: the caller already holds rand() #k (first_r), fetched together with its neighbours' draws
__device__ EntryOut entry_eval(const ChainArgs &A, const PlpEntry &e, uint8_t mate_base, uint8_t mate_bq, bool mate_handled, bool self_handled,
                               unsigned long long k, uint32_t thresh, uint8_t F, uint8_t Aallele, bool have_first = false, uint32_t first_r = 0)
{
    EntryOut o; o.draws = 0; o.mark_self = o.mark_mate = o.filt = o.tally = o.npatch = 0; o.ok = true;
    o.pbase[0] = o.pbase[1] = o.pmate[0] = o.pmate[1] = 0;
    if (e.skip || e.bq == 0 || self_handled) return o;                               // :1270
    uint8_t R = e.base, M = 0; int rbq = e.bq, mbq = 0;
    if (e.mate >= 0 && !mate_handled) { M = mate_base; mbq = mate_bq; }               // getBaseWithRPOcheck :387-432
    if (M == 'N') mbq = 0;
    if (R == 'N') rbq = 0;
    uint8_t base = R;
    if (M && M != R && mbq > rbq) base = M;
    if (base == 'N') { o.mark_self = 1; o.mark_mate = M ? 1 : 0; return o; }         // :584-592
    const unsigned long long k0 = k;
    uint32_t r;
    if (have_first) { if (k + 64 > A.M) { o.ok = false; return o; } r = first_r; k++; }
    else if (!next_rand(A, k, r)) { o.ok = false; return o; }
    const bool heads = r < thresh;                                                    // coinToss :332-335
    auto tally_base = [&](uint8_t b) { int gi = gcat_index(b); o.tally = gi < 4 ? (uint8_t)(3 + gi) : 0; };
    auto other = [&](uint8_t &d) -> bool {                                            // selectMutantAllele(A)
        uint32_t pick; if (!select_allele(A, k, (uint32_t)gcat_index(Aallele), pick)) return false;
        d = (uint8_t)"GCAT"[pick]; return true;
    };
    if (!heads) {
        if (base == F) o.tally = 1;
        else { tally_base(base); o.mark_self = 1; o.mark_mate = M ? 1 : 0; }
    } else if (!M && R == F) {                                                        // case 1
        o.pbase[0] = Aallele; o.pmate[0] = 0; o.npatch = 1; o.tally = 2; o.filt = 1; o.mark_self = 1;
    } else if (!M) {                                                                  // case 2
        o.filt = 2;
        if (R == Aallele) { uint8_t d; if (!other(d)) { o.ok = false; return o; } o.pbase[0] = d; o.pmate[0] = 0; o.npatch = 1; base = d; }
        tally_base(base); o.mark_self = 1;
    } else if (R == F && M == F) {                                                    // case 3
        o.pbase[0] = Aallele; o.pmate[0] = 0; o.pbase[1] = Aallele; o.pmate[1] = 1; o.npatch = 2;
        o.mark_self = o.mark_mate = 1; o.tally = 2; o.filt = 1;
    } else if (R == F) {                                                              // case 4 (M != F)
        o.pbase[0] = Aallele; o.pmate[0] = 0; o.npatch = 1; o.mark_self = 1;
        if (M == Aallele) { uint8_t d; if (!other(d)) { o.ok = false; return o; } o.pbase[1] = d; o.pmate[1] = 1; o.npatch = 2; if (base == M) base = d; }
        o.mark_mate = 1; o.filt = 3;
        if (base == F) o.tally = 2; else tally_base(base);
    } else if (M == F) {                                                              // case 5 (R != F)
        o.pbase[0] = Aallele; o.pmate[0] = 1; o.npatch = 1; o.mark_mate = 1;
        if (R == Aallele) { uint8_t d; if (!other(d)) { o.ok = false; return o; } o.pbase[1] = d; o.pmate[1] = 0; o.npatch = 2; if (base == R) base = d; }
        o.mark_self = 1; o.filt = 3;
        if (base == F) o.tally = 2; else tally_base(base);
    } else {                                                                          // case 6
        o.filt = 3;
        if (R == Aallele) { uint8_t d; if (!other(d)) { o.ok = false; return o; } o.pbase[o.npatch] = d; o.pmate[o.npatch] = 0; o.npatch++; if (base == R) base = d; }
        if (M == Aallele) { uint8_t d; if (!other(d)) { o.ok = false; return o; } o.pbase[o.npatch] = d; o.pmate[o.npatch] = 1; o.npatch++; if (base == M) base = d; }
        tally_base(base); o.mark_self = o.mark_mate = 1;
    }
    o.draws = (uint32_t)(k - k0);
    return o;
}

// ------------------------------------------------------------------------------------------
// expected draws (mean, variance) per chunk: centres and widths of the phase-1 windows
// ------------------------------------------------------------------------------------------
__global__ void chunk_stats_kernel(const uint32_t *__restrict__ cx, int64_t n_walk, int64_t L, int P, double *__restrict__ mean, double *__restrict__ var)
{
    // one warp per chunk: count the loci whose reference base is not one of GCAT (exactly one draw each)
    const int lane = threadIdx.x & 31;
    const int j = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (j >= P) return;
    const int64_t g0 = (int64_t)j * L, g1 = (g0 + L < n_walk) ? g0 + L : n_walk;
    long long nx = 0;
    for (int64_t w = (g0 >> 5) + lane; w <= ((g1 - 1) >> 5); w += 32) {
        uint32_t v = cx[w];
        const int64_t lo = w << 5;
        if (lo < g0) v &= ~0u << (uint32_t)(g0 - lo);
        if (lo + 32 > g1) v &= (g1 - lo >= 32) ? ~0u : ((1u << (uint32_t)(g1 - lo)) - 1u);
        nx += __popc(v);
    }
    for (int s = 16; s; s >>= 1) nx += __shfl_xor_sync(0xffffffffu, nx, s);
    if (lane == 0) {
        const double n4 = (double)((g1 - g0) - nx);
        atomicAdd(&mean[j], n4 * (4.0 / 3.0) + (double)nx);
        atomicAdd(&var[j], n4 * (4.0 / 9.0));
    }
}

// one warp per hit target: expected number of toss draws and its variance
__global__ void expect_kernel(const HitTarget *__restrict__ hits, size_t H, const unsigned long long *__restrict__ eoff, const PlpEntry *__restrict__ ent,
                              const uint8_t *const *__restrict__ contig_seq, int64_t L, double *__restrict__ mean, double *__restrict__ var)
{
    const int lane = threadIdx.x & 31;
    const size_t h = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (h >= H) return;
    const HitTarget ht = hits[h];
    const uint8_t F = contig_seq[ht.tid][ht.pos];
    const double p = (double)ht.thresh / 2147483648.0;
    const PlpEntry *e = ent + eoff[h];
    const uint32_t n = (uint32_t)(eoff[h + 1] - eoff[h]);
    double m = 0, v = 0;
    for (uint32_t j = lane; j < n; j += 32) {
        const PlpEntry x = e[j];
        if (x.skip || x.bq == 0) continue;
        uint8_t R = x.base, M = 0; int rbq = x.bq, mbq = 0;
        if (x.mate >= 0) { M = e[x.mate].base; mbq = e[x.mate].bq; }
        if (M == 'N') mbq = 0;
        if (R == 'N') rbq = 0;
        uint8_t base = R; if (M && M != R && mbq > rbq) base = M;
        if (base == 'N') continue;
        m += 1.0;
        if (x.mate >= 0) {
            // the mate tosses too only if this entry comes up tails on the reference base (:619-620)
            const PlpEntry y = e[x.mate];
            if (!(y.skip || y.bq == 0 || y.base == 'N')) {
                const double q = (base == F) ? (1.0 - p) : 0.0;
                m -= (1.0 - q); v += q * (1.0 - q);                 // the mate was counted as a sure toss in its own iteration
            }
        }
        v += 0.02;                                                  // extra picks when a read already carries the mutant allele
    }
    for (int s = 16; s; s >>= 1) { m += __shfl_xor_sync(0xffffffffu, m, s); v += __shfl_xor_sync(0xffffffffu, v, s); }
    if (lane == 0) {
        const int j = (int)(ht.locus_index / L);
        atomicAdd(&mean[j], m); atomicAdd(&var[j], v);
    }
}

// ------------------------------------------------------------------------------------------
// phase 1: chunk maps
// ------------------------------------------------------------------------------------------
// attemptToMutateBase over the whole pileup of hit h, counting draws only.  0 ok, else CHAIN_* bits.
// "handled" marks only ever point forward (an entry marks the first LATER entry of its QNAME), so one bit per entry is enough;
// the bits live in local memory (deep panels: thousands of entries per pileup, dozens of marks).
__device__ int dry_apply(const ChainArgs &A, size_t h, int64_t g, unsigned long long &k)
{
    const HitTarget ht = A.hits[h];
    const uint8_t Fb = A.contig_seq[ht.tid][ht.pos];
    uint32_t pick;
    if (!select_allele(A, k, locus_class(A, g), pick)) return CHAIN_OVERRUN;                                 // :1197
    uint8_t allele = (uint8_t)"GCAT"[pick];
    if (ht.base == 'G' || ht.base == 'C' || ht.base == 'A' || ht.base == 'T') allele = ht.base;           // :1199-1203
    const PlpEntry *ents = A.ent + A.eoff[h];
    const uint32_t n = (uint32_t)(A.eoff[h + 1] - A.eoff[h]);
    if (n > (uint32_t)MAX_PILEUP) return CHAIN_COMPLEX;
    uint32_t marks[(MAX_PILEUP + 31) / 32];
    const uint32_t nw = (n + 31) >> 5;
    for (uint32_t i = 0; i < nw; i++) marks[i] = 0;
    for (uint32_t j = 0; j < n; j++) {
        const PlpEntry e = ents[j];
        if (e.skip || e.bq == 0) continue;
        if ((marks[j >> 5] >> (j & 31)) & 1u) continue;
        uint8_t mb = 0, mq = 0; bool mh = false;
        if (e.mate >= 0) { const PlpEntry y = ents[e.mate]; mb = y.base; mq = y.bq; mh = ((marks[(uint32_t)e.mate >> 5] >> ((uint32_t)e.mate & 31)) & 1u) != 0; }
        const EntryOut o = entry_eval(A, e, mb, mq, mh, false, k, ht.thresh, Fb, allele);
        if (!o.ok) return CHAIN_OVERRUN;
        k += o.draws;
        if (o.mark_mate && e.mate >= 0) marks[(uint32_t)e.mate >> 5] |= 1u << ((uint32_t)e.mate & 31);
    }
    return 0;
}

__device__ __forceinline__ size_t first_hit_at_or_after(const HitTarget *hits, size_t H, int64_t g)
{
    size_t lo = 0, hi = H;
    while (lo < hi) { size_t mid = (lo + hi) >> 1; if (hits[mid].locus_index < g) lo = mid + 1; else hi = mid; }
    return lo;
}

// ---- phase 1 on staged planes ------------------------------------------------------------------------------------
// A block owns one SLICE of the start-offset window of one GROUP of consecutive chunks.  All its walkers stand at the
// same locus between rounds, so a round needs only the loci [g, gc) and the draws from the lowest walker up to what the
// highest one can reach: those are staged in shared memory, the three planes of a 32-position word side by side
// (one 16-byte load fetches a word of each plane).
struct SegPlanes { const uint4 *e, *c; unsigned long long kb; int64_t gb; uint32_t we_n; unsigned long long M; };

constexpr int P1_THREADS = 128;
constexpr int P1_SEG     = 4096;               // loci per round at most
constexpr int P1_EW_CAP  = 1024;               // staged draw words (32768 draws)
constexpr int P1_CW_CAP  = P1_SEG / 32 + 2;
constexpr size_t P1_SMEM = (size_t)(P1_EW_CAP + P1_CW_CAP) * sizeof(uint4);

// One step = one window of 32 draws from kr against 32 loci from gr, both shifted into place.  A stage of the step runs the lock step to
// the first draw that does not end its locus (z, one-hot); that locus then takes the next draw of the window that does (y, one-hot).
// Every draw that ends nothing delays the loci by one place against the draws (`skew`), so the next stage compares the same window with
// the locus planes shifted once more: P1_STAGES stages share one set of loads (~19 loci per step instead of ~4; the kernel is bound by
// integer issue: C2, one B200: 1 stage 19.8 ms, 3: 13.9, 4: 13.0, 5: 12.4, 6: 12.2).  No branch and no inner loop: a lone walker is one dependency chain.  `done`: the draws consumed so far (ones below
// the cursor), `nonend`: those of them that ended no locus.  A locus that finds no ending draw in the window (y = 0) takes the rest of
// the window and stays the current locus of the next step; later stages then see a full `done` and change nothing.
constexpr int P1_STAGES = 6;
__device__ __forceinline__ int walk_seg(const SegPlanes &P, uint32_t &gr, const uint32_t gto, uint32_t &kr)
{
    while (gr + 32u <= gto) {                                             // a full window of loci ahead
        const uint32_t a = kr & 31u, b = gr & 31u, we = kr >> 5, wc = gr >> 5;
        if (we + 2u > P.we_n) return (P.kb + kr + 96ull > P.M) ? CHAIN_OVERRUN : CHAIN_COMPLEX;
        const uint4 ea = P.e[we], eb = P.e[we + 1], ca = P.c[wc], cb = P.c[wc + 1];
        const uint32_t e0 = __funnelshift_r(ea.x, eb.x, a), e1 = __funnelshift_r(ea.y, eb.y, a), ej = __funnelshift_r(ea.z, eb.z, a);
        const uint32_t c0 = __funnelshift_r(ca.x, cb.x, b), c1 = __funnelshift_r(ca.y, cb.y, b), cx = __funnelshift_r(ca.z, cb.z, b);
        uint32_t done = 0u, nonend = 0u, skew = 0u;
#pragma unroll
        for (int s = 0; s < P1_STAGES; s++) {
            const uint32_t s0 = c0 << skew, s1 = c1 << skew, sx = cx << skew;      // locus gr + i - skew stands at draw kr + i
            const uint32_t term = (((e0 ^ s0) | (e1 ^ s1) | sx) & ~ej) | done;     // bit i: draw kr+i ends its locus (or is behind the cursor)
            const uint32_t z = ~term & (term + 1u);                                // first draw that does not (0: none, the window is used up)
            const uint32_t m0 = (s0 & z) ? 0xffffffffu : 0u, m1 = (s1 & z) ? 0xffffffffu : 0u, mx = (sx & z) ? 0xffffffffu : 0u;
            const uint32_t ends = ((e0 ^ m0) | (e1 ^ m1) | mx) & ~ej;              // draws of the window that would end that locus
            const uint32_t above = ends & ~(z | (z - 1u));                         // ... after the failed one
            const uint32_t y = above & (0u - above);                               // the first of them (0: none in this window)
            nonend |= y - z;                                                       // draws [z, y) ended nothing (y = 0: from z to the top)
            done = y | (y - 1u);                                                   // cursor behind y (y = 0: behind the window)
            if (s + 1 < P1_STAGES) skew = (uint32_t)__popc(nonend);
        }
        const uint32_t d = (uint32_t)__popc(done);
        kr += d; gr += d - (uint32_t)__popc(nonend);
    }
    while (gr < gto) {                                                    // the last loci of the stretch: one stage, pairs past the end masked
        const uint32_t a = kr & 31u, b = gr & 31u, we = kr >> 5, wc = gr >> 5;
        if (we + 2u > P.we_n) return (P.kb + kr + 96ull > P.M) ? CHAIN_OVERRUN : CHAIN_COMPLEX;
        const uint4 ea = P.e[we], eb = P.e[we + 1], ca = P.c[wc], cb = P.c[wc + 1];
        const uint32_t e0 = __funnelshift_r(ea.x, eb.x, a), e1 = __funnelshift_r(ea.y, eb.y, a), ej = __funnelshift_r(ea.z, eb.z, a);
        const uint32_t c0 = __funnelshift_r(ca.x, cb.x, b), c1 = __funnelshift_r(ca.y, cb.y, b), cx = __funnelshift_r(ca.z, cb.z, b);
        const uint32_t n = min(32u, gto - gr);
        const uint32_t beyond = n >= 32u ? 0u : 0xffffffffu << n;         // pairs past the end of the stretch never stop the lock step
        const uint32_t term = (((e0 ^ c0) | (e1 ^ c1) | cx) & ~ej) | beyond;   // bit i: draw kr+i ends locus gr+i
        const uint32_t z = ~term & (term + 1u);                            // lowest pair that does not (0: none)
        const uint32_t m0 = (c0 & z) ? 0xffffffffu : 0u, m1 = (c1 & z) ? 0xffffffffu : 0u, mx = (cx & z) ? 0xffffffffu : 0u;
        const uint32_t ends = ((e0 ^ m0) | (e1 ^ m1) | mx) & ~ej;           // draws of the window that would end that locus
        const uint32_t above = ends & ~(z | (z - 1u));                     // ... after the failed one
        const uint32_t y = above & (0u - above);                           // the first of them (0: none in this window)
        const uint32_t t = min((uint32_t)__popc(z - 1u), n);               // loci passed in lock step
        gr += t + (y ? 1u : 0u);
        kr += y ? (uint32_t)__popc(y - 1u) + 1u : (z ? 32u : n);
    }
    return 0;
}

// walk [g, g_to) including the targets inside, counting draws only
__device__ int dry_walk(const ChainArgs &A, const SegPlanes &P, int64_t g, const int64_t g_to, size_t h, unsigned long long &k)
{
    if (k < P.kb) return CHAIN_COMPLEX;
    uint32_t gr = (uint32_t)(g - P.gb), kr = (uint32_t)(k - P.kb);
    int rc = 0;
    while (h < A.H && A.hits[h].locus_index < g_to) {
        const int64_t gt = A.hits[h].locus_index;
        if ((rc = walk_seg(P, gr, (uint32_t)(gt - P.gb), kr))) return rc;
        k = P.kb + kr;
        if ((rc = dry_apply(A, h, gt, k))) return rc;
        if (k - P.kb >= ((unsigned long long)P.we_n << 5)) return (k + 96ull > P.M) ? CHAIN_OVERRUN : CHAIN_COMPLEX;
        kr = (uint32_t)(k - P.kb); gr = (uint32_t)(gt + 1 - P.gb); h++;
    }
    if ((rc = walk_seg(P, gr, (uint32_t)(g_to - P.gb), kr))) return rc;
    k = P.kb + kr;
    return 0;
}

// group q = chunks [f0, f0 + nf): one start-offset window [klo, klo + W), cut into S slices of w offsets (blocks b0 ..)
struct GroupDesc { unsigned long long klo; uint32_t W, w, S, b0; int32_t f0, nf; unsigned long long toff; };   // toff: walker slot of window index 0 (= where the group's entry -> exit table begins)
struct SliceDesc { int32_t q; uint32_t i0, n; unsigned long long off; };        // window indices [i0, i0 + n); walker slots at off
// survivors of one slice at the end of one chunk: (lowest window index of the class, draw offset) pairs in `pool`
struct BoundaryList { unsigned long long off; uint32_t cnt; uint32_t pad; };

__device__ __forceinline__ uint32_t isqrt_up(uint32_t x) { uint32_t r = (uint32_t)sqrtf((float)x) + 1u; return r; }

// One block per slice.  kbuf/lobuf: two ping-pong halves of `stride` slots each.
__global__ void __launch_bounds__(P1_THREADS)      // (forcing 12 blocks per SM = 40 registers was measured: 12.6 ms instead of 11.7)
phase1_kernel(ChainArgs A, int64_t L, const GroupDesc *__restrict__ groups, const SliceDesc *__restrict__ slices,
              unsigned long long *__restrict__ kbuf, uint32_t *__restrict__ lobuf, unsigned long long stride,
              BoundaryList *__restrict__ lists /* [block][max_nf] */, int max_nf, unsigned long long *__restrict__ pool_k, uint32_t *__restrict__ pool_lo,
              unsigned long long *__restrict__ pool_used, unsigned long long pool_cap, unsigned int *__restrict__ flags, unsigned long long *__restrict__ dbg,
              int block0 /* index of this launch's first slice (a retry launches single slices) */)
{
    extern __shared__ uint4 p1_smem[];
    uint4 *se = p1_smem, *sc = p1_smem + P1_EW_CAP;
    __shared__ uint32_t s_warp[P1_THREADS / 32];
    __shared__ int s_bad;
    __shared__ unsigned long long s_off, s_kmin, s_kmax;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned int bx = blockIdx.x + (unsigned int)block0;
    const SliceDesc sd = slices[bx];
    const GroupDesc gd = groups[sd.q];
    const int64_t g0 = (int64_t)gd.f0 * L, gend = ((int64_t)(gd.f0 + gd.nf) * L < A.n_walk) ? (int64_t)(gd.f0 + gd.nf) * L : A.n_walk;
    unsigned long long *kb[2] = {kbuf + sd.off, kbuf + stride + sd.off};
    uint32_t *lb[2] = {lobuf + sd.off, lobuf + stride + sd.off};
    uint32_t alive = sd.n;
    for (uint32_t i = tid; i < alive; i += P1_THREADS) { kb[0][i] = gd.klo + sd.i0 + i; lb[0][i] = sd.i0 + i; }
    if (tid == 0) { s_bad = 0; s_kmin = gd.klo + sd.i0; s_kmax = gd.klo + sd.i0 + sd.n - 1; }
    __syncthreads();
    int cur = 0, r = 0;
    int64_t g = g0, step = 64;
    const unsigned long long plane_words = (A.M >> 5) + 160ull;              // words the draw planes hold (padding included)
    long long t_prev = dbg ? clock64() : 0, t_start = t_prev; unsigned long long t_early = 0;
    while (g < gend) {
        if (dbg && tid == 0) { const long long t = clock64(); if (alive > (uint32_t)P1_THREADS) t_early += (unsigned long long)(t - t_prev); atomicAdd(&dbg[alive > (uint32_t)P1_THREADS ? 4 : 5], (unsigned long long)(t - t_prev)); t_prev = t; }
        const int64_t fine_end = (g0 + (int64_t)(r + 1) * L < gend) ? g0 + (int64_t)(r + 1) * L : gend;
        int64_t gc = g + step; if (gc > fine_end || fine_end - gc < step / 2) gc = fine_end;
        if (gc - g > P1_SEG) gc = g + P1_SEG;
        const unsigned long long kmin = s_kmin, kmax = s_kmax;               // lowest / highest walker (targets can reorder walkers)
        const unsigned long long kbase = kmin & ~31ull;
        const size_t h0 = first_hit_at_or_after(A.hits, A.H, g);
        // draws the highest walker can reach in this round: 4/3 per locus and 8 sigma, plus the pileups of the targets inside
        uint32_t we_n;
        for (;;) {
            const size_t h1 = first_hit_at_or_after(A.hits, A.H, gc);
            const uint32_t len = (uint32_t)(gc - g);
            const unsigned long long need = (kmax - kbase) + (unsigned long long)len + len / 3u + 8ull * isqrt_up(len) + 3ull * (A.eoff[h1] - A.eoff[h0]) + 64ull * (h1 - h0) + 192ull;
            const unsigned long long w = (need >> 5) + 3ull;
            if (w <= (unsigned long long)P1_EW_CAP) { we_n = (uint32_t)w; break; }
            if (gc - g <= 64) { if (tid == 0) atomicOr(flags, (unsigned int)CHAIN_COMPLEX); return; }     // the slice itself does not fit
            gc = g + (((gc - g) / 2 + 31) & ~(int64_t)31);
        }
        {
            const unsigned long long ew0 = kbase >> 5; const size_t cw0 = (size_t)(g >> 5);
            const uint32_t wc_n = (uint32_t)((gc - g + 31) >> 5) + 2u;
            for (uint32_t i = tid; i < we_n; i += P1_THREADS) {
                uint4 v;
                if (ew0 + i < plane_words) { v.x = A.e0[ew0 + i]; v.y = A.e1[ew0 + i]; v.z = A.ej[ew0 + i]; }
                else { v.x = 0xAAAAAAAAu; v.y = 0xCCCCCCCCu; v.z = 0u; }
                v.w = 0; se[i] = v;
            }
            for (uint32_t i = tid; i < wc_n; i += P1_THREADS) { uint4 v; v.x = A.c0[cw0 + i]; v.y = A.c1[cw0 + i]; v.z = A.cx[cw0 + i]; v.w = 0; sc[i] = v; }
        }
        __syncthreads();
        SegPlanes SP; SP.e = se; SP.c = sc; SP.kb = kbase; SP.gb = g & ~(int64_t)31; SP.we_n = we_n; SP.M = A.M;
        int bad = 0;
        if (dbg && tid == 0) { atomicAdd(&dbg[0], (unsigned long long)alive * (unsigned long long)(gc - g)); atomicAdd(&dbg[3], 1ull); }
        if (tid == 0) { s_kmin = ~0ull; s_kmax = 0ull; }                    // every thread has read them; the barrier above orders this
        unsigned long long tmin = ~0ull, tmax = 0ull;
        for (uint32_t i = tid; i < alive; i += P1_THREADS) {
            unsigned long long k = kb[cur][i];
            bad |= dry_walk(A, SP, g, gc, h0, k);
            kb[cur][i] = k;
            if (k < tmin) tmin = k;
            if (k > tmax) tmax = k;
        }
        if (bad) atomicOr(&s_bad, bad);
        __syncthreads();
        if (tmin != ~0ull) { atomicMin(&s_kmin, tmin); atomicMax(&s_kmax, tmax); }
        if (s_bad) { if (tid == 0) atomicOr(flags, (unsigned int)s_bad); return; }
        // drop walkers that met their left neighbour (they stay together from here on); order is kept
        uint32_t total = 0;
        for (uint32_t base = 0; base < alive; base += P1_THREADS) {
            const uint32_t i = base + tid;
            bool keep = false; unsigned long long k = 0; uint32_t lo = 0;
            if (i < alive) { k = kb[cur][i]; lo = lb[cur][i]; keep = (i == 0) || (kb[cur][i - 1] != k); }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) s_warp[wid] = __popc(m);
            __syncthreads();
            uint32_t before = 0, tile_total = 0;
            for (int w = 0; w < P1_THREADS / 32; w++) { const uint32_t c = s_warp[w]; if (w < wid) before += c; tile_total += c; }
            if (keep) { const uint32_t o = total + before + __popc(m & ((1u << lane) - 1u)); kb[cur ^ 1][o] = k; lb[cur ^ 1][o] = lo; }
            total += tile_total;
            __syncthreads();
        }
        alive = total; cur ^= 1;
        g = gc; if (step < P1_SEG) step *= 2;
        if (g == fine_end) {                              // end of chunk f0 + r: the survivors are that boundary's map
            if (tid == 0) s_off = atomicAdd(pool_used, (unsigned long long)alive);
            __syncthreads();
            const unsigned long long off = s_off;
            if (off + alive > pool_cap) { if (tid == 0) atomicOr(flags, (unsigned int)CHAIN_COMPLEX); return; }
            for (uint32_t i = tid; i < alive; i += P1_THREADS) { pool_k[off + i] = kb[cur][i]; pool_lo[off + i] = lb[cur][i]; }
            if (tid == 0) { BoundaryList bl; bl.off = off; bl.cnt = alive; bl.pad = 0; lists[(size_t)bx * max_nf + r] = bl; }
            r++;
        }
        __syncthreads();
    }
    if (tid == 0 && dbg) {
        atomicAdd(&dbg[1], (unsigned long long)alive); atomicMax(&dbg[2], (unsigned long long)alive);
        const unsigned long long tot = (unsigned long long)(clock64() - t_start);
        atomicMax(&dbg[6], tot);
        dbg[8 + 2 * (size_t)bx] = tot; dbg[9 + 2 * (size_t)bx] = t_early;       // per block: total, early rounds
    }
}

// draw offset at the end of chunk r of group gd, for the walker that entered the group at offset k: the class of its
// slice with the largest lowest-index <= its own window index
__device__ __forceinline__ bool boundary_lookup(const GroupDesc &gd, int r, unsigned long long k, const BoundaryList *__restrict__ lists, int max_nf,
                                                const unsigned long long *__restrict__ pool_k, const uint32_t *__restrict__ pool_lo, unsigned long long &k_out)
{
    if (k < gd.klo || k - gd.klo >= gd.W) return false;
    const uint32_t idx = (uint32_t)(k - gd.klo);
    uint32_t sl = idx / gd.w; if (sl >= gd.S) sl = gd.S - 1;
    const BoundaryList bl = lists[(size_t)(gd.b0 + sl) * max_nf + r];
    const uint32_t *lo = pool_lo + bl.off;
    uint32_t a = 0, b = bl.cnt;                         // last i with lo[i] <= idx (lo[0] = first index of the slice <= idx)
    while (b - a > 1) { const uint32_t mid = (a + b) >> 1; if (lo[mid] <= idx) a = mid; else b = mid; }
    k_out = pool_k[bl.off + a];
    return true;
}

// phase 2a, preparation: the map of a group as a flat table, exit offset per window index (the survivors of a slice at the group's last chunk end
// are classes of consecutive window indices).  It is written over the walker slots of phase 1, which are free by now: one block per slice.
__global__ void __launch_bounds__(128)
map_fill_kernel(const GroupDesc *__restrict__ groups, const SliceDesc *__restrict__ slices, const BoundaryList *__restrict__ lists, int max_nf,
                const unsigned long long *__restrict__ pool_k, const uint32_t *__restrict__ pool_lo, unsigned long long *__restrict__ table, int block0)
{
    const unsigned int bx = blockIdx.x + (unsigned int)block0;
    const SliceDesc sd = slices[bx];
    const GroupDesc gd = groups[sd.q];
    const BoundaryList bl = lists[(size_t)bx * max_nf + (gd.nf - 1)];
    unsigned long long *t = table + sd.off;                        // window index sd.i0 + j <-> t[j]
    for (uint32_t i = threadIdx.x; i < bl.cnt; i += blockDim.x) {
        const uint32_t a = pool_lo[bl.off + i] - sd.i0, b = (i + 1 < bl.cnt) ? pool_lo[bl.off + i + 1] - sd.i0 : sd.n;
        const unsigned long long k = pool_k[bl.off + i];
        for (uint32_t j = a; j < b; j++) t[j] = k;
    }
}

// phase 2a: the exact walker goes through the groups in order from the exact entry offset k_in -- one dependent load per group (the next group's
// descriptor is fetched while the table answers).  gk[q] = exact draw offset at the start of group q.
__global__ void __launch_bounds__(32)
compose_kernel(int G, const GroupDesc *__restrict__ groups, const unsigned long long *__restrict__ table,
               const unsigned long long *__restrict__ k_in, unsigned long long *__restrict__ gk, unsigned long long *__restrict__ k_end, unsigned int *__restrict__ flags,
               unsigned long long *__restrict__ miss /* [0] group whose window the walker missed, [1] its exact entry offset */)
{
    if (threadIdx.x) return;
    unsigned long long k = *k_in;
    GroupDesc gd = groups[0];
    for (int q = 0; q < G; q++) {
        const GroupDesc nx = groups[q + 1 < G ? q + 1 : q];
        gk[q] = k;
        if (k < gd.klo || k - gd.klo >= gd.W) { miss[0] = (unsigned long long)q; miss[1] = k; atomicOr(flags, (unsigned int)CHAIN_MISS); return; }
        k = table[gd.toff + (k - gd.klo)];
        gd = nx;
    }
    *k_end = k;
}

// A shard that is entered with an offset it does not know yet (its predecessors are still working) prepares the answer:
// for every survivor class of the FIRST group's last boundary, the offset at the end of the shard's last group.  When the exact
// entry offset arrives, the exit offset is one lookup (entry_kernel) and can travel on at once.
__global__ void precompose_kernel(int G, const GroupDesc *__restrict__ groups, const BoundaryList *__restrict__ lists, int max_nf,
                                  const unsigned long long *__restrict__ pool_k, const uint32_t *__restrict__ pool_lo, unsigned long long *__restrict__ exit_k)
{
    const GroupDesc g0 = groups[0];
    for (uint32_t sl = blockIdx.x; sl < g0.S; sl += gridDim.x) {
        const BoundaryList bl = lists[(size_t)(g0.b0 + sl) * max_nf + (g0.nf - 1)];
        for (uint32_t i = threadIdx.x; i < bl.cnt; i += blockDim.x) {
            unsigned long long k = pool_k[bl.off + i];
            bool ok = true;
            for (int q = 1; q < G && ok; q++) {
                const GroupDesc gd = groups[q];
                unsigned long long kn;
                ok = boundary_lookup(gd, gd.nf - 1, k, lists, max_nf, pool_k, pool_lo, kn);
                k = kn;
            }
            exit_k[bl.off + i] = ok ? k : ~0ull;
        }
    }
}

// exact entry offset -> offset at the end of the shard (one thread); ~0 when the offset lies outside the simulated window
__global__ void entry_kernel(const GroupDesc *__restrict__ groups, const BoundaryList *__restrict__ lists, int max_nf, const uint32_t *__restrict__ pool_lo,
                             const unsigned long long *__restrict__ exit_k, const unsigned long long *__restrict__ k_in, unsigned long long *__restrict__ k_out)
{
    if (threadIdx.x || blockIdx.x) return;
    const GroupDesc gd = groups[0];
    const unsigned long long k = *k_in;
    if (k < gd.klo || k - gd.klo >= gd.W) { *k_out = ~0ull; return; }
    const uint32_t idx = (uint32_t)(k - gd.klo);
    uint32_t sl = idx / gd.w; if (sl >= gd.S) sl = gd.S - 1;
    const BoundaryList bl = lists[(size_t)(gd.b0 + sl) * max_nf + (gd.nf - 1)];
    const uint32_t *lo = pool_lo + bl.off;
    uint32_t a = 0, b = bl.cnt;
    while (b - a > 1) { const uint32_t mid = (a + b) >> 1; if (lo[mid] <= idx) a = mid; else b = mid; }
    *k_out = bl.cnt ? exit_k[bl.off + a] : ~0ull;
}

// phase 2b: every chunk learns its exact entry and exit offsets from its group's boundary lists
__global__ void boundary_kernel(int P, int nf_per_group, const GroupDesc *__restrict__ groups, const BoundaryList *__restrict__ lists, int max_nf,
                                const unsigned long long *__restrict__ pool_k, const uint32_t *__restrict__ pool_lo,
                                const unsigned long long *__restrict__ gk, ChunkDesc *__restrict__ chunks, unsigned int *__restrict__ flags)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= P) return;
    const int q = f / nf_per_group, r = f - q * nf_per_group;
    const GroupDesc gd = groups[q];
    const unsigned long long k = gk[q];
    unsigned long long kin = k, kout = 0;
    bool ok = true;
    if (r > 0) ok = boundary_lookup(gd, r - 1, k, lists, max_nf, pool_k, pool_lo, kin);
    ok = ok && boundary_lookup(gd, r, k, lists, max_nf, pool_k, pool_lo, kout);
    if (!ok) { atomicOr(flags, (unsigned int)CHAIN_MISS); return; }
    chunks[f].k_in = kin; chunks[f].k_out = kout;
}

// ------------------------------------------------------------------------------------------
// phase 3 / serial chain: one warp per chunk, exact
// ------------------------------------------------------------------------------------------
// STAGED (the one-warp serial chain, launched with CK_SMEM bytes of dynamic shared memory): the pileup of the current target, its
// handled flags and the draws it can toss with are staged in shared memory, so that a batch of 32 entries costs no round trip to
// global memory at all -- what makes deep panels (thousands of entries per target) run at ~10 ns per entry instead of 47.
constexpr uint32_t CK_CAP = (uint32_t)MAX_PILEUP;
constexpr size_t CK_SMEM = (size_t)CK_CAP * sizeof(PlpEntry) + CK_CAP + (size_t)(CK_CAP + 64) * sizeof(int32_t) + 64;
template <bool STAGED>
__global__ void __launch_bounds__(128)
chain_kernel(ChainArgs A, const ChunkDesc *__restrict__ chunks, int n_chunks, unsigned long long *__restrict__ draws_out, unsigned int *__restrict__ flags)
{
    extern __shared__ uint4 ck_smem[];
    const int lane = threadIdx.x & 31;
    const int c = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (c >= n_chunks) return;
    const ChunkDesc cd = chunks[c];
    int64_t g = cd.g0; unsigned long long k = cd.k_in;
    unsigned long long odd_bloom = (n_chunks == 1) ? *A.odd_bloom : 0ull;       // one chunk = the serial chain: odd patches handed in by an earlier shard are in the list already
    size_t h = first_hit_at_or_after(A.hits, A.H, g);
    for (; h < A.H && A.hits[h].locus_index < cd.g1; h++) {
        const HitTarget ht = A.hits[h];
        if (!walk_loci<true>(A, g, ht.locus_index, k)) { if (lane == 0) atomicOr(flags, (unsigned int)CHAIN_OVERRUN); return; }
        // ---- the target locus itself -----------------------------------------------------------
        const unsigned long long k_at = k;
        const uint8_t Fb = A.contig_seq[ht.tid][ht.pos];
        uint32_t pick;
        if (!select_allele(A, k, locus_class(A, g), pick)) { if (lane == 0) atomicOr(flags, (unsigned int)CHAIN_OVERRUN); return; }     // :1197
        uint8_t allele = (uint8_t)"GCAT"[pick];
        if (ht.base == 'G' || ht.base == 'C' || ht.base == 'A' || ht.base == 'T') allele = ht.base;                // :1199-1203
        const unsigned long long e0 = A.eoff[h], e1 = A.eoff[h + 1];
        PlpEntry *ents = A.ent + e0;
        uint8_t *hf = A.hflag + e0;
        const uint32_t n = (uint32_t)(e1 - e0);
        uint32_t ref_cnt = 0, mut_cnt = 0, err0 = 0, err1 = 0, err2 = 0, err3 = 0, fP = 0, fK = 0, fO = 0;
        uint32_t j0 = 0;
        // odd patches made at EARLIER targets (the list only grows at later loci, so it is fixed for this target)
        __syncwarp();
        const unsigned int n_odd = min(*(volatile unsigned int *)A.n_odd, A.odd_cap);
        unsigned long long new_bloom = 0;
        bool st = false;
        PlpEntry *s_ent = NULL; uint8_t *s_hf = NULL; int32_t *s_R = NULL; unsigned long long k_stage = 0; uint32_t n_stage = 0;
        if (STAGED && n <= CK_CAP) {
            st = true;
            s_ent = reinterpret_cast<PlpEntry *>(ck_smem); s_hf = reinterpret_cast<uint8_t *>(s_ent + CK_CAP);
            s_R = reinterpret_cast<int32_t *>(s_hf + ((CK_CAP + 15u) & ~15u));
            __syncwarp();
            for (uint32_t i = lane; i < n; i += 32) { reinterpret_cast<uint4 *>(s_ent)[i] = reinterpret_cast<const uint4 *>(ents)[i]; s_hf[i] = 0; }
            k_stage = k;
            const unsigned long long left = A.M > k + 1 ? A.M - k - 1 : 0ull;
            n_stage = (uint32_t)min((unsigned long long)(n + 64u), left);
            for (uint32_t i = lane; i < n_stage; i += 32) s_R[i] = A.R[k_stage + i];
            __syncwarp();
        }
        // (not staged:) the entries of the next batch and the 32 draws a batch can toss with are fetched ahead, so that a batch waits
        // for one round trip to memory (mates, handled flags) instead of three
        PlpEntry e_pref; e_pref.skip = 1; e_pref.bq = 0; e_pref.mate = -1; e_pref.base = 0; e_pref.ord = 0; e_pref.qpos = 0; e_pref.pad = 0;
        uint32_t pref_j0 = 0xffffffffu;
        while (j0 < n) {
            const uint32_t j = j0 + lane;
            const bool in = j < n;
            PlpEntry e; e.skip = 1; e.bq = 0; e.mate = -1; e.base = 0; e.ord = 0; e.qpos = 0; e.pad = 0;
            if (st) { if (in) e = s_ent[j]; }
            else {
                if (pref_j0 == j0) e = e_pref; else if (in) e = ents[j];
                const uint32_t jn = j0 + 32u + lane;
                e_pref.skip = 1; e_pref.bq = 0; e_pref.mate = -1; e_pref.base = 0; e_pref.ord = 0; e_pref.qpos = 0;
                if (jn < n) e_pref = ents[jn];
                pref_j0 = j0 + 32u;
            }
            const bool r_ok = k + 96ull <= A.M;
            uint32_t r_spec = 0u;
            if (r_ok) { const unsigned long long ri = k - k_stage + (unsigned long long)lane; r_spec = (st && ri < n_stage) ? (uint32_t)s_R[ri] : (uint32_t)A.R[k + lane]; }
            const uint8_t *hfr = st ? s_hf : hf;
            const bool handled = in ? hfr[j] != 0 : true;
            uint8_t mate_base = 0, mate_bq = 0; PlpEntry me_; me_.ord = 0; me_.qpos = 0; me_.skip = 0;
            bool mate_handled = false;
            if (in && e.mate >= 0) { me_ = st ? s_ent[e.mate] : ents[e.mate]; mate_base = me_.base; mate_bq = me_.bq; mate_handled = hfr[e.mate] != 0; }
            if (n_odd && in) {                        // bases an earlier odd patch rewrote (see OddPatch)
                if (odd_bloom & odd_bit(e.ord)) e.base = odd_view(A.odd, n_odd, e.ord, e.qpos, ht.tid, ht.pos, e.base);
                if (e.mate >= 0 && (odd_bloom & odd_bit(me_.ord))) mate_base = odd_view(A.odd, n_odd, me_.ord, me_.qpos, ht.tid, ht.pos, mate_base);
            }
            // does this entry toss?  needed to give every lane its draw index
            bool tosses = false;
            if (in && !e.skip && e.bq != 0 && !handled) {
                uint8_t R = e.base, M = 0; int rbq = e.bq, mbq = 0;
                if (e.mate >= 0 && !mate_handled) { M = mate_base; mbq = mate_bq; }
                if (M == 'N') mbq = 0;
                if (R == 'N') rbq = 0;
                uint8_t base = R; if (M && M != R && mbq > rbq) base = M;
                tosses = base != 'N';
            }
            const unsigned tossmask = __ballot_sync(0xffffffffu, tosses);
            const uint32_t my_idx = __popc(tossmask & ((1u << lane) - 1u));
            const unsigned long long my_k = k + my_idx;
            const uint32_t my_r = __shfl_sync(0xffffffffu, r_spec, my_idx);
            EntryOut o = entry_eval(A, e, mate_base, mate_bq, mate_handled, handled, my_k, ht.thresh, Fb, allele, r_ok, my_r);
            // a lane "breaks" the speculation of the lanes after it when it used more than its one draw, or
            // when it marks an entry of this batch as handled
            const bool marks_in_batch = in && o.mark_mate && e.mate >= 0 && (uint32_t)e.mate < j0 + 32;
            const bool breaks = !o.ok || o.draws > (tosses ? 1u : 0u) || marks_in_batch;
            const unsigned bmask = __ballot_sync(0xffffffffu, breaks);
            const uint32_t last = bmask ? (uint32_t)(__ffs(bmask) - 1) : 31u;         // commit lanes [0, last]
            if (__ballot_sync(0xffffffffu, !o.ok && (uint32_t)lane <= last)) { if (lane == 0) atomicOr(flags, (unsigned int)CHAIN_OVERRUN); return; }
            const bool commit = in && (uint32_t)lane <= last;
            if (commit) {
                uint8_t *hfw = st ? s_hf : hf;
                if (o.mark_self) hfw[j] = 1;
                if (o.mark_mate && e.mate >= 0) hfw[e.mate] = 1;
                for (int p = 0; p < o.npatch; p++) {
                    unsigned int slot = atomicAdd(A.n_patches, 1u);
                    const PlpEntry &pe = o.pmate[p] ? me_ : e;
                    if (slot < A.patch_cap) {
                        Patch pt; pt.ord = pe.ord; pt.qpos = pe.qpos; pt.base = o.pbase[p]; pt.pad = (uint32_t)h;
                        A.patches[slot] = pt;
                    }
                    if (o.pmate[p] && me_.skip) {     // the mate sits in a D/N here: the patch lands on a base of a later locus
                        unsigned int os = atomicAdd(A.n_odd, 1u);
                        if (os < A.odd_cap) { OddPatch q; q.ord = pe.ord; q.qpos = pe.qpos; q.base = o.pbase[p]; q.h = (uint32_t)h; q.tid = ht.tid; q.pos = ht.pos; A.odd[os] = q; }
                        else set_err(A.err, SSB_E_NOMEM, (unsigned long long)h);
                        new_bloom |= odd_bit(pe.ord);
                    }
                }
            }
            const uint32_t used = commit ? o.draws : 0u;
            uint32_t tot = used;
            for (int s = 16; s; s >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, s);
            k += tot;
            ref_cnt += __popc(__ballot_sync(0xffffffffu, commit && o.tally == 1));
            mut_cnt += __popc(__ballot_sync(0xffffffffu, commit && o.tally == 2));
            err0 += __popc(__ballot_sync(0xffffffffu, commit && o.tally == 3));
            err1 += __popc(__ballot_sync(0xffffffffu, commit && o.tally == 4));
            err2 += __popc(__ballot_sync(0xffffffffu, commit && o.tally == 5));
            err3 += __popc(__ballot_sync(0xffffffffu, commit && o.tally == 6));
            fP |= __ballot_sync(0xffffffffu, commit && o.filt == 1);
            fK |= __ballot_sync(0xffffffffu, commit && o.filt == 2);
            fO |= __ballot_sync(0xffffffffu, commit && o.filt == 3);
            __syncwarp();
            j0 += last + 1;
        }
        for (int sft = 16; sft; sft >>= 1) new_bloom |= __shfl_xor_sync(0xffffffffu, new_bloom, sft);
        odd_bloom |= new_bloom;
        __threadfence();
        if (lane == 0) {
            ssb_target_result &r = A.res[ht.target];
            r.ref_base = Fb; r.mutant_allele = allele;
            // the filter only moves UNDETECTED -> PASS (cases 1,3), -> MASKED (case 2, unless MASKED_OVL), -> MASKED_OVL (cases 4-6)
            r.filter = fO ? SSB_F_MASKED_OVL : fK ? SSB_F_MASKED : fP ? SSB_F_PASS : SSB_F_UNDETECTED;
            r.ref_cnt = (int32_t)ref_cnt; r.mut_cnt = (int32_t)mut_cnt;
            r.err_cnt[0] = (int32_t)err0; r.err_cnt[1] = (int32_t)err1; r.err_cnt[2] = (int32_t)err2; r.err_cnt[3] = (int32_t)err3;
            r.rng_offset = (int64_t)k_at;
        }
        g += 1;
    }
    if (cd.k_out != ~0ull) {
        // finish the chunk and compare with what phase 1/2 predicted
        if (!walk_loci<true>(A, g, cd.g1, k)) { if (lane == 0) atomicOr(flags, (unsigned int)CHAIN_OVERRUN); return; }
        if (cd.k_out != CHUNK_WALK_ONLY && k != cd.k_out && lane == 0) atomicOr(flags, (unsigned int)CHAIN_INCONSISTENT);
    }
    if (lane == 0) { if (c == n_chunks - 1) *draws_out = k; if (n_chunks == 1) *A.odd_bloom = odd_bloom; }
}
