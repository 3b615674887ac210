// spike_run.cuh -- one run of the spike path over one shard of the input: the order of its stages on the context's stream,
// and the few points where the host has to look at a number.  (Included at the end of spike.cu.)
//
// Stages, in issue order ("sync" = the host waits for a handful of scalars that a kernel wrote into mapped pinned memory --
// no copy engine is involved, so these waits do not queue behind the bulk transfers of a streamed run):
//
//   parse ........................................................ sync 1: lines, kept reads, first error
//   keep flags, sortedness, compaction
//   output order (radix sort by end), output offsets
//   mates, coverage runs ......................................... sync 2: runs, covered loci, fold, max span
//   per-locus start/end counts, max depth, local target bounds
//      [shards: all-gather summaries, max-reduce the target bounds]
//   target scan, hits, pileup sizes ............................... sync 3: hits, pileup entries
//   pileup gather, reference classes, expected draws .............. sync 4: means / variances -> window geometry (host)
//   EMIT, tallies of the non-target loci (exception list + generic)
//      [shards: all-gather expected draws -> window centre of this shard]
//   rand() stream, phase 1 (window maps), [shards: precompose]
//      [shards: receive the exact offset, look the exit offset up (sync), send it on]
//   compose, chunk boundaries, phase 3 (apply) .................... sync 5: flags (fallbacks: serial chain)
//      [shards: agree that nobody changed an offset after sending it; forward spiked bases of straddling reads]
//   patches; SEQ_ERROR records .................................... sync 6: record count; results back
//
// Everything runs on one stream: emit and the tallies beside the chain kernels slowed both down by more than the overlap
// gave (DESIGN.md section 7).
#include "exchange.cuh"
#include <chrono>
#include <string>

namespace {

struct RunScalars {                 // written by kernels of the run, mirrored to the host on demand
    unsigned long long n_lines, n_keep, exc_count, n_float;
    DevErr err;
    unsigned long long fold; unsigned int maxspan, maxdepth;
    unsigned int n_runs, pad0; unsigned long long n_cov;
    unsigned int H, pad1; unsigned long long E; long long last_hit_locus;
    unsigned int flags, n_odd, n_patches, n_fwd;
    unsigned long long odd_bloom, draws, pool_used, k_out, k_end;
    unsigned long long n_se, first_strad, halo_lines, miss[2];
    long long carry_t, carry_h;
    unsigned long long max_end;
    unsigned long long total_out, n_owned;
};

__global__ void copy_words_kernel(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst, unsigned int n)
{
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
    __threadfence_system();
}
// plain device-to-device copy of bytes by SM threads (keeps the copy engines free for the host link); 16-byte words where both
// sides allow it
__global__ void copy_bytes_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, size_t n)
{
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)src | (uintptr_t)dst) & 15) == 0) {
        const size_t nv = n >> 4;
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src); uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        for (size_t i = tid; i < nv; i += nt) d4[i] = s4[i];
        for (size_t i = (nv << 4) + tid; i < n; i += nt) dst[i] = src[i];
    } else if ((((uintptr_t)src ^ (uintptr_t)dst) & 15) == 0) {
        const size_t head = (16 - ((uintptr_t)dst & 15)) & 15, h = head < n ? head : n;
        for (size_t i = tid; i < h; i += nt) dst[i] = src[i];
        const size_t nv = (n - h) >> 4;
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src + h); uint4 *d4 = reinterpret_cast<uint4 *>(dst + h);
        for (size_t i = tid; i < nv; i += nt) d4[i] = s4[i];
        for (size_t i = h + (nv << 4) + tid; i < n; i += nt) dst[i] = src[i];
    } else {
        // different alignment: aligned 16-byte stores, the source words shifted into place from 4-byte loads
        const size_t head = (16 - ((uintptr_t)dst & 15)) & 15, h = head < n ? head : n;
        for (size_t i = tid; i < h; i += nt) dst[i] = src[i];
        const size_t nv = (n - h) >> 4;
        uint4 *d4 = reinterpret_cast<uint4 *>(dst + h);
        const uint8_t *sb = src + h;
        const uint32_t a = (uint32_t)((uintptr_t)sb & 3u);
        const uint32_t *sw = reinterpret_cast<const uint32_t *>(sb - a);
        for (size_t i = tid; i + 1 < nv; i += nt) {             // the last word may not read past the end of the source
            const uint32_t w0 = sw[4 * i], w1 = sw[4 * i + 1], w2 = sw[4 * i + 2], w3 = sw[4 * i + 3], w4 = sw[4 * i + 4];
            uint4 o; o.x = __funnelshift_r(w0, w1, a * 8); o.y = __funnelshift_r(w1, w2, a * 8); o.z = __funnelshift_r(w2, w3, a * 8); o.w = __funnelshift_r(w3, w4, a * 8);
            d4[i] = o;
        }
        const size_t done = nv ? h + ((nv - 1) << 4) : h;
        for (size_t i = done + tid; i < n; i += nt) dst[i] = src[i];
    }
}
__global__ void out_total_kernel(unsigned long long *__restrict__ out_off, const unsigned long long *__restrict__ olen, size_t K, unsigned long long *__restrict__ total)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) { const unsigned long long t = out_off[K - 1] + olen[K - 1]; *total = t; out_off[K] = t; }
}
// Output order = end order: (tid, end) keys packed into 32 bits when the contigs and the largest end of a kept read allow it
// (one contig of 59 Mb: 26 bits = four radix passes over 4-byte keys instead of five over 8-byte keys)
__global__ void pack_end_kernel(const unsigned long long *__restrict__ k_end, size_t K, int pos_bits, uint32_t *__restrict__ key32, uint32_t *__restrict__ iota)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o < K) { const unsigned long long e = k_end[o]; key32[o] = ((uint32_t)(e >> 32) << pos_bits) | (uint32_t)e; iota[o] = (uint32_t)o; }
}
__global__ void unpack_end_kernel(const uint32_t *__restrict__ key32, size_t K, int pos_bits, unsigned long long *__restrict__ s_end)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o < K) { const uint32_t u = key32[o]; s_end[o] = ((unsigned long long)(pos_bits >= 32 ? 0u : u >> pos_bits) << 32) | (pos_bits >= 32 ? u : (u & ((1u << pos_bits) - 1u))); }
}
__global__ void first_strad_kernel(const unsigned long long *__restrict__ k_end, const uint32_t *__restrict__ k_rec, const SamRec *__restrict__ recs, size_t K, Range rg,
                                   unsigned long long *__restrict__ first_strad)
{
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o < K && k_end[o] - 1 >= rg.hi) atomicMin(first_strad, (unsigned long long)recs[k_rec[o]].line_off);
}
__global__ void hit_totals_kernel(const uint32_t *__restrict__ hidx, const uint32_t *__restrict__ hitflag, size_t T, const HitTarget *__restrict__ hits,
                                  unsigned int *__restrict__ H, long long *__restrict__ last_locus)
{
    if (blockIdx.x || threadIdx.x) return;
    const unsigned int h = hidx[T - 1] + hitflag[T - 1];
    *H = h;
    *last_locus = h ? (long long)hits[h - 1].locus_index : -1;
}
__global__ void copy_u64_kernel(const unsigned long long *__restrict__ src, unsigned long long *__restrict__ dst) { if (!blockIdx.x && !threadIdx.x) *dst = *src; }
// targets consumed by this shard and the shards before it (shards processed one after the other): the first target whose locus
// lies beyond this shard's last covered locus, and the last ordinal used before it
__global__ void carry_kernel(const long long *__restrict__ vmax, size_t T, long long ord_end, long long carry_t, long long carry_h, long long *__restrict__ out_t, long long *__restrict__ out_h)
{
    if (blockIdx.x || threadIdx.x) return;
    size_t lo = (size_t)carry_t, hi = T;               // h_t is strictly increasing in t: first t >= carry_t with h_t >= ord_end
    while (lo < hi) { const size_t mid = (lo + hi) >> 1; if (vmax[mid] + (long long)mid < ord_end) lo = mid + 1; else hi = mid; }
    *out_t = (long long)lo;
    *out_h = lo > (size_t)carry_t ? vmax[lo - 1] + (long long)(lo - 1) : carry_h;
}
__global__ void chunks_init_kernel(ChunkDesc *__restrict__ chunks, int P, int64_t Lc, int64_t n_walk)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= P) return;
    ChunkDesc c; c.g0 = (int64_t)f * Lc; c.g1 = (int64_t)(f + 1) * Lc < n_walk ? (int64_t)(f + 1) * Lc : n_walk; c.k_in = 0; c.k_out = ~0ull;
    chunks[f] = c;
}
__global__ void serial_chunk_kernel(ChunkDesc *__restrict__ c, int64_t n_walk, unsigned long long k_in, unsigned long long k_out)
{
    if (blockIdx.x || threadIdx.x) return;
    c->g0 = 0; c->g1 = n_walk; c->k_in = k_in; c->k_out = k_out;
}
// odd patches handed over by the previous shard: the read is named by its line index from the end of that shard's body
struct OddFwd { uint32_t from_end, qpos, base; int32_t tid, pos; uint32_t pad; };
__global__ void odd_import_kernel(const OddFwd *__restrict__ in, unsigned int n, unsigned long long halo_lines, const uint32_t *__restrict__ keep, const uint32_t *__restrict__ kord,
                                  OddPatch *__restrict__ odd, unsigned int *__restrict__ n_odd, unsigned long long *__restrict__ bloom, DevErr *err)
{
    if (blockIdx.x || threadIdx.x) return;
    unsigned long long b = 0; unsigned int m = 0;
    for (unsigned int i = 0; i < n; i++) {
        const OddFwd f = in[i];
        if (f.from_end == 0 || f.from_end > halo_lines || !keep[halo_lines - f.from_end]) { set_err(err, SSB_E_SHARD, i); continue; }
        OddPatch q; q.ord = kord[halo_lines - f.from_end]; q.qpos = f.qpos; q.base = f.base; q.h = 0; q.tid = f.tid; q.pos = f.pos;
        odd[m++] = q; b |= odd_bit(q.ord);
    }
    *n_odd = m; *bloom = b;
}
__global__ void odd_export_kernel(const OddPatch *__restrict__ odd, const unsigned int *__restrict__ n_odd, unsigned int odd_cap, const unsigned long long *__restrict__ k_end,
                                  const uint32_t *__restrict__ k_rec, unsigned long long n_lines, Range rg, OddFwd *__restrict__ out, unsigned int *__restrict__ n_out, unsigned int cap)
{
    if (blockIdx.x || threadIdx.x) return;
    const unsigned int n = min(*n_odd, odd_cap); unsigned int m = 0;
    for (unsigned int i = 0; i < n; i++) {
        const OddPatch q = odd[i];
        if (owns_last(k_end[q.ord], rg)) continue;                 // the read ends inside this shard: nobody later sees it
        if (m < cap) { OddFwd f; f.from_end = (uint32_t)(n_lines - k_rec[q.ord]); f.qpos = q.qpos; f.base = q.base; f.tid = q.tid; f.pos = q.pos; f.pad = 0; out[m] = f; }
        m++;
    }
    *n_out = m;
}
// number of alignment lines that start inside the first halo_bytes of the body
__global__ void halo_lines_kernel(const SamRec *__restrict__ recs, size_t N, unsigned long long halo_bytes, unsigned long long *__restrict__ out)
{
    if (blockIdx.x || threadIdx.x) return;
    size_t lo = 0, hi = N;
    while (lo < hi) { const size_t mid = (lo + hi) >> 1; if (recs[mid].line_off < halo_bytes) lo = mid + 1; else hi = mid; }
    *out = lo;
}

// ------------------------------------------------------------------------------------------
// device arena: one stream-ordered allocation per array, all released at the end of the run
// ------------------------------------------------------------------------------------------
struct Arena {
    cudaStream_t s; std::vector<void *> ptrs; bool failed = false;
    explicit Arena(cudaStream_t s_) : s(s_) {}
    template <typename T> T *get(size_t n)
    {
        void *p = NULL;
        if (cudaMallocAsync(&p, (n ? n : 1) * sizeof(T), s) != cudaSuccess) { failed = true; cudaGetLastError(); return NULL; }
        ptrs.push_back(p);
        return (T *)p;
    }
    ~Arena() { for (void *p : ptrs) cudaFreeAsync(p, s); }
};

inline int grid_for(size_t n, int block) { size_t g = (n + block - 1) / block; return (int)(g ? g : 1); }

// what one shard hands to the next when the shards of an input are processed one after the other on one device
struct SeqState {
    unsigned long long k = 0;                 // rand() calls consumed so far
    long long carry_t = 0, carry_h = -1;      // targets consumed so far, last covered ordinal one of them used
    long long ord_base = 0;                   // covered loci so far
    std::vector<FwdPatch> fwd;                // spiked bases of reads the next shard writes
    std::vector<OddFwd> odd;                  // odd patches on reads that reach into the next shard
    unsigned long long first_strad = ~0ull;   // body offset of the first line the next shard has to see again (~0: none)
    unsigned int maxspan = 0;
};

struct ShardPlan {
    int index = 0, count = 1;
    Range rg{0ull, ~0ull};
    size_t halo_bytes = 0;
    ssb_exchange *xc = NULL;                  // cooperating shards (count > 1, all at work at the same time)
    SeqState *seq = NULL;                     // or: shards one after the other (in: state after the previous shard, out: after this one)
    bool last = true;                         // no shard follows (sequential mode; cooperating shards know from index / count)
};

} // namespace

// ---------------------------------------------------------------------------------------------
struct ssb_spike {
    ssb_ctx *ctx;
    int n_contigs;
    int p1_resident;                          // blocks of phase1_kernel the device holds at once
    char *d_names; uint32_t *d_name_off;
    uint8_t **d_seq_ptrs; int64_t *d_lens;
    std::vector<uint8_t *> d_seqs;
    RngTables *d_rng_tab;
    ssb_seq_error *d_se; size_t n_se;          // SEQ_ERROR records of the last run (device resident until asked for)
    // run plumbing
    cudaEvent_t ev_pub, ev_t[16];
    RunScalars *d_sc, *h_sc;                   // device scalars and their mapped pinned mirror
    uint8_t *h_map; size_t h_map_bytes;        // mapped pinned scratch: descriptors kernels read, small arrays kernels write
    DevTarget *d_tg; std::vector<DevTarget> tg_host;           // targets of the last run (uploaded again only when they change)
    std::vector<std::string> names;                            // @SQ names (host copy: the streamed run cuts the body by coordinate)
    std::vector<std::pair<ssb_seq_error *, size_t>> se_chunks;  // SEQ_ERROR records of a streamed run: one device array per piece, fetched on demand
    bool se_chunked;
    uint8_t *h_res; size_t h_res_bytes;                        // mapped pinned buffer the per-target results are written into
    // buffers of the streamed host run (kept between calls: allocating and freeing gigabytes per call costs more than the run)
    uint8_t *st_staging[3], *st_work[2], *st_obuf[2]; size_t st_slot; cudaStream_t st_out; std::vector<cudaEvent_t> st_ev;
};

namespace {
void spike_free(ssb_spike *sp)
{
    for (uint8_t *d : sp->d_seqs) if (d) cudaFree(d);
    if (sp->d_se) cudaFree(sp->d_se);
    if (sp->d_names) cudaFree(sp->d_names);
    if (sp->d_name_off) cudaFree(sp->d_name_off);
    if (sp->d_seq_ptrs) cudaFree(sp->d_seq_ptrs);
    if (sp->d_lens) cudaFree(sp->d_lens);
    if (sp->d_rng_tab) cudaFree(sp->d_rng_tab);
    if (sp->d_sc) cudaFree(sp->d_sc);
    if (sp->d_tg) cudaFree(sp->d_tg);
    if (sp->h_sc) cudaFreeHost(sp->h_sc);
    if (sp->h_map) cudaFreeHost(sp->h_map);
    if (sp->h_res) cudaFreeHost(sp->h_res);
    for (int i = 0; i < 3; i++) if (sp->st_staging[i]) cudaFree(sp->st_staging[i]);
    for (int i = 0; i < 2; i++) { if (sp->st_work[i]) cudaFree(sp->st_work[i]); if (sp->st_obuf[i]) cudaFree(sp->st_obuf[i]); }
    for (cudaEvent_t e : sp->st_ev) if (e) cudaEventDestroy(e);
    if (sp->st_out) cudaStreamDestroy(sp->st_out);
    for (auto &c : sp->se_chunks) if (c.first) cudaFree(c.first);
    if (sp->ev_pub) cudaEventDestroy(sp->ev_pub);
    for (int i = 0; i < 16; i++) if (sp->ev_t[i]) cudaEventDestroy(sp->ev_t[i]);
    delete sp;
}
} // namespace

extern "C" int ssb_spike_create(ssb_ctx *ctx, const ssb_contig *contigs, int n_contigs, ssb_spike **out)
{
    if (!ctx || !out || n_contigs < 0 || (n_contigs && !contigs)) return SSB_E_ARG;
    *out = NULL;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    ssb_spike *sp = new ssb_spike();
    sp->ctx = ctx; sp->n_contigs = n_contigs; sp->d_se = NULL; sp->n_se = 0; sp->se_chunked = false; sp->h_res = NULL; sp->h_res_bytes = 0;
    for (int i = 0; i < 3; i++) sp->st_staging[i] = NULL;
    for (int i = 0; i < 2; i++) { sp->st_work[i] = NULL; sp->st_obuf[i] = NULL; }
    sp->st_slot = 0; sp->st_out = NULL;
    for (int i = 0; i < n_contigs; i++) sp->names.push_back(contigs[i].name ? contigs[i].name : "");
    sp->d_names = NULL; sp->d_name_off = NULL; sp->d_seq_ptrs = NULL; sp->d_lens = NULL; sp->d_rng_tab = NULL;
    sp->d_sc = sp->h_sc = NULL; sp->h_map = NULL; sp->h_map_bytes = 0; sp->d_tg = NULL;
    sp->ev_pub = NULL;
    for (int i = 0; i < 16; i++) sp->ev_t[i] = NULL;
    // every exit below releases what has been allocated so far
#define SPK_CREATE(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(ctx->err, sizeof ctx->err, "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); spike_free(sp); return SSB_E_CUDA; } } while (0)
    std::vector<char> names; std::vector<uint32_t> off; std::vector<int64_t> lens; std::vector<uint8_t *> ptrs;
    off.push_back(0);
    for (int i = 0; i < n_contigs; i++) {
        const char *nm = contigs[i].name ? contigs[i].name : "";
        names.insert(names.end(), nm, nm + strlen(nm));
        off.push_back((uint32_t)names.size());
        uint8_t *d = NULL;
        if (contigs[i].seq && contigs[i].len > 0) {
            SPK_CREATE(cudaMalloc(&d, (size_t)contigs[i].len + 64));
            sp->d_seqs.push_back(d);
            SPK_CREATE(cudaMemcpy(d, contigs[i].seq, (size_t)contigs[i].len, cudaMemcpyHostToDevice));
        } else sp->d_seqs.push_back(d);
        ptrs.push_back(d); lens.push_back(d ? contigs[i].len : 0);
    }
    { int occ = 1; SPK_CREATE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, phase1_kernel, P1_THREADS, P1_SMEM)); sp->p1_resident = occ * ctx->sm_count; }
    SPK_CREATE(cudaMalloc(&sp->d_names, names.size() + 1));
    SPK_CREATE(cudaMalloc(&sp->d_name_off, off.size() * sizeof(uint32_t)));
    SPK_CREATE(cudaMalloc(&sp->d_seq_ptrs, (ptrs.size() + 1) * sizeof(uint8_t *)));
    SPK_CREATE(cudaMalloc(&sp->d_lens, (lens.size() + 1) * sizeof(int64_t)));
    if (!names.empty()) SPK_CREATE(cudaMemcpy(sp->d_names, names.data(), names.size(), cudaMemcpyHostToDevice));
    SPK_CREATE(cudaMemcpy(sp->d_name_off, off.data(), off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (n_contigs) {
        SPK_CREATE(cudaMemcpy(sp->d_seq_ptrs, ptrs.data(), ptrs.size() * sizeof(uint8_t *), cudaMemcpyHostToDevice));
        SPK_CREATE(cudaMemcpy(sp->d_lens, lens.data(), lens.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    }
    // seed-independent skip-ahead table: x^(t*RNG_SEG) mod P, t < RNG_TPB (host integer arithmetic, a few ms)
    RngTables *tab = new RngTables();
    uint32_t step[GLIBC_DEG], cur[GLIBC_DEG], tmp[GLIBC_DEG];
    glibc_poly_xpow(RNG_SEG, step);
    glibc_poly_xpow(0, cur);
    for (int t = 0; t < RNG_TPB; t++) {
        memcpy(tab->seg[t], cur, sizeof cur);
        glibc_poly_mulmod(cur, step, tmp); memcpy(cur, tmp, sizeof cur);
    }
    cudaError_t e1 = cudaMalloc(&sp->d_rng_tab, sizeof(RngTables));
    if (e1 == cudaSuccess) e1 = cudaMemcpy(sp->d_rng_tab, tab, sizeof(RngTables), cudaMemcpyHostToDevice);
    delete tab;
    SPK_CREATE(e1);
    // events, mapped scalars
    SPK_CREATE(cudaEventCreateWithFlags(&sp->ev_pub, cudaEventDisableTiming));
    for (int i = 0; i < 16; i++) SPK_CREATE(cudaEventCreate(&sp->ev_t[i]));
    SPK_CREATE(cudaMalloc(&sp->d_sc, sizeof(RunScalars)));
    SPK_CREATE(cudaHostAlloc((void **)&sp->h_sc, sizeof(RunScalars), cudaHostAllocMapped));
    sp->h_map_bytes = (size_t)32 << 20;
    SPK_CREATE(cudaHostAlloc((void **)&sp->h_map, sp->h_map_bytes, cudaHostAllocMapped));
#undef SPK_CREATE
    *out = sp;
    return SSB_OK;
}

extern "C" void ssb_spike_destroy(ssb_spike *sp)
{
    if (!sp) return;
    cudaSetDevice(sp->ctx->device);
    cudaStreamSynchronize(sp->ctx->stream);
    spike_free(sp);
}

#define SPK_CHECK_ARENA(ar) do { if ((ar).failed) { snprintf(ctx->err, sizeof ctx->err, "spike: device allocation failed"); return SSB_E_NOMEM; } } while (0)

namespace {

// CUB wrappers: temp storage from the arena
template <typename T> int scan_sum(Arena &ar, ssb_ctx *ctx, const T *in, T *out, size_t n)
{
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(NULL, bytes, in, out, n, ar.s);
    void *tmp = ar.get<uint8_t>(bytes); SPK_CHECK_ARENA(ar);
    SSB_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, bytes, in, out, n, ar.s));
    ctx->launches += 2;
    return SSB_OK;
}
template <typename T> int scan_sum_incl(Arena &ar, ssb_ctx *ctx, const T *in, T *out, size_t n)
{
    size_t bytes = 0;
    cub::DeviceScan::InclusiveSum(NULL, bytes, in, out, n, ar.s);
    void *tmp = ar.get<uint8_t>(bytes); SPK_CHECK_ARENA(ar);
    SSB_CUDA(ctx, cub::DeviceScan::InclusiveSum(tmp, bytes, in, out, n, ar.s));
    ctx->launches += 2;
    return SSB_OK;
}
template <typename T> int scan_max_excl(Arena &ar, ssb_ctx *ctx, const T *in, T *out, size_t n, T init)
{
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveScan(NULL, bytes, in, out, MaxOp(), init, n, ar.s);
    void *tmp = ar.get<uint8_t>(bytes); SPK_CHECK_ARENA(ar);
    SSB_CUDA(ctx, cub::DeviceScan::ExclusiveScan(tmp, bytes, in, out, MaxOp(), init, n, ar.s));
    ctx->launches += 2;
    return SSB_OK;
}
template <typename T> int scan_max_incl(Arena &ar, ssb_ctx *ctx, const T *in, T *out, size_t n)
{
    size_t bytes = 0;
    cub::DeviceScan::InclusiveScan(NULL, bytes, in, out, MaxOp(), n, ar.s);
    void *tmp = ar.get<uint8_t>(bytes); SPK_CHECK_ARENA(ar);
    SSB_CUDA(ctx, cub::DeviceScan::InclusiveScan(tmp, bytes, in, out, MaxOp(), n, ar.s));
    ctx->launches += 2;
    return SSB_OK;
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) { float ms = 0; if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); return 0; } return ms; }
double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct ShardSummary { unsigned long long n_cov, body_bytes, halo_bytes, first_strad; unsigned int maxspan, pad; };
struct ShardExpect { double mean, var; unsigned long long H, pad; };
struct ShardVerdict { unsigned long long k_out; unsigned int dirty, n_odd_fwd; };
struct HandOff { unsigned long long k; unsigned int n_odd, pad; };

// The whole run of one shard.
int run_shard(ssb_spike *sp, const ShardPlan &pl, const uint8_t *d_sam, size_t n, uint8_t *d_out, size_t out_cap,
              const ssb_target *targets, size_t T, unsigned seed, ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes)
{
    ssb_ctx *ctx = sp->ctx;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    memset(stats, 0, sizeof *stats);
    *out_bytes = 0;
    const char *dbg_env = getenv("SSB_CHAIN_DEBUG");
    const bool dbg_t = dbg_env != NULL;
    const double t_host0 = now_ms();
    auto dbg_mark = [&](const char *what) { if (dbg_t) fprintf(stderr, "[spike %d/%d] %-14s %.3f ms (host)\n", pl.index, pl.count, what, now_ms() - t_host0); };
    const Range rg = pl.rg;
    ssb_exchange *xc = pl.count > 1 ? pl.xc : NULL;
    SeqState *seq = pl.seq;
    const bool is_last = seq ? pl.last : pl.index == pl.count - 1;
    if (pl.count > 1 && !xc && !seq) return SSB_E_ARG;

    if (sp->d_se) { cudaFreeAsync(sp->d_se, s); sp->d_se = NULL; }
    sp->n_se = 0;
    if (!pl.seq) { for (auto &c : sp->se_chunks) if (c.first) cudaFreeAsync(c.first, s); sp->se_chunks.clear(); sp->se_chunked = false; }
    stats->in_bytes = (int64_t)n;
    Arena ar(s);
    // declared after the arena, so destroyed first: nothing may still run when the arena gives its memory back
    struct Drain { cudaStream_t s; ~Drain() { cudaStreamSynchronize(s); } } drain{s};

    RunScalars *dsc = sp->d_sc; volatile RunScalars *hsc = sp->h_sc;
    RunScalars *hsc_dev = NULL; uint8_t *hmap_dev = NULL;
    SSB_CUDA(ctx, cudaHostGetDevicePointer((void **)&hsc_dev, sp->h_sc, 0));
    SSB_CUDA(ctx, cudaHostGetDevicePointer((void **)&hmap_dev, sp->h_map, 0));
    auto publish = [&]() -> int {               // scalars -> host, and wait for them
        SSB_LAUNCH(ctx, copy_words_kernel, 1, 64, 0, s, (const uint32_t *)dsc, (uint32_t *)hsc_dev, (unsigned int)(sizeof(RunScalars) / 4));
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_pub, s));
        SSB_CUDA(ctx, cudaEventSynchronize(sp->ev_pub));
        return SSB_OK;
    };
    auto fail_dev = [&](const char *stage) -> int {
        const int code = hsc->err.code; const unsigned long long where = hsc->err.where;
        snprintf(ctx->err, sizeof ctx->err, "spike/%s: %s (at %llu)", stage, ssb_strerror(code), where);
        return code;
    };
    // mapped pinned scratch, handed out front to back
    size_t map_used = 0;
    auto map_get = [&](size_t bytes, uint8_t **h, uint8_t **d) -> int {
        bytes = (bytes + 255) & ~(size_t)255;
        if (map_used + bytes > sp->h_map_bytes) {
            // grow: nothing handed out earlier in this run may still be in use -> only allowed before the first hand-out
            if (map_used) { snprintf(ctx->err, sizeof ctx->err, "spike: mapped scratch exhausted"); return SSB_E_NOMEM; }
            SSB_CUDA(ctx, cudaStreamSynchronize(s));
            cudaFreeHost(sp->h_map); sp->h_map = NULL; sp->h_map_bytes = 0;
            SSB_CUDA(ctx, cudaHostAlloc((void **)&sp->h_map, bytes + ((size_t)4 << 20), cudaHostAllocMapped));
            sp->h_map_bytes = bytes + ((size_t)4 << 20);
            SSB_CUDA(ctx, cudaHostGetDevicePointer((void **)&hmap_dev, sp->h_map, 0));
        }
        *h = sp->h_map + map_used; *d = hmap_dev + map_used; map_used += bytes;
        return SSB_OK;
    };

    SSB_CUDA(ctx, cudaMemsetAsync(dsc, 0, sizeof(RunScalars), s));
    SSB_CUDA(ctx, cudaMemsetAsync(&dsc->first_strad, 0xff, sizeof(unsigned long long), s));
    const unsigned int odd_cap = 1u << 16;
    OddPatch *d_odd = ar.get<OddPatch>(odd_cap); SPK_CHECK_ARENA(ar);
    unsigned int *d_nodd = &dsc->n_odd; unsigned long long *d_bloom = &dsc->odd_bloom;
    DevErr *d_err = &dsc->err;
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[0], s));

    // ---------------------------------------------------------------- parse
    size_t N = 0, K = 0;
    SamRec *recs = NULL; uint32_t *keep = NULL; unsigned long long *pkey = NULL;      // per line: the record, kept?, sortedness key (written by the tokeniser)
    unsigned long long *exc_list = NULL, exc_cap = 0, n_list = 0;
    const bool no_list = getenv("SSB_NO_EXC_LIST") != NULL;
    if (n) {
        const size_t n_tiles = (n + samparse::TILE - 1) / samparse::TILE;
        unsigned long long *tile_state = ar.get<unsigned long long>(n_tiles);
        unsigned int *ticket = ar.get<unsigned int>(1);
        size_t rec_cap = n / 96 + 4096;
        exc_cap = n / 96 + 65536;
        exc_list = ar.get<unsigned long long>(exc_cap); SPK_CHECK_ARENA(ar);
        SSB_CUDA(ctx, cudaFuncSetAttribute(samparse::parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, samparse::SMEM_BYTES));
        for (int attempt = 0; attempt < 2; attempt++) {
            recs = ar.get<SamRec>(rec_cap); keep = ar.get<uint32_t>(rec_cap); pkey = ar.get<unsigned long long>(rec_cap); SPK_CHECK_ARENA(ar);
            SSB_CUDA(ctx, cudaMemsetAsync(tile_state, 0, n_tiles * sizeof(unsigned long long), s));
            SSB_CUDA(ctx, cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s));
            if (attempt) { SSB_CUDA(ctx, cudaMemsetAsync(dsc, 0, sizeof(RunScalars), s)); SSB_CUDA(ctx, cudaMemsetAsync(&dsc->first_strad, 0xff, sizeof(unsigned long long), s)); }
            samparse::ContigNames names{sp->d_names, sp->d_name_off, sp->n_contigs, (const uint8_t *const *)sp->d_seq_ptrs, sp->d_lens,
                                        no_list ? NULL : exc_list, &dsc->exc_count, exc_cap, rg.lo, &dsc->n_keep, &dsc->n_float, &dsc->max_end, keep, pkey};
            int occ = 1;
            SSB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, samparse::parse_kernel, samparse::THREADS, samparse::SMEM_BYTES));
            if (occ < 1) occ = 1;
            int grid = (int)(n_tiles < (size_t)ctx->sm_count * occ ? n_tiles : (size_t)ctx->sm_count * occ);     // persistent: exactly the resident blocks
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_PARSE, samparse::parse_kernel, grid, samparse::THREADS, samparse::SMEM_BYTES, s,
                         d_sam, n, names, recs, rec_cap, tile_state, ticket, &dsc->n_lines, reinterpret_cast<SpikeErr *>(d_err));
            int rc; if ((rc = publish())) return rc;                                  // sync 1
            N = (size_t)hsc->n_lines; K = (size_t)hsc->n_keep; n_list = hsc->exc_count;
            if (hsc->err.code == SSB_E_NOMEM && attempt == 0) { rec_cap = N + 16; continue; }
            if (hsc->err.code) { snprintf(ctx->err, sizeof ctx->err, "spike/parse: %s (SAM body offset %llu)", ssb_strerror(hsc->err.code), (unsigned long long)hsc->err.where); return hsc->err.code; }
            break;
        }
    }
    stats->n_lines = (int64_t)N;
    stats->n_kept = (int64_t)K;
    if (N && hsc->n_float)       // float-typed optional fields: judged out of line (errors surface at the next look at the error word)
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, samparse::aux_float_kernel, grid_for(N, 128), 128, 0, s, d_sam, n, recs, N, reinterpret_cast<SpikeErr *>(d_err));
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[1], s));
    dbg_mark("parsed");

    // ---------------------------------------------------------------- keep / sortedness / compaction
    uint32_t *kord = NULL;
    uint32_t *k_rec = NULL, *nxt = NULL, *prv = NULL; EmitDesc *k_desc = NULL; uint8_t *cplx = NULL, *k_bits = NULL;
    unsigned long long *k_start = NULL, *k_end = NULL, *k_hash = NULL; uint32_t *k_hash32 = NULL;
    unsigned long long *d_halo_lines = &dsc->halo_lines;
    if (N) {
        kord = ar.get<uint32_t>(N);
        unsigned long long *pmax = ar.get<unsigned long long>(N);
        k_rec = ar.get<uint32_t>(K); k_desc = ar.get<EmitDesc>(K); nxt = ar.get<uint32_t>(K);
        k_start = ar.get<unsigned long long>(K); k_end = ar.get<unsigned long long>(K); k_hash = ar.get<unsigned long long>(K); k_hash32 = ar.get<uint32_t>(K); k_bits = ar.get<uint8_t>(K);
        SPK_CHECK_ARENA(ar);
        int rc;
        if ((rc = scan_sum(ar, ctx, keep, kord, N))) return rc;
        if ((rc = scan_max_excl(ar, ctx, pkey, pmax, N, 0ull))) return rc;
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, compact_kernel, grid_for(N, 256), 256, 0, s, recs, N, keep, kord, pkey, pmax, k_rec, k_start, k_end, k_desc,
                     k_hash, k_hash32, k_bits, &dsc->fold, &dsc->maxspan, d_err, rg, (unsigned long long)pl.halo_bytes);
        if (pl.halo_bytes) SSB_LAUNCH(ctx, halo_lines_kernel, 1, 32, 0, s, recs, N, (unsigned long long)pl.halo_bytes, d_halo_lines);
        if (K && (pl.count > 1 || seq)) SSB_LAUNCH(ctx, first_strad_kernel, grid_for(K, 256), 256, 0, s, k_end, k_rec, recs, K, rg, &dsc->first_strad);
    }
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[2], s));

    // ---------------------------------------------------------------- output order, output offsets
    uint32_t *perm = NULL; unsigned long long *s_end = NULL, *out_off = NULL, *ord_off = NULL;
    EmitDesc *d_edesc = NULL;
    if (K) {
        int rc;
        uint32_t *iota = ar.get<uint32_t>(K); perm = ar.get<uint32_t>(K); s_end = ar.get<unsigned long long>(K);
        unsigned long long *olen = ar.get<unsigned long long>(K); out_off = ar.get<unsigned long long>(K + 1); ord_off = ar.get<unsigned long long>(K);
        d_edesc = ar.get<EmitDesc>(K);
        SPK_CHECK_ARENA(ar);
        int tid_bits = 0; while ((1ll << tid_bits) < (long long)sp->n_contigs && tid_bits < 31) tid_bits++;
        int pos_bits = 1; while (pos_bits < 32 && (1ull << pos_bits) <= hsc->max_end) pos_bits++;
        size_t bytes = 0;
        if (pos_bits + tid_bits <= 32 && !getenv("SSB_SORT64")) {
            uint32_t *key32 = ar.get<uint32_t>(K), *skey32 = ar.get<uint32_t>(K);
            cub::DeviceRadixSort::SortPairs(NULL, bytes, key32, skey32, iota, perm, K, 0, pos_bits + tid_bits, s);
            void *tmp = ar.get<uint8_t>(bytes); SPK_CHECK_ARENA(ar);
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, pack_end_kernel, grid_for(K, 256), 256, 0, s, k_end, K, pos_bits, key32, iota);
            SSB_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, bytes, key32, skey32, iota, perm, K, 0, pos_bits + tid_bits, s));   // stable: ties keep input order
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, unpack_end_kernel, grid_for(K, 256), 256, 0, s, skey32, K, pos_bits, s_end);
        } else {
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, iota_kernel, grid_for(K, 256), 256, 0, s, iota, K);
            cub::DeviceRadixSort::SortPairs(NULL, bytes, k_end, s_end, iota, perm, K, 0, 32 + tid_bits + 1, s);
            void *tmp = ar.get<uint8_t>(bytes); SPK_CHECK_ARENA(ar);
            SSB_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, bytes, k_end, s_end, iota, perm, K, 0, 32 + tid_bits + 1, s));   // stable: ties keep input order
        }
        ctx->launches += 8;
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, outlen_kernel, grid_for(K, 256), 256, 0, s, perm, s_end, k_desc, K, rg, olen, d_edesc, &dsc->n_owned);
        if ((rc = scan_sum(ar, ctx, olen, out_off, K))) return rc;
        SSB_LAUNCH(ctx, out_total_kernel, 1, 32, 0, s, out_off, olen, K, &dsc->total_out);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, ordoff_kernel, grid_for(K, 256), 256, 0, s, perm, out_off, K, ord_off);
        if (out_cap < n + 1) {                 // the output may not fit: look before writing
            if ((rc = publish())) return rc;
            if (hsc->total_out > out_cap) { snprintf(ctx->err, sizeof ctx->err, "spike: output needs %llu bytes, capacity %zu", (unsigned long long)hsc->total_out, out_cap); return SSB_E_ARG; }
        }
    }

    // ---------------------------------------------------------------- M: mates, coverage runs
    size_t R = 0; int64_t n_cov = 0;
    CovRun *runs = NULL; uint8_t *cls = NULL; uint32_t *cum_s = NULL, *cum_e = NULL;
    unsigned long long *pm = NULL, *ce = NULL, *cbase = NULL, *newcov = NULL; uint32_t *rflag = NULL, *rid = NULL;
    if (K) {
        int rc;
        prv = ar.get<uint32_t>(K); cplx = ar.get<uint8_t>(K);
        pm = ar.get<unsigned long long>(K); ce = ar.get<unsigned long long>(K); cbase = ar.get<unsigned long long>(K); newcov = ar.get<unsigned long long>(K);
        rflag = ar.get<uint32_t>(K); rid = ar.get<uint32_t>(K);
        SPK_CHECK_ARENA(ar);
        SSB_CUDA(ctx, cudaMemsetAsync(prv, 0xff, K * sizeof(uint32_t), s));
        SSB_CUDA(ctx, cudaMemsetAsync(cplx, 0, K, s));
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, mates_kernel, grid_for(K, MATES_TPB), MATES_TPB, 0, s, d_sam, recs, k_rec, k_start, k_end, k_hash32, K, nxt, prv, cplx);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, clipend_kernel, grid_for(K, 256), 256, 0, s, k_end, K, rg, ce);
        if ((rc = scan_max_excl(ar, ctx, ce, pm, K, 0ull))) return rc;
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, newcov_kernel, grid_for(K, 256), 256, 0, s, k_start, ce, pm, K, rg, rflag, newcov);
        if ((rc = scan_sum_incl(ar, ctx, rflag, rid, K))) return rc;
        if ((rc = scan_sum(ar, ctx, newcov, cbase, K))) return rc;
        SSB_LAUNCH(ctx, cover_totals_kernel, 1, 32, 0, s, rid, cbase, newcov, K, &dsc->n_runs, &dsc->n_cov);
    }
    { int rc; if ((rc = publish())) return rc; }                                          // sync 2
    if (hsc->err.code) return fail_dev("sorted");
    R = hsc->n_runs; n_cov = (int64_t)hsc->n_cov;
    const unsigned int h_maxspan = hsc->maxspan;
    const unsigned long long h_first_strad = hsc->first_strad, h_halo_lines = hsc->halo_lines;
    stats->totalFoldCoverage = (int64_t)hsc->fold;
    stats->n_runs = (int64_t)R;
    stats->numberOfLociCovered = n_cov;
    if (K) {
        runs = ar.get<CovRun>(R); cum_s = ar.get<uint32_t>((size_t)n_cov + 1); cum_e = ar.get<uint32_t>((size_t)n_cov + 1); SPK_CHECK_ARENA(ar);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, runs_kernel, grid_for(K, 256), 256, 0, s, k_start, ce, pm, rflag, rid, cbase, K, rg, runs);
        SSB_CUDA(ctx, cudaMemsetAsync(cum_e, 0, ((size_t)n_cov + 1) * sizeof(uint32_t), s));       // loci before the first read end
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, cum_fill_kernel, grid_for(K, 256), 256, 0, s, k_start, K, runs, R, n_cov, cum_s);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, cum_fill_kernel, grid_for(K, 256), 256, 0, s, s_end, K, runs, R, n_cov, cum_e);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, maxdepth_kernel, ctx->sm_count * 8, 256, 0, s, cum_s, cum_e, n_cov, &dsc->maxdepth);
    }
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[3], s));
    dbg_mark("covered");

    // ---------------------------------------------------------------- shards: who owns how many loci
    long long ord_base = 0, total_cov = n_cov;
    double t_xc = 0;
    std::vector<ShardSummary> summ;
    if (xc) {
        int rc;
        ShardSummary me; me.n_cov = (unsigned long long)n_cov; me.body_bytes = n; me.halo_bytes = pl.halo_bytes; me.first_strad = h_first_strad; me.maxspan = h_maxspan; me.pad = 0;
        summ.resize((size_t)xc->n);
        const double t0 = now_ms();
        if ((rc = xc->allgather(&me, summ.data(), sizeof me))) return rc;
        t_xc += now_ms() - t0;
        total_cov = 0;
        for (int g = 0; g < xc->n; g++) { if (g < pl.index) ord_base += (long long)summ[g].n_cov; total_cov += (long long)summ[g].n_cov; }
        // every read that reaches into the next shard must be among the lines repeated in front of it
        for (int g = 0; g + 1 < xc->n; g++)
            if (summ[g].first_strad != ~0ull && summ[g].first_strad + summ[g + 1].halo_bytes < summ[g].body_bytes) {
                snprintf(ctx->err, sizeof ctx->err, "spike: shard %d has reads reaching into shard %d that start before its halo (largest read span %u)", g, g + 1, summ[g].maxspan);
                return SSB_E_SHARD;
            }
    } else if (seq) { ord_base = seq->ord_base; total_cov = is_last ? ord_base + n_cov : -1; }
    stats->locus_base = ord_base;

    // ---------------------------------------------------------------- targets
    size_t H = 0; unsigned long long E = 0; long long last_hit_locus = -1;
    HitTarget *hits = NULL; ssb_target_result *d_res = NULL; unsigned long long *eoff = NULL;
    long long *vmax = NULL;
    if (T) {
        int rc;
        // upload the table only when it changed since the last run
        std::vector<DevTarget> ht(T);
        for (size_t t = 0; t < T; t++) {
            memset(&ht[t], 0, sizeof ht[t]);
            ht[t].c_tid = targets[t].c_tid; ht[t].locus = targets[t].locus; ht[t].base = targets[t].base;
            const double thr = (double)targets[t].af * 2147483648.0;          // coinToss: rand() < p * (RAND_MAX + 1.0), p a float promoted to double
            ht[t].thresh = thr > 0 ? (thr >= 2147483648.0 ? 2147483648u : (uint32_t)ceil(thr)) : 0u;
        }
        if (!sp->d_tg || sp->tg_host.size() != T || memcmp(sp->tg_host.data(), ht.data(), T * sizeof(DevTarget)) != 0) {
            SSB_CUDA(ctx, cudaStreamSynchronize(s));
            if (sp->d_tg) { cudaFree(sp->d_tg); sp->d_tg = NULL; }
            SSB_CUDA(ctx, cudaMalloc(&sp->d_tg, T * sizeof(DevTarget)));
            SSB_CUDA(ctx, cudaMemcpy(sp->d_tg, ht.data(), T * sizeof(DevTarget), cudaMemcpyHostToDevice));
            sp->tg_host.swap(ht);
        }
        DevTarget *d_tg = sp->d_tg;
        d_res = ar.get<ssb_target_result>(T);
        long long *v = ar.get<long long>(T); vmax = ar.get<long long>(T);
        uint32_t *hitflag = ar.get<uint32_t>(T), *hidx = ar.get<uint32_t>(T);
        hits = ar.get<HitTarget>(T);
        unsigned long long *cnt = ar.get<unsigned long long>(T + 1); eoff = ar.get<unsigned long long>(T + 1);
        SPK_CHECK_ARENA(ar);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, target_lb_kernel, grid_for(T, 256), 256, 0, s, d_tg, T, runs, R, n_cov, rg, ord_base,
                     seq ? 1 : 0, pl.index, seq ? seq->carry_t : 0ll, seq ? seq->carry_h : -1ll, v);
        if (xc) { const double t0 = now_ms(); if ((rc = xc->allreduce_max_i64(v, T, s))) return rc; t_xc += now_ms() - t0; }
        if ((rc = scan_max_incl(ar, ctx, v, vmax, T))) return rc;
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, target_status_kernel, grid_for(T, 256), 256, 0, s, d_tg, T, vmax, runs, R, n_cov, ord_base, total_cov, is_last ? 1 : 0, d_res, hitflag);
        if ((rc = scan_sum(ar, ctx, hitflag, hidx, T))) return rc;
        SSB_CUDA(ctx, cudaMemsetAsync(hits, 0xff, T * sizeof(HitTarget), s));                       // tid < 0: not a hit
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, hits_kernel, grid_for(T, 256), 256, 0, s, d_tg, T, hitflag, hidx, d_res, ord_base, hits);
        SSB_LAUNCH(ctx, hit_totals_kernel, 1, 32, 0, s, hidx, hitflag, T, hits, &dsc->H, &dsc->last_hit_locus);
        SSB_CUDA(ctx, cudaMemsetAsync(cnt, 0, (T + 1) * sizeof(unsigned long long), s));
        if (K) SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, gather_count_kernel, grid_for(T * 32, 128), 128, 0, s, hits, T, k_start, k_end, K, &dsc->maxspan, cnt, d_err);
        if ((rc = scan_sum(ar, ctx, cnt, eoff, T + 1))) return rc;
        SSB_LAUNCH(ctx, copy_u64_kernel, 1, 32, 0, s, eoff + T, &dsc->E);
        if (seq) SSB_LAUNCH(ctx, carry_kernel, 1, 32, 0, s, vmax, T, ord_base + (long long)n_cov, seq->carry_t, seq->carry_h, &dsc->carry_t, &dsc->carry_h);
        if ((rc = publish())) return rc;                                                          // sync 3
        if (hsc->err.code) return fail_dev("gather");
        H = hsc->H; E = hsc->E; last_hit_locus = hsc->last_hit_locus;
    }
    stats->n_hits = (int64_t)H;
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[4], s));
    dbg_mark("targets");

    // ---------------------------------------------------------------- gather + rng + chain
    // every shard but the last walks all its loci: the offset at its end is what the next shard starts from
    const int64_t n_walk = is_last ? (H ? last_hit_locus + 1 : 0) : n_cov;
    const bool have_walk = n_walk > 0;
    unsigned long long k_in = seq ? seq->k : 0ull, k_out_final = k_in;
    bool k_in_known = !xc || pl.index == 0;
    Patch *patches = NULL; unsigned int patch_cap = 0;
    std::vector<OddFwd> odd_in, odd_out;
    if (seq) odd_in = seq->odd;
    bool chain_ran = false, sent = false;
    unsigned long long sent_k_out = 0;
    constexpr int RC_OVERRUN = 12345;

    // chain state (allocated only when there is something to walk)
    PlpEntry *ent = NULL; uint8_t *hflag = NULL;
    int P = 1; int64_t Lc = n_walk; int Rg = 1, Rg0 = 1, G = 1; bool Rg_fixed = false, wt_fixed = false; uint32_t wt = 16384;
    const double *h_mean = NULL, *h_var = NULL;
    unsigned int *d_flags = &dsc->flags, *n_patches = &dsc->n_patches;
    unsigned long long *d_draws = &dsc->draws, *d_pool_used = &dsc->pool_used;
    ChunkDesc *d_chunks = NULL, *d_serial = NULL; unsigned long long *d_gk = NULL;
    uint8_t *sw_d = NULL;
    ChainArgs A;
    memset(&A, 0, sizeof A);
    unsigned long long k_base = 0, M_abs = 0, stream_extra = 0;
    const unsigned long long halo_lines = h_halo_lines;

    auto import_odd = [&]() -> int {           // odd patches handed in by the shard before: part of the list before this shard's chain starts
        if (odd_in.empty()) return SSB_OK;
        if (!N) { snprintf(ctx->err, sizeof ctx->err, "spike: odd patches for a shard without reads"); return SSB_E_SHARD; }
        OddFwd *d_in = ar.get<OddFwd>(odd_in.size()); SPK_CHECK_ARENA(ar);
        SSB_CUDA(ctx, cudaMemcpyAsync(d_in, odd_in.data(), odd_in.size() * sizeof(OddFwd), cudaMemcpyHostToDevice, s));
        SSB_CUDA(ctx, cudaStreamSynchronize(s));
        SSB_LAUNCH(ctx, odd_import_kernel, 1, 32, 0, s, d_in, (unsigned int)odd_in.size(), halo_lines, keep, kord, d_odd, d_nodd, d_bloom, d_err);
        return SSB_OK;
    };
    auto reset_state = [&]() -> int {
        if (E) SSB_CUDA(ctx, cudaMemsetAsync(hflag, 0, E, s));
        SSB_CUDA(ctx, cudaMemsetAsync(n_patches, 0, sizeof(unsigned int), s));
        SSB_CUDA(ctx, cudaMemsetAsync(d_nodd, 0, sizeof(unsigned int), s));
        SSB_CUDA(ctx, cudaMemsetAsync(d_bloom, 0, sizeof(unsigned long long), s));
        SSB_CUDA(ctx, cudaMemsetAsync(d_flags, 0, sizeof(unsigned int), s));
        return import_odd();
    };
    // (re)generation of the rand() stream [k_base, M_abs) and its bit planes; the pointers in A are pre-offset so that kernels
    // index them with absolute draw numbers
    auto make_stream = [&](unsigned long long from, unsigned long long to) -> int {
        k_base = from / RNG_BLOCK * RNG_BLOCK;
        const unsigned long long M = (to - k_base + RNG_BLOCK - 1) / RNG_BLOCK * RNG_BLOCK;
        M_abs = k_base + M;
        const size_t nblocks = (size_t)(M / RNG_BLOCK);
        // per-block polynomials x^(310 + k_base + b*RNG_BLOCK) mod P: seed independent, built on the host (31x31 products)
        std::vector<uint32_t> bp(nblocks * GLIBC_DEG);
        uint32_t stepb[GLIBC_DEG], cur[GLIBC_DEG], tmpb[GLIBC_DEG];
        glibc_poly_xpow(RNG_BLOCK, stepb);
        glibc_poly_xpow(310 + k_base, cur);
        for (size_t b = 0; b < nblocks; b++) { memcpy(&bp[b * GLIBC_DEG], cur, sizeof cur); glibc_poly_mulmod(cur, stepb, tmpb); memcpy(cur, tmpb, sizeof cur); }
        const size_t ewords = (size_t)(M >> 5) + 160;
        int32_t *Rs = ar.get<int32_t>(M + 64);
        uint32_t *pe0 = ar.get<uint32_t>(ewords), *pe1 = ar.get<uint32_t>(ewords), *pej = ar.get<uint32_t>(ewords);
        SPK_CHECK_ARENA(ar);
        uint8_t *bp_h = NULL, *bp_d = NULL;                       // the generator reads its polynomial straight from mapped host memory (once per block)
        { int rcm; if ((rcm = map_get(bp.size() * sizeof(uint32_t), &bp_h, &bp_d))) return rcm; }
        memcpy(bp_h, bp.data(), bp.size() * sizeof(uint32_t));
        const uint32_t *d_bp = (const uint32_t *)bp_d;
        SSB_CUDA(ctx, cudaMemsetAsync(pe0 + (M >> 5), 0xAA, 160 * 4, s)); SSB_CUDA(ctx, cudaMemsetAsync(pe1 + (M >> 5), 0xCC, 160 * 4, s)); SSB_CUDA(ctx, cudaMemsetAsync(pej + (M >> 5), 0, 160 * 4, s));   // all four classes in every nibble: see walk_loci
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[12], s));
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, rng_fill_kernel, (int)nblocks, RNG_TPB, 0, s, d_bp, sp->d_rng_tab, (const uint32_t *)sw_d, Rs, M, pe0, pe1, pej);
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[13], s));
        A.R = Rs - k_base; A.e0 = pe0 - (k_base >> 5); A.e1 = pe1 - (k_base >> 5); A.ej = pej - (k_base >> 5); A.M = M_abs;
        return SSB_OK;
    };
    auto serial_span = [&](unsigned long long from) -> unsigned long long {          // generous stream end for one serial pass from `from`
        return from + (unsigned long long)((double)n_walk * 1.34 + 8.0 * sqrt((double)n_walk + 1.0)) + 3 * E + (1u << 17) + stream_extra;
    };
    // one serial pass over the shard from an exact offset: the plain chain, always right.  RC_OVERRUN: the stream was too short.
    auto serial_chain = [&](unsigned long long from) -> int {
        int rc2;
        if (!A.R || from < k_base || serial_span(from) > M_abs) { if ((rc2 = make_stream(from, serial_span(from)))) return rc2; }
        if ((rc2 = reset_state())) return rc2;
        SSB_LAUNCH(ctx, serial_chunk_kernel, 1, 32, 0, s, d_serial, n_walk, from, is_last ? ~0ull : CHUNK_WALK_ONLY);
        SSB_CUDA(ctx, cudaFuncSetAttribute(chain_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CK_SMEM));
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, chain_kernel<true>, 1, 32, CK_SMEM, s, A, d_serial, 1, d_draws, d_flags);
        if ((rc2 = publish())) return rc2;
        return (hsc->flags & CHAIN_OVERRUN) ? RC_OVERRUN : SSB_OK;
    };
    auto serial_chain_retry = [&](unsigned long long from) -> int {
        for (int attempt = 0; attempt < 12; attempt++) {
            const int rc2 = serial_chain(from);
            if (rc2 != RC_OVERRUN) return rc2;
            stream_extra = stream_extra ? stream_extra * 2 : (unsigned long long)n_walk + (1u << 20);
        }
        snprintf(ctx->err, sizeof ctx->err, "spike/chain: rand() stream exhausted");
        return SSB_E_STATE;
    };
    auto export_odd = [&]() -> int {           // odd patches on reads that reach into the next shard change what that shard sees
        odd_out.clear();
        if (!(xc || seq) || !hsc->n_odd) return SSB_OK;
        OddFwd *d_of = ar.get<OddFwd>(odd_cap); unsigned int *d_nof = ar.get<unsigned int>(1); SPK_CHECK_ARENA(ar);
        SSB_LAUNCH(ctx, odd_export_kernel, 1, 32, 0, s, d_odd, d_nodd, odd_cap, k_end, k_rec, (unsigned long long)N, rg, d_of, d_nof, odd_cap);
        unsigned int nof = 0;
        SSB_CUDA(ctx, cudaMemcpyAsync(&nof, d_nof, 4, cudaMemcpyDeviceToHost, s));
        SSB_CUDA(ctx, cudaStreamSynchronize(s));
        if (nof > odd_cap) nof = odd_cap;
        odd_out.resize(nof);
        if (nof) { SSB_CUDA(ctx, cudaMemcpyAsync(odd_out.data(), d_of, nof * sizeof(OddFwd), cudaMemcpyDeviceToHost, s)); SSB_CUDA(ctx, cudaStreamSynchronize(s)); }
        return SSB_OK;
    };
    auto send_offset = [&](unsigned long long k) -> int {
        if (!xc || pl.index + 1 >= pl.count || sent) return SSB_OK;
        HandOff out; out.k = k; out.n_odd = 0; out.pad = 0;
        const int rc2 = xc->send_next(&out, sizeof out);
        sent = true; sent_k_out = k;
        dbg_mark("offset out");
        return rc2;
    };

    if (!T) {                                   // the chain kernels index these even when there is no target
        eoff = ar.get<unsigned long long>(2); hits = ar.get<HitTarget>(1); d_res = ar.get<ssb_target_result>(1); SPK_CHECK_ARENA(ar);
        SSB_CUDA(ctx, cudaMemsetAsync(eoff, 0, 16, s));
    }
    if (have_walk) {
        int rc;
        ent = ar.get<PlpEntry>(E); hflag = ar.get<uint8_t>(E);
        patch_cap = (unsigned int)(2 * E + 16);
        patches = ar.get<Patch>(patch_cap);
        SPK_CHECK_ARENA(ar);
        if (H) {
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, gather_fill_kernel, grid_for(H * 32, 128), 128, 0, s, d_sam, recs, k_rec, hits, H, k_start, k_end, K, &dsc->maxspan, eoff, ent);
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, gather_mate_kernel, grid_for(H * 32, 128), 128, 0, s, d_sam, recs, k_rec, k_start, k_end, k_hash, K, nxt, hits, H, eoff, ent);
        }
        // reference classes of the covered loci the chain walks over
        cls = ar.get<uint8_t>((size_t)n_walk + 64); SPK_CHECK_ARENA(ar);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, cls_kernel, grid_for((size_t)n_walk, 256), 256, 0, s, runs, R, n_walk, (const uint8_t *const *)sp->d_seq_ptrs, sp->d_lens, cls, d_err);
        const size_t cwords = (size_t)((n_walk + 31) >> 5) + 160;
        uint32_t *pc0 = ar.get<uint32_t>(cwords), *pc1 = ar.get<uint32_t>(cwords), *pcx = ar.get<uint32_t>(cwords);
        SPK_CHECK_ARENA(ar);
        SSB_CUDA(ctx, cudaMemsetAsync(pc0, 0, cwords * 4, s)); SSB_CUDA(ctx, cudaMemsetAsync(pc1, 0, cwords * 4, s)); SSB_CUDA(ctx, cudaMemsetAsync(pcx, 0xff, cwords * 4, s));
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, cls_pack_kernel, grid_for(((size_t)n_walk + 31) & ~(size_t)31, 256), 256, 0, s, cls, n_walk, pc0, pc1, pcx);

        // ---- expected draws per chunk: window centres / widths, and the stream length
        const char *env_serial = getenv("SSB_CHAIN_SERIAL");
        const char *env_chunk = getenv("SSB_CHAIN_CHUNK");                 // loci per chunk (testing / tuning)
        // the chunked formulation pays off when the walk between targets dominates; every phase-1 walker dry-runs the pileups it
        // passes one entry at a time, so dense deep panels (pileup entries comparable to walked loci) stay on the one-warp serial
        // chain, which evaluates 32 entries per step (measured, tools/panel_probe.py: 2000x, 2000 targets: 1.75 s chunked, 0.2 s serial)
        const bool sparse_targets = (unsigned long long)E * 16ull < (unsigned long long)n_walk;
        if (!(env_serial && env_serial[0] == '1') && ((n_walk >= (1 << 20) && sparse_targets) || env_chunk)) {
            Lc = n_walk / 4096; if (Lc < 8192) Lc = 8192;              // phase 3 walks one chunk per warp: short chunks keep its chain short
            if (env_chunk && atoll(env_chunk) >= 64) Lc = atoll(env_chunk);
            Lc = (Lc + 31) & ~(int64_t)31;
            P = (int)((n_walk + Lc - 1) / Lc);
            if (P < 2) { P = 1; Lc = n_walk; }
        }
        double *d_mean = ar.get<double>((size_t)P), *d_var = ar.get<double>((size_t)P);
        d_chunks = ar.get<ChunkDesc>((size_t)P); d_serial = ar.get<ChunkDesc>(1);
        SPK_CHECK_ARENA(ar);
        uint8_t *mh = NULL, *md = NULL, *sw_h = NULL;
        if ((rc = map_get((size_t)P * 16, &mh, &md))) return rc;
        if ((rc = map_get(61 * 4, &sw_h, &sw_d))) return rc;
        uint32_t seedw[61];
        glibc_seed_window(seed, seedw);
        memcpy(sw_h, seedw, sizeof seedw);
        SSB_CUDA(ctx, cudaMemsetAsync(d_mean, 0, P * sizeof(double), s)); SSB_CUDA(ctx, cudaMemsetAsync(d_var, 0, P * sizeof(double), s));
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, chunk_stats_kernel, grid_for((size_t)P * 32, 128), 128, 0, s, pcx, n_walk, Lc, P, d_mean, d_var);
        if (H) SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, expect_kernel, grid_for(H * 32, 128), 128, 0, s, hits, H, eoff, ent, (const uint8_t *const *)sp->d_seq_ptrs, Lc, d_mean, d_var);
        SSB_LAUNCH(ctx, copy_words_kernel, 8, 256, 0, s, (const uint32_t *)d_mean, (uint32_t *)md, (unsigned int)(P * 2));
        SSB_LAUNCH(ctx, copy_words_kernel, 8, 256, 0, s, (const uint32_t *)d_var, (uint32_t *)(md + (size_t)P * 8), (unsigned int)(P * 2));
        if ((rc = publish())) return rc;                                                          // sync 4
        if (hsc->err.code) return fail_dev("reference");
        h_mean = (const double *)mh; h_var = h_mean + P;
        A.c0 = pc0; A.c1 = pc1; A.cx = pcx; A.n_walk = n_walk;
        A.hits = hits; A.H = H; A.eoff = eoff; A.ent = ent; A.hflag = hflag; A.res = d_res;
        A.patches = patches; A.n_patches = n_patches; A.patch_cap = patch_cap;
        A.odd = d_odd; A.n_odd = d_nodd; A.odd_cap = odd_cap; A.odd_bloom = d_bloom;
        A.contig_seq = (const uint8_t *const *)sp->d_seq_ptrs; A.err = d_err;
        // groups of Rg consecutive chunks share one start-offset window; the window is cut into slices of ~wt offsets
        Rg = (int)(114688 / Lc); if (Rg < 1) Rg = 1;                        // phase 1 works on groups of ~112 k loci (see spike_chain.cuh)
        Rg0 = Rg;
        if (const char *e = getenv("SSB_CHAIN_GROUP")) { if (atoi(e) >= 1) { Rg = atoi(e); Rg_fixed = true; } }
        if (const char *e = getenv("SSB_CHAIN_SLICE")) { if (atoi(e) >= 1) { wt = (uint32_t)atoi(e); wt_fixed = true; } }
        G = (P + Rg - 1) / Rg;
        d_gk = ar.get<unsigned long long>((size_t)G); SPK_CHECK_ARENA(ar);
    }
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[5], s));
    dbg_mark("gathered");

    // ---------------------------------------------------------------- emit
    if (K) {
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[8], s));
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_EMIT, emit_kernel, ctx->sm_count * 8, 256, 0, s, d_sam, n, d_edesc, out_off, K, d_out);
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[9], s));
    }

    // ---------------------------------------------------------------- tallies of the non-target loci (no odd patch known yet)
    unsigned long long *err64 = NULL; unsigned int *minus = NULL;
    TallyArgs TA;
    memset(&TA, 0, sizeof TA);
    const bool use_list = exc_list && !no_list && n_list <= exc_cap;
    auto tally_pass = [&]() -> int {
        SSB_CUDA(ctx, cudaMemsetAsync(err64, 0, ((size_t)n_cov + 1) * sizeof(unsigned long long), s));
        SSB_CUDA(ctx, cudaMemsetAsync(minus, 0, ((size_t)n_cov + 1) * sizeof(unsigned int), s));
        if (use_list) {
            if (n_list) SSB_LAUNCH_P(ctx, SSB_K_SPIKE_TALLY, tally_resolve_kernel, grid_for((size_t)n_list, 128), 128, 0, s, TA, exc_list, n_list, keep, kord);
        } else {
            KMeta *kmeta = ar.get<KMeta>(K); SPK_CHECK_ARENA(ar);
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_TALLY, kmeta_kernel, grid_for(K, 256), 256, 0, s, recs, k_rec, K, kmeta);
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_TALLY, tally_fast_kernel, grid_for(K * 32, 128), 128, 0, s, TA, kmeta);
        }
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_TALLY, tally_kernel, grid_for(K, 128), 128, 0, s, TA);
        return SSB_OK;
    };
    if (n_cov) {
        int rc;
        err64 = ar.get<unsigned long long>((size_t)n_cov + 1); minus = ar.get<unsigned int>((size_t)n_cov + 1);
        SPK_CHECK_ARENA(ar);
        TA.sam = d_sam; TA.recs = recs; TA.k_rec = k_rec; TA.k_start = k_start; TA.k_end = k_end; TA.k_hash = k_hash; TA.k_bits = k_bits; TA.K = K;
        TA.nxt = nxt; TA.prv = prv; TA.cplx = cplx; TA.maxspan = h_maxspan; TA.runs = runs; TA.R = R;
        TA.contig_seq = (const uint8_t *const *)sp->d_seq_ptrs; TA.contig_len = sp->d_lens; TA.err64 = err64; TA.minus = minus; TA.err = d_err;
        TA.odd = d_odd; TA.n_odd = d_nodd; TA.odd_bloom = d_bloom; TA.listed_only = use_list ? 1 : 0; TA.rg = rg;
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[10], s));
        if ((rc = tally_pass())) return rc;
        SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[11], s));
    }

    // ---- shards: where in the stream does this shard begin (expected), and how sure is that
    double c_in = (double)k_in, v_in = 0;
    if (xc) {
        int rc;
        ShardExpect me; me.mean = 0; me.var = 0; me.H = H; me.pad = 0;
        if (have_walk) for (int f = 0; f < P; f++) { me.mean += h_mean[f]; me.var += h_var[f]; }
        std::vector<ShardExpect> all((size_t)xc->n);
        const double t0 = now_ms();
        if ((rc = xc->allgather(&me, all.data(), sizeof me))) return rc;
        t_xc += now_ms() - t0;
        c_in = 0;
        for (int g = 0; g < pl.index; g++) { c_in += all[g].mean; v_in += all[g].var; }
    }

    if (have_walk) {
        int rc;
        bool parallel = P > 1;
        // window geometry of the groups (host): centre = expected offset, half width = `sigmas` standard deviations
        double sigmas = 4.0;
        if (const char *e = getenv("SSB_CHAIN_SIGMA")) { const double v = atof(e); if (v >= 0.5 && v <= 12.0) sigmas = v; }
        std::vector<GroupDesc> h_groups; std::vector<SliceDesc> h_slices;
        unsigned long long woff = 0; double cm_end = 0, cv_end = 0;
        auto make_geometry = [&](double centre, double var0, bool exact_entry) {
            G = (P + Rg - 1) / Rg;
            h_groups.assign((size_t)G, GroupDesc()); h_slices.clear(); woff = 0;
            double cm = centre, cv = var0;
            for (int q = 0; q < G; q++) {
                GroupDesc &gd = h_groups[q];
                gd.f0 = q * Rg; gd.nf = (gd.f0 + Rg <= P) ? Rg : P - gd.f0;
                const bool one = q == 0 && exact_entry;
                const double half = one ? 0.0 : sigmas * sqrt(cv) + 32.0;    // a walker outside its group's window (6e-5 per group at 4 sigma) is walked again on its own
                double lo = cm - half; if (lo < 0) lo = 0;
                gd.klo = (unsigned long long)lo; gd.W = one ? 1u : (uint32_t)(cm + half - (double)gd.klo) + 2u;
                uint32_t S = (gd.W + wt - 1) / wt; gd.w = (gd.W + S - 1) / S; S = (gd.W + gd.w - 1) / gd.w;
                gd.S = S; gd.b0 = (uint32_t)h_slices.size(); gd.toff = woff;
                for (uint32_t sl = 0; sl < S; sl++) {
                    SliceDesc sd; sd.q = q; sd.i0 = sl * gd.w; sd.n = (sd.i0 + gd.w <= gd.W) ? gd.w : gd.W - sd.i0; sd.off = woff; woff += sd.n;
                    h_slices.push_back(sd);
                }
                for (int f = gd.f0; f < gd.f0 + gd.nf; f++) { cm += h_mean[f]; cv += h_var[f]; }
            }
            cm_end = cm; cv_end = cv;
        };
        // Every slice is one block, and a block lives as long as its group is long: more slices than the device holds at once means a second
        // round of blocks behind the first (a shard far down the stream has windows several times as wide as the first one's).  Longer groups
        // need fewer slices and less work, at the price of a longer lone-walker tail: the shortest group length whose slices (at their widest) fill at most 85 % of the device.
        size_t resident = (size_t)sp->p1_resident;
        if (const char *e = getenv("SSB_P1_RESIDENT")) { if (atoi(e) >= 1) resident = (size_t)atoi(e); }          // (tests: a device that holds only a few blocks)
        auto choose_geometry = [&](double centre, double var0, bool exact_entry) {
            static const int num[] = {2, 3, 4, 6, 8, 12, 16, 24, 32};       // group length in halves of the base length
            if (!wt_fixed) wt = 16384;
            for (size_t i = 0; i < sizeof num / sizeof num[0]; i++) {
                if (!Rg_fixed) { Rg = Rg0 * num[i] / 2; if (Rg < 1) Rg = 1; }
                make_geometry(centre, var0, exact_entry);
                if (Rg_fixed || h_slices.size() * 20 <= resident * 17 || Rg >= P) break;     // 85 %: room to narrow the slices below (tools/sweep_late_shard.sh)
            }
            // ... and the narrowest slices that still fit: the same work in more blocks keeps more warps in flight in the long tail of a group
            // (C2, one B200: 16384 offsets per slice 12.2 ms, 12288 11.7, 10240 10.9)
            if (!wt_fixed && h_slices.size() <= resident) {
                for (uint32_t w = wt - 1024; w >= 4096; w -= 1024) {
                    const uint32_t keep = wt;
                    wt = w; make_geometry(centre, var0, exact_entry);
                    if (h_slices.size() > resident) { wt = keep; make_geometry(centre, var0, exact_entry); break; }
                }
            }
        };

        int n_retries = 0;
        bool chain_done = false;
        for (int attempt = 0; attempt < 8 && !chain_done; attempt++) {
            if (!parallel) {
                // ---- the one-warp serial chain (small inputs, dense panels, and every fallback)
                if (!k_in_known) {
                    HandOff ho;
                    const double t0 = now_ms();
                    if ((rc = xc->recv_prev(&ho, sizeof ho))) return rc;
                    stats->ms_handoff_wait += (float)(now_ms() - t0);
                    k_in = ho.k; k_in_known = true;
                    dbg_mark("offset in");
                }
                if ((rc = serial_chain_retry(k_in))) return rc;
                k_out_final = hsc->draws;
                stats->chain_mode = 1;
                if ((rc = send_offset(k_out_final))) return rc;
                chain_done = true;
                break;
            }
            const bool exact_entry = k_in_known;
            double v_extra = 0.0;                               // SSB_CHAIN_EXTRA_VAR: widen the windows as if that many draws' variance lay in front (measurement: a late shard's phase 1 on one GPU)
            if (const char *e = getenv("SSB_CHAIN_EXTRA_VAR")) { const double v = atof(e); if (v > 0) v_extra = v; }
            choose_geometry(exact_entry ? (double)k_in : c_in, (exact_entry ? 0.0 : v_in) + v_extra, exact_entry);
            const size_t n_slices = h_slices.size();
            const unsigned long long pool_cap = woff + (1ull << 20);
            // the stream must cover the top of the last window (and everything a lone walker can reach)
            const unsigned long long need_to = (unsigned long long)(cm_end + 8.0 * sqrt(cv_end)) + 3 * E + (1u << 17) + stream_extra;
            if ((rc = make_stream(h_groups[0].klo, need_to))) return rc;
            if ((rc = reset_state())) return rc;
            constexpr int SPARE = 32;                           // single-walker slices for groups whose window the exact walker missed
            const unsigned long long wstride = woff + SPARE;
            BoundaryList *d_lists = ar.get<BoundaryList>((n_slices + SPARE) * (size_t)Rg);
            unsigned long long *kbuf = ar.get<unsigned long long>(2 * wstride), *pool_k = ar.get<unsigned long long>(pool_cap), *exit_k = NULL;
            uint32_t *lobuf = ar.get<uint32_t>(2 * wstride), *pool_lo = ar.get<uint32_t>(pool_cap);
            GroupDesc *d_groups = ar.get<GroupDesc>((size_t)G); SliceDesc *d_slices = ar.get<SliceDesc>(n_slices + SPARE);
            unsigned long long *d_kin = ar.get<unsigned long long>(1);
            if (!exact_entry) exit_k = ar.get<unsigned long long>(pool_cap);
            SPK_CHECK_ARENA(ar);
            {   // descriptors: host -> mapped scratch -> device arrays by a kernel (no copy engine: it may be busy with the host link)
                static_assert(sizeof(GroupDesc) % 4 == 0 && sizeof(SliceDesc) % 4 == 0, "descriptor words");
                uint8_t *gh = NULL, *gd_ = NULL, *sh_ = NULL, *sd_ = NULL;
                if ((rc = map_get(G * sizeof(GroupDesc), &gh, &gd_))) return rc;
                if ((rc = map_get(n_slices * sizeof(SliceDesc), &sh_, &sd_))) return rc;
                memcpy(gh, h_groups.data(), G * sizeof(GroupDesc)); memcpy(sh_, h_slices.data(), n_slices * sizeof(SliceDesc));
                SSB_LAUNCH(ctx, copy_words_kernel, 4, 256, 0, s, (const uint32_t *)gd_, (uint32_t *)d_groups, (unsigned int)(G * sizeof(GroupDesc) / 4));
                SSB_LAUNCH(ctx, copy_words_kernel, 16, 256, 0, s, (const uint32_t *)sd_, (uint32_t *)d_slices, (unsigned int)(n_slices * sizeof(SliceDesc) / 4));
            }
            SSB_LAUNCH(ctx, chunks_init_kernel, (P + 127) / 128, 128, 0, s, d_chunks, P, Lc, n_walk);
            unsigned long long *d_dbg = NULL;
            if (dbg_t) { d_dbg = ar.get<unsigned long long>(8 + 2 * n_slices); SPK_CHECK_ARENA(ar); SSB_CUDA(ctx, cudaMemsetAsync(d_dbg, 0, (8 + 2 * n_slices) * 8, s)); }
            SSB_CUDA(ctx, cudaMemsetAsync(d_pool_used, 0, 8, s));
            SSB_CUDA(ctx, cudaMemsetAsync(d_lists, 0, (n_slices + SPARE) * (size_t)Rg * sizeof(BoundaryList), s));
            SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[14], s));
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, phase1_kernel, (int)n_slices, P1_THREADS, P1_SMEM, s, A, Lc, d_groups, d_slices, kbuf, lobuf, wstride,
                         d_lists, Rg, pool_k, pool_lo, d_pool_used, pool_cap, d_flags, d_dbg, 0);
            SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[15], s));
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, map_fill_kernel, (int)n_slices, 128, 0, s, d_groups, d_slices, d_lists, Rg, pool_k, pool_lo, kbuf, 0);     // group maps as flat tables (over the walker slots)
            if (d_dbg) {
                unsigned long long h_dbg[8];
                SSB_CUDA(ctx, cudaMemcpyAsync(h_dbg, d_dbg, 64, cudaMemcpyDeviceToHost, s));
                SSB_CUDA(ctx, cudaStreamSynchronize(s));
                fprintf(stderr, "[chain %d] chunks=%d L=%lld groups=%d slices=%zu walkers=%llu walker-loci=%llu rounds=%llu final survivors: sum %llu max %llu\n",
                        pl.index, P, (long long)Lc, G, n_slices, woff, h_dbg[0], h_dbg[3], h_dbg[1], h_dbg[2]);
                fprintf(stderr, "[chain %d] phase 1 block cycles: rounds with > %d walkers %.3g (avg per block), later rounds %.3g, slowest block %.3g\n", pl.index, P1_THREADS,
                        (double)h_dbg[4] / (double)n_slices, (double)h_dbg[5] / (double)n_slices, (double)h_dbg[6]);
            }
            if (!exact_entry) {
                // ---- shards: prepare the answer, then the exact offset arrives and the exit offset leaves
                SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, precompose_kernel, (int)(h_groups[0].S < 1024 ? h_groups[0].S : 1024), 128, 0, s, G, d_groups, d_lists, Rg, pool_k, pool_lo, exit_k);
                HandOff ho;
                const double t0 = now_ms();
                if ((rc = xc->recv_prev(&ho, sizeof ho))) return rc;
                stats->ms_handoff_wait += (float)(now_ms() - t0);
                k_in = ho.k; k_in_known = true;
                dbg_mark("offset in");
                uint8_t *kh = NULL, *kd = NULL;
                if ((rc = map_get(8, &kh, &kd))) return rc;
                *(volatile unsigned long long *)kh = k_in;
                SSB_LAUNCH(ctx, copy_u64_kernel, 1, 32, 0, s, (const unsigned long long *)kd, d_kin);
                SSB_LAUNCH(ctx, entry_kernel, 1, 32, 0, s, d_groups, d_lists, Rg, pool_lo, exit_k, d_kin, &dsc->k_out);
                if ((rc = publish())) return rc;
                if (hsc->flags & CHAIN_OVERRUN) { stream_extra = stream_extra ? stream_extra * 2 : (unsigned long long)(M_abs - k_base); continue; }   // again, now from the exact offset
                if (hsc->flags) { parallel = false; continue; }                                   // phase 1 gave up: walk serially from the exact offset
                if (hsc->k_out != ~0ull) { if ((rc = send_offset(hsc->k_out))) return rc; }       // else: a window was missed on the way; the composition below finds out where
            } else {
                uint8_t *kh = NULL, *kd = NULL;
                if ((rc = map_get(8, &kh, &kd))) return rc;
                *(volatile unsigned long long *)kh = k_in;
                SSB_LAUNCH(ctx, copy_u64_kernel, 1, 32, 0, s, (const unsigned long long *)kd, d_kin);
            }
            // ---- compose from the exact offset, chunk boundaries, phase 3.  A walker that leaves its group's window is walked through
            //      that group again on its own (one block, exact entry), and the composition is repeated.
            bool restart = false;
            for (int retry = 0; retry <= SPARE; retry++) {
                SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, compose_kernel, 1, 32, 0, s, G, d_groups, kbuf, d_kin, d_gk, &dsc->k_end, d_flags, dsc->miss);
                SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, boundary_kernel, (P + 127) / 128, 128, 0, s, P, Rg, d_groups, d_lists, Rg, pool_k, pool_lo, d_gk, d_chunks, d_flags);
                if ((rc = publish())) return rc;                                                  // did the exact walker stay inside every window?
                if (!hsc->flags) {
                    if ((rc = send_offset(hsc->k_end))) return rc;                                // the exit offset leaves as soon as the maps are composed
                    SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, chain_kernel<false>, grid_for((size_t)P * 32, 128), 128, 0, s, A, d_chunks, P, d_draws, d_flags);
                    if ((rc = publish())) return rc;                                              // sync 5
                }
                if (dbg_t) fprintf(stderr, "[chain %d] flags after phases 1-3: %u, odd patches %u\n", pl.index, (unsigned)hsc->flags, (unsigned)hsc->n_odd);
                if (hsc->flags == (unsigned int)CHAIN_MISS && retry < SPARE) {
                    const int q = (int)hsc->miss[0]; const unsigned long long km = hsc->miss[1];
                    if (dbg_t) fprintf(stderr, "[chain %d] window of group %d missed (offset %llu, window [%llu, +%u)): walking it alone\n", pl.index, q, km, h_groups[q].klo, h_groups[q].W);
                    if (km < k_base || km + 64 > M_abs) { restart = true; break; }                // outside the generated stream: start over with a longer one
                    GroupDesc gd = h_groups[q];
                    gd.klo = km; gd.W = 1; gd.w = 1; gd.S = 1; gd.b0 = (uint32_t)(n_slices + retry); gd.toff = woff + retry;
                    h_groups[q] = gd;
                    SliceDesc sd; sd.q = q; sd.i0 = 0; sd.n = 1; sd.off = woff + retry;
                    uint8_t *gh = NULL, *gd_ = NULL, *sh_ = NULL, *sd_ = NULL;
                    if ((rc = map_get(sizeof gd, &gh, &gd_))) return rc;
                    if ((rc = map_get(sizeof sd, &sh_, &sd_))) return rc;
                    memcpy(gh, &gd, sizeof gd); memcpy(sh_, &sd, sizeof sd);
                    SSB_LAUNCH(ctx, copy_words_kernel, 1, 32, 0, s, (const uint32_t *)gd_, (uint32_t *)(d_groups + q), (unsigned int)(sizeof gd / 4));
                    SSB_LAUNCH(ctx, copy_words_kernel, 1, 32, 0, s, (const uint32_t *)sd_, (uint32_t *)(d_slices + n_slices + retry), (unsigned int)(sizeof sd / 4));
                    if ((rc = reset_state())) return rc;
                    SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, phase1_kernel, 1, P1_THREADS, P1_SMEM, s, A, Lc, d_groups, d_slices, kbuf, lobuf, wstride,
                                 d_lists, Rg, pool_k, pool_lo, d_pool_used, pool_cap, d_flags, (unsigned long long *)NULL, (int)(n_slices + retry));
                    SSB_LAUNCH_P(ctx, SSB_K_SPIKE_CHAIN, map_fill_kernel, 1, 128, 0, s, d_groups, d_slices, d_lists, Rg, pool_k, pool_lo, kbuf, (int)(n_slices + retry));
                    n_retries++;
                    continue;
                }
                break;
            }
            if (restart) { stream_extra = stream_extra ? stream_extra * 2 : (unsigned long long)(M_abs - k_base); continue; }
            if (hsc->flags & CHAIN_OVERRUN) { stream_extra = stream_extra ? stream_extra * 2 : (unsigned long long)(M_abs - k_base); continue; }
            if (hsc->flags || hsc->n_odd) { parallel = false; continue; }                          // too complex / odd patches (or misses without end): the plain serial chain decides
            k_out_final = is_last ? hsc->draws : hsc->k_end;
            stats->chain_mode = P;
            stats->n_window_retries = n_retries;
            chain_done = true;
        }
        if (!chain_done) { snprintf(ctx->err, sizeof ctx->err, "spike/chain: rand() stream exhausted"); return SSB_E_STATE; }
        if (hsc->err.code) return fail_dev("chain");
        chain_ran = true;
        if ((rc = send_offset(k_out_final))) return rc;
        if ((rc = export_odd())) return rc;
    } else {
        // nothing to walk here: the offset passes through
        int rc;
        if (xc && pl.index > 0) {
            HandOff ho;
            const double t0 = now_ms();
            if ((rc = xc->recv_prev(&ho, sizeof ho))) return rc;
            stats->ms_handoff_wait += (float)(now_ms() - t0);
            k_in = ho.k; k_in_known = true;
        }
        k_out_final = k_in;
        if ((rc = send_offset(k_out_final))) return rc;
    }
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[6], s));

    // ---- shards: did anybody change an offset (or a base a later shard looks at) after sending?  then the shards behind it
    // run again, one after the other, each from the exact state of its predecessor
    if (xc) {
        int rc;
        const bool dirty = sent && (sent_k_out != k_out_final || !odd_out.empty());
        ShardVerdict me; me.k_out = k_out_final; me.dirty = dirty ? 1u : 0u; me.n_odd_fwd = (unsigned int)odd_out.size();
        std::vector<ShardVerdict> all((size_t)xc->n);
        const double t0 = now_ms();
        if ((rc = xc->allgather(&me, all.data(), sizeof me))) return rc;
        t_xc += now_ms() - t0;
        int first_dirty = -1;
        for (int g = 0; g < xc->n; g++) if (all[g].dirty) { first_dirty = g; break; }
        if (first_dirty >= 0 && pl.index >= first_dirty) {
            if (dbg_t) fprintf(stderr, "[chain %d] second round from shard %d\n", pl.index, first_dirty);
            if (pl.index > first_dirty) {
                HandOff ho;
                if ((rc = xc->recv_prev(&ho, sizeof ho))) return rc;
                std::vector<OddFwd> in(ho.n_odd);
                if (ho.n_odd && (rc = xc->recv_prev(in.data(), in.size() * sizeof(OddFwd)))) return rc;
                if (ho.k != k_in || !in.empty() || !odd_in.empty()) {
                    k_in = ho.k; odd_in = in;
                    if (have_walk) {
                        if ((rc = serial_chain_retry(k_in))) return rc;
                        if (hsc->err.code) return fail_dev("chain");
                        k_out_final = hsc->draws; stats->chain_mode = 1;
                        if ((rc = export_odd())) return rc;
                    } else { k_out_final = k_in; odd_out = in; }
                }
            }
            if (pl.index + 1 < pl.count) {
                HandOff out; out.k = k_out_final; out.n_odd = (unsigned int)odd_out.size(); out.pad = 0;
                if ((rc = xc->send_next(&out, sizeof out))) return rc;
                if (out.n_odd && (rc = xc->send_next(odd_out.data(), odd_out.size() * sizeof(OddFwd)))) return rc;
            }
        }
    }
    dbg_mark("chain-end");
    stats->rng_k_in = (int64_t)k_in; stats->rng_k_out = (int64_t)k_out_final;
    stats->rng_draws = (int64_t)k_out_final;

    // ---------------------------------------------------------------- patches
    std::vector<FwdPatch> fwd_out, fwd_in;
    {
        int rc;
        // bases this shard spiked into reads the next shard writes
        if ((xc || seq) && chain_ran && patches) {
            // written by the kernel straight into mapped host memory (a handful of entries: reads that straddle the cut AND were spiked)
            const unsigned int fwd_cap = patch_cap < 32768u ? patch_cap : 32768u;
            uint8_t *fh = NULL, *fd = NULL;
            if ((rc = map_get((size_t)fwd_cap * sizeof(FwdPatch), &fh, &fd))) return rc;
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, fwd_collect_kernel, 16, 256, 0, s, patches, &dsc->n_patches, k_rec, k_end, rg, (unsigned long long)N, (FwdPatch *)fd, &dsc->n_fwd, fwd_cap, d_err);
            if ((rc = publish())) return rc;
            if (hsc->err.code) return fail_dev("forward");
            const unsigned int nf = hsc->n_fwd < fwd_cap ? hsc->n_fwd : fwd_cap;
            fwd_out.assign((const FwdPatch *)fh, (const FwdPatch *)fh + nf);
        }
        if (xc) {
            unsigned long long cnt_out = fwd_out.size(), cnt_in = 0;
            const double t0 = now_ms();
            if ((rc = xc->shift(&cnt_out, 8, &cnt_in, 8))) return rc;
            fwd_in.resize((size_t)cnt_in);
            if ((rc = xc->shift(fwd_out.data(), fwd_out.size() * sizeof(FwdPatch), fwd_in.data(), fwd_in.size() * sizeof(FwdPatch)))) return rc;
            t_xc += now_ms() - t0;
        } else if (seq) fwd_in = seq->fwd;
        // bases the previous shard spiked into reads this shard writes: first, so that this shard's own (later) loci win
        if (!fwd_in.empty()) {
            if (!K) { snprintf(ctx->err, sizeof ctx->err, "spike: forwarded bases for a shard without reads"); return SSB_E_SHARD; }
            // several bases for one position: the one made at the latest locus wins (the list is short)
            std::vector<FwdPatch> uniq;
            for (const FwdPatch &f : fwd_in) {
                bool found = false;
                for (FwdPatch &u : uniq) if (u.from_end == f.from_end && u.qpos == f.qpos) { if (f.order >= u.order) u = f; found = true; break; }
                if (!found) uniq.push_back(f);
            }
            uint8_t *ih = NULL, *id_ = NULL;
            if ((rc = map_get(uniq.size() * sizeof(FwdPatch), &ih, &id_))) return rc;
            memcpy(ih, uniq.data(), uniq.size() * sizeof(FwdPatch));
            SSB_LAUNCH(ctx, fwd_apply_kernel, 4, 128, 0, s, (const FwdPatch *)id_, (unsigned int)uniq.size(), halo_lines, keep, kord, recs, k_end, ord_off, rg, d_out, d_err);
        }
        if (chain_ran && patches) {
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, patch_kernel, 64, 256, 0, s, patches, &dsc->n_patches, recs, k_rec, k_end, ord_off, rg, d_out);
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, odd_fix_kernel, 4, 128, 0, s, d_odd, d_nodd, odd_cap, patches, &dsc->n_patches, recs, k_rec, k_end, ord_off, rg, d_out);
        }
        stats->n_forwarded = (int64_t)fwd_out.size();
    }
    dbg_mark("patched");

    // ---------------------------------------------------------------- SEQ_ERROR records
    if (n_cov) {
        int rc;
        if (hsc->n_odd) { if ((rc = tally_pass())) return rc; }                                 // odd patches change bases later loci see: tally again with the list
        if (H) SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, tally_clear_hits_kernel, grid_for(H, 256), 256, 0, s, hits, H, err64);
        uint32_t *sflag = ar.get<uint32_t>((size_t)n_cov), *sidx = ar.get<uint32_t>((size_t)n_cov);
        SPK_CHECK_ARENA(ar);
        SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, tally_flag_kernel, grid_for((size_t)n_cov, 256), 256, 0, s, err64, n_cov, sflag);
        if ((rc = scan_sum(ar, ctx, sflag, sidx, (size_t)n_cov))) return rc;
        SSB_LAUNCH(ctx, se_total_kernel, 1, 32, 0, s, sidx, sflag, n_cov, &dsc->n_se);
        if ((rc = publish())) return rc;                                                          // sync 6
        if (hsc->err.code) return fail_dev("reference");
        sp->n_se = (size_t)hsc->n_se;
        if (sp->n_se) {
            SSB_CUDA(ctx, cudaMallocAsync((void **)&sp->d_se, sp->n_se * sizeof(ssb_seq_error), s));
            SSB_LAUNCH_P(ctx, SSB_K_SPIKE_OTHER, tally_emit_kernel, grid_for((size_t)n_cov, 256), 256, 0, s, err64, minus, sflag, sidx, n_cov, runs, R,
                         cum_s, cum_e, (const uint8_t *const *)sp->d_seq_ptrs, ord_base, sp->d_se);
        }
    }
    SSB_CUDA(ctx, cudaEventRecord(sp->ev_t[7], s));
    // per-target results: written by a kernel into mapped host memory.  Shards processed one after the other only report the targets
    // they consumed (a contiguous run of the table, plus the left-over tail on the last shard): the rest is SSB_T_ELSEWHERE.
    size_t r_lo = 0, r_hi = T;
    if (T && d_res) {
        { int rc; if ((rc = publish())) return rc; }
        if (seq) { r_lo = (size_t)seq->carry_t; r_hi = is_last ? T : (size_t)hsc->carry_t; if (r_hi < r_lo) r_hi = r_lo; }
        const size_t nb = (r_hi - r_lo) * sizeof(ssb_target_result);
        if (nb > sp->h_res_bytes) {
            SSB_CUDA(ctx, cudaStreamSynchronize(s));
            if (sp->h_res) { cudaFreeHost(sp->h_res); sp->h_res = NULL; sp->h_res_bytes = 0; }
            SSB_CUDA(ctx, cudaHostAlloc((void **)&sp->h_res, nb + (nb >> 2) + 4096, cudaHostAllocMapped));
            sp->h_res_bytes = nb + (nb >> 2) + 4096;
        }
        if (nb) {
            uint8_t *hr_dev = NULL;
            SSB_CUDA(ctx, cudaHostGetDevicePointer((void **)&hr_dev, sp->h_res, 0));
            static_assert(sizeof(ssb_target_result) % 4 == 0, "result words");
            SSB_LAUNCH(ctx, copy_words_kernel, 64, 256, 0, s, (const uint32_t *)(d_res + r_lo), (uint32_t *)hr_dev, (unsigned int)(nb / 4));
        }
    }
    { int rc; if ((rc = publish())) return rc; }
    SSB_CUDA(ctx, cudaStreamSynchronize(s));
    if (hsc->err.code) return fail_dev("finish");
    if (T && d_res) {
        if (seq) for (size_t t = 0; t < T; t++) if (t < r_lo || t >= r_hi) { memset(&results[t], 0, sizeof results[t]); results[t].status = SSB_T_ELSEWHERE; results[t].at_tid = -1; results[t].at_pos = -1; results[t].rng_offset = -1; }
        if (r_hi > r_lo) memcpy(results + r_lo, sp->h_res, (r_hi - r_lo) * sizeof(ssb_target_result));
    }
    *out_bytes = (size_t)hsc->total_out;
    stats->out_bytes = (int64_t)hsc->total_out;
    stats->alignmentCount = (int64_t)hsc->n_owned;                                        // every read is written exactly once, by the shard that owns its last base (:1275,:1365)
    stats->maxDepth = (int64_t)hsc->maxdepth;
    if (hsc->total_out > out_cap) { snprintf(ctx->err, sizeof ctx->err, "spike: output needs %llu bytes, capacity %zu", (unsigned long long)hsc->total_out, out_cap); return SSB_E_ARG; }
    if (hsc->maxdepth > (unsigned int)MAX_PILEUP) { snprintf(ctx->err, sizeof ctx->err, "spike: pileup depth %u exceeds MAX_PILEUP_SIZE", hsc->maxdepth); return SSB_E_DEPTH; }
    if (seq) {
        seq->k = k_out_final; seq->ord_base = ord_base + n_cov;
        if (T) { seq->carry_t = hsc->carry_t; seq->carry_h = hsc->carry_h; }
        seq->fwd.swap(fwd_out); seq->odd.swap(odd_out);
        seq->first_strad = h_first_strad; seq->maxspan = h_maxspan;
    }
    stats->ms_parse = ev_ms(sp->ev_t[0], sp->ev_t[1]);
    stats->ms_sort = ev_ms(sp->ev_t[1], sp->ev_t[2]);
    stats->ms_cover = ev_ms(sp->ev_t[2], sp->ev_t[3]);
    stats->ms_gather = ev_ms(sp->ev_t[3], sp->ev_t[5]);
    stats->ms_chain = have_walk ? ev_ms(sp->ev_t[5], sp->ev_t[6]) : 0;
    if (have_walk && A.R) stats->ms_rng = ev_ms(sp->ev_t[12], sp->ev_t[13]);
    if (have_walk && stats->chain_mode > 1) stats->ms_phase1 = ev_ms(sp->ev_t[14], sp->ev_t[15]);
    stats->ms_patch = ev_ms(sp->ev_t[6], sp->ev_t[7]);
    if (K) { stats->ms_emit = ev_ms(sp->ev_t[8], sp->ev_t[9]); }
    if (n_cov) stats->ms_tally = ev_ms(sp->ev_t[10], sp->ev_t[11]);
    stats->ms_exchange = (float)t_xc;
    stats->ms_total = (float)(now_ms() - t_host0);
    return SSB_OK;
}

} // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
namespace {
int plan_from_shard(const ssb_spike_shard *sh, ssb_exchange *xc, ShardPlan &pl)
{
    if (!sh) return SSB_OK;
    if (sh->count < 1 || sh->index < 0 || sh->index >= sh->count || sh->lo_tid < 0 || sh->hi_tid < 0 || sh->lo_pos < 0 || sh->hi_pos < 0 ||
        sh->lo_pos > 0xffffffffll || sh->hi_pos > 0xffffffffll) return SSB_E_ARG;
    pl.index = sh->index; pl.count = sh->count;
    pl.rg.lo = ((unsigned long long)(uint32_t)sh->lo_tid << 32) | (unsigned long long)sh->lo_pos;
    pl.rg.hi = ((unsigned long long)(uint32_t)sh->hi_tid << 32) | (unsigned long long)sh->hi_pos;
    if (sh->index == 0) pl.rg.lo = 0;
    if (sh->index == sh->count - 1) pl.rg.hi = ~0ull;
    if (pl.rg.lo >= pl.rg.hi) return SSB_E_ARG;
    pl.halo_bytes = (size_t)sh->halo_bytes;
    pl.xc = xc;
    if (sh->count > 1 && (!xc || xc->n != sh->count || xc->rank != sh->index)) return SSB_E_ARG;
    return SSB_OK;
}
} // namespace

extern "C" int ssb_spike_run_shard_device(ssb_spike *sp, const ssb_spike_shard *shard, ssb_exchange *xc, const uint8_t *d_sam, size_t n, uint8_t *d_out, size_t out_cap,
                                          const ssb_target *targets, size_t n_targets, unsigned seed,
                                          ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes)
{
    if (!sp || (!d_sam && n) || (!d_out && n) || (n_targets && (!targets || !results)) || !stats || !out_bytes) return SSB_E_ARG;
    if (((uintptr_t)d_sam & 15) != 0) return SSB_E_ARG;
    ShardPlan pl;
    int rc = plan_from_shard(shard, xc, pl);
    if (rc) return rc;
    if (pl.halo_bytes > n) return SSB_E_ARG;
    rc = run_shard(sp, pl, d_sam, n, d_out, out_cap, targets, n_targets, seed, results, stats, out_bytes);
    if (rc && rc != SSB_E_PEER && pl.xc && pl.count > 1) pl.xc->abort_group();       // nobody may be left waiting for this shard
    return rc;
}

extern "C" int ssb_spike_run_device(ssb_spike *sp, const uint8_t *d_sam, size_t n, uint8_t *d_out, size_t out_cap,
                                    const ssb_target *targets, size_t n_targets, unsigned seed,
                                    ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes)
{
    return ssb_spike_run_shard_device(sp, NULL, NULL, d_sam, n, d_out, out_cap, targets, n_targets, seed, results, stats, out_bytes);
}

extern "C" int ssb_spike_run_shard_host(ssb_spike *sp, const ssb_spike_shard *shard, ssb_exchange *xc, const uint8_t *sam, size_t n, uint8_t *out, size_t out_cap,
                                        const ssb_target *targets, size_t n_targets, unsigned seed,
                                        ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes)
{
    if (!sp || (!sam && n) || (!out && n) || !stats || !out_bytes) return SSB_E_ARG;
    ssb_ctx *ctx = sp->ctx;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    uint8_t *d_in = NULL, *d_out = NULL;
    struct Bufs { uint8_t **a, **b; cudaStream_t s; ~Bufs() { if (*a) cudaFreeAsync(*a, s); if (*b) cudaFreeAsync(*b, s); cudaStreamSynchronize(s); } } bufs{&d_in, &d_out, ctx->stream};
    SSB_CUDA(ctx, cudaMallocAsync((void **)&d_in, n + 64, ctx->stream));
    SSB_CUDA(ctx, cudaMallocAsync((void **)&d_out, n + 64, ctx->stream));
    if (n) SSB_CUDA(ctx, cudaMemcpyAsync(d_in, sam, n, cudaMemcpyHostToDevice, ctx->stream));
    int rc = ssb_spike_run_shard_device(sp, shard, xc, d_in, n, d_out, n + 1, targets, n_targets, seed, results, stats, out_bytes);
    if (rc == SSB_OK) {
        if (*out_bytes > out_cap) { snprintf(ctx->err, sizeof ctx->err, "spike: output needs %zu bytes, capacity %zu", *out_bytes, out_cap); rc = SSB_E_ARG; }
        else if (*out_bytes) {
            cudaError_t e = cudaMemcpyAsync(out, d_out, *out_bytes, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) { snprintf(ctx->err, sizeof ctx->err, "spike: copy back: %s", cudaGetErrorString(e)); rc = SSB_E_CUDA; }
        }
    }
    return rc;
}

namespace {
// A host-resident body of any size on ONE device, in bounded device memory: the body is cut into coordinate shards of about
// `piece` bytes that are processed one after the other, each from the exact state its predecessor left (rand() offset, targets
// consumed, covered-locus count, spiked bases of straddling reads) -- so no windows of candidate offsets are needed -- while the
// host link works in both directions: H2D of shard i+1, i+2 || compute of shard i || D2H of shard i-1's output.
//   staging[3]  H2D targets (own lines of a shard)
//   work[2]     [lines of the previous shard that reach into this one][own lines], start 16-byte aligned
//   obuf[2]     output lines of a shard until they have gone back
int run_stream_host(ssb_spike *sp, const uint8_t *sam, size_t n, uint8_t *out, size_t out_cap, const ssb_target *targets, size_t T, unsigned seed,
                    ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes, size_t piece)
{
    ssb_ctx *ctx = sp->ctx;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    memset(stats, 0, sizeof *stats);
    *out_bytes = 0;
    int count = (int)((n + piece - 1) / piece);
    std::vector<ssb_spike_shard> plan((size_t)count); std::vector<size_t> off((size_t)count), len((size_t)count);
    std::vector<const char *> nm; for (const std::string &x : sp->names) nm.push_back(x.c_str());
    count = ssb_spike_plan_shards(sam, n, nm.data(), (int)nm.size(), count, 0, plan.data(), off.data(), len.data());
    if (count < 1) return SSB_E_ARG;
    size_t slot = 0; for (int i = 0; i < count; i++) if (len[i] > slot) slot = len[i];
    slot = (slot + 255) & ~(size_t)255;
    const size_t halo_cap = (size_t)64 << 20;
    cudaStream_t sc = ctx->stream, sIn = ctx->copy_stream;
    const double t_alloc = now_ms();
    if (!sp->st_out) SSB_CUDA(ctx, cudaStreamCreateWithFlags(&sp->st_out, cudaStreamNonBlocking));
    cudaStream_t sOut = sp->st_out;
    if (slot > sp->st_slot) {
        SSB_CUDA(ctx, cudaStreamSynchronize(sc)); SSB_CUDA(ctx, cudaStreamSynchronize(sIn)); SSB_CUDA(ctx, cudaStreamSynchronize(sOut));
        for (int i = 0; i < 3; i++) { if (sp->st_staging[i]) cudaFree(sp->st_staging[i]); sp->st_staging[i] = NULL; }
        for (int i = 0; i < 2; i++) { if (sp->st_work[i]) cudaFree(sp->st_work[i]); if (sp->st_obuf[i]) cudaFree(sp->st_obuf[i]); sp->st_work[i] = sp->st_obuf[i] = NULL; }
        sp->st_slot = 0;
        for (int i = 0; i < 3; i++) SSB_CUDA(ctx, cudaMalloc(&sp->st_staging[i], slot + 256));
        for (int i = 0; i < 2; i++) { SSB_CUDA(ctx, cudaMalloc(&sp->st_work[i], slot + halo_cap + 512)); SSB_CUDA(ctx, cudaMalloc(&sp->st_obuf[i], slot + halo_cap + 512)); }
        sp->st_slot = slot;
    }
    slot = sp->st_slot;
    uint8_t **staging = sp->st_staging, **work = sp->st_work, **obuf = sp->st_obuf;
    while (sp->st_ev.size() < (size_t)count * 4) { cudaEvent_t e = NULL; SSB_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); sp->st_ev.push_back(e); }
    cudaEvent_t *ev_in = sp->st_ev.data(), *ev_free = ev_in + count, *ev_done = ev_in + 2 * count, *ev_out = ev_in + 3 * count;
    // whatever happens, nothing of this run may still be in flight when the caller gets its buffers back
    struct Quiesce { cudaStream_t a, b, c; ~Quiesce() { cudaStreamSynchronize(a); cudaStreamSynchronize(b); cudaStreamSynchronize(c); } } quiesce{sc, sIn, sOut};
    if (getenv("SSB_CHAIN_DEBUG")) fprintf(stderr, "[stream] buffers and events: %.3f ms\n", now_ms() - t_alloc);
    auto copy_in = [&](int j) -> int {              // own lines of shard j -> staging[j % 3] (once the slot's previous tenant has been consumed)
        if (j >= count) return SSB_OK;
        if (j >= 3) SSB_CUDA(ctx, cudaStreamWaitEvent(sIn, ev_free[j - 3], 0));
        if (len[j]) SSB_CUDA(ctx, cudaMemcpyAsync(staging[j % 3], sam + off[j], len[j], cudaMemcpyHostToDevice, sIn));
        SSB_CUDA(ctx, cudaEventRecord(ev_in[j], sIn));
        return SSB_OK;
    };
    int rc;
    const bool dbg = getenv("SSB_CHAIN_DEBUG") != NULL;
    const double t_setup = now_ms();
    for (int j = 0; j < 3; j++) if ((rc = copy_in(j))) return rc;
    if (dbg) fprintf(stderr, "[stream] %d pieces, slot %zu bytes; first copies queued at %.3f ms\n", count, slot, now_ms() - t_setup);
    SeqState st;
    std::vector<ssb_target_result> res_tmp(T ? T : 1);
    for (size_t t = 0; t < T; t++) { memset(&results[t], 0, sizeof results[t]); results[t].status = SSB_T_ELSEWHERE; }
    for (auto &c : sp->se_chunks) if (c.first) cudaFree(c.first);
    sp->se_chunks.clear(); sp->se_chunked = true;
    size_t out_off = 0, prev_n = 0, n_se_total = 0; uint8_t *prev_body = NULL;
    const double t0 = now_ms();
    for (int i = 0; i < count; i++) {
        const double t_piece = now_ms();
        // ---- compose the body: the tail of the previous body that reaches into this shard, then the own lines
        size_t halo = 0;
        if (i > 0 && st.first_strad != ~0ull) {
            if (st.first_strad > prev_n) return SSB_E_STATE;
            halo = prev_n - (size_t)st.first_strad;
            if (halo > halo_cap) { snprintf(ctx->err, sizeof ctx->err, "spike: %zu bytes of alignment lines reach from one piece of the stream into the next (limit %zu)", halo, halo_cap); return SSB_E_SHARD; }
        }
        uint8_t *body = work[i & 1];                                          // 16-byte aligned start (cudaMalloc); the halo goes to the very front
        if (halo) SSB_LAUNCH(ctx, copy_bytes_kernel, ctx->sm_count * 2, 256, 0, sc, (const uint8_t *)(prev_body + st.first_strad), body, halo);
        SSB_CUDA(ctx, cudaStreamWaitEvent(sc, ev_in[i], 0));
        if (len[i]) SSB_LAUNCH(ctx, copy_bytes_kernel, ctx->sm_count * 8, 256, 0, sc, (const uint8_t *)staging[i % 3], body + halo, len[i]);
        SSB_CUDA(ctx, cudaEventRecord(ev_free[i], sc));
        if ((rc = copy_in(i + 3))) return rc;
        const size_t nb = halo + len[i];
        // ---- the output buffer must have gone back before it is written again
        if (i >= 2) SSB_CUDA(ctx, cudaStreamWaitEvent(sc, ev_out[i - 2], 0));
        ShardPlan pl;
        pl.index = i; pl.count = count; pl.seq = &st; pl.last = i == count - 1; pl.halo_bytes = halo;
        pl.rg.lo = i == 0 ? 0ull : (((unsigned long long)(uint32_t)plan[i].lo_tid << 32) | (unsigned long long)plan[i].lo_pos);
        pl.rg.hi = i == count - 1 ? ~0ull : (((unsigned long long)(uint32_t)plan[i].hi_tid << 32) | (unsigned long long)plan[i].hi_pos);
        ssb_spike_stats s1; size_t ob = 0;
        const double t_run = now_ms();
        if ((rc = run_shard(sp, pl, body, nb, obuf[i & 1], slot + halo_cap + 256, targets, T, seed, res_tmp.data(), &s1, &ob))) return rc;
        const double t_ran = now_ms();
        SSB_CUDA(ctx, cudaEventRecord(ev_done[i], sc));
        // ---- output lines back to the host while the next shard is at work
        if (out_off + ob > out_cap) { snprintf(ctx->err, sizeof ctx->err, "spike: output needs more than %zu bytes", out_cap); return SSB_E_ARG; }
        SSB_CUDA(ctx, cudaStreamWaitEvent(sOut, ev_done[i], 0));
        if (ob) SSB_CUDA(ctx, cudaMemcpyAsync(out + out_off, obuf[i & 1], ob, cudaMemcpyDeviceToHost, sOut));
        SSB_CUDA(ctx, cudaEventRecord(ev_out[i], sOut));
        out_off += ob;
        // ---- results of this shard
        for (size_t t = 0; t < T; t++) if (res_tmp[t].status != SSB_T_ELSEWHERE) results[t] = res_tmp[t];
        if (sp->n_se) { sp->se_chunks.push_back(std::make_pair(sp->d_se, sp->n_se)); n_se_total += sp->n_se; sp->d_se = NULL; sp->n_se = 0; }      // stays on the device until asked for
        stats->alignmentCount += s1.alignmentCount; stats->numberOfLociCovered += s1.numberOfLociCovered; stats->totalFoldCoverage += s1.totalFoldCoverage;
        if (s1.maxDepth > stats->maxDepth) stats->maxDepth = s1.maxDepth;
        stats->n_lines += s1.n_lines - 0; stats->n_kept += s1.n_kept; stats->n_runs += s1.n_runs; stats->n_hits += s1.n_hits;
        stats->ms_parse += s1.ms_parse; stats->ms_sort += s1.ms_sort; stats->ms_emit += s1.ms_emit; stats->ms_cover += s1.ms_cover; stats->ms_gather += s1.ms_gather;
        stats->ms_rng += s1.ms_rng; stats->ms_chain += s1.ms_chain; stats->ms_patch += s1.ms_patch; stats->ms_phase1 += s1.ms_phase1; stats->ms_tally += s1.ms_tally;
        if (s1.chain_mode > stats->chain_mode) stats->chain_mode = s1.chain_mode;
        stats->rng_k_out = s1.rng_k_out; stats->rng_draws = s1.rng_draws;
        prev_body = body; prev_n = nb;
        if (dbg) fprintf(stderr, "[stream] piece %d: queued %.3f ms, run %.3f ms, after %.3f ms (halo %zu bytes, out %zu)\n", i, t_run - t_piece, t_ran - t_run, now_ms() - t_ran, halo, ob);
    }
    const double t_loop = now_ms();
    SSB_CUDA(ctx, cudaStreamSynchronize(sOut));
    SSB_CUDA(ctx, cudaStreamSynchronize(sc));
    if (dbg) fprintf(stderr, "[stream] loop %.3f ms, drain %.3f ms, setup before the loop %.3f ms\n", t_loop - t0, now_ms() - t_loop, t0 - t_setup);
    sp->n_se = n_se_total;
    stats->in_bytes = (int64_t)n; stats->out_bytes = (int64_t)out_off;
    stats->n_forwarded = count;                     // pieces the body was streamed in
    stats->ms_total = (float)(now_ms() - t0);
    *out_bytes = out_off;
    return SSB_OK;
}
} // namespace

extern "C" int ssb_spike_run_host(ssb_spike *sp, const uint8_t *sam, size_t n, uint8_t *out, size_t out_cap,
                                  const ssb_target *targets, size_t n_targets, unsigned seed,
                                  ssb_target_result *results, ssb_spike_stats *stats, size_t *out_bytes)
{
    if (!sp || (!sam && n) || (!out && n) || (n_targets && (!targets || !results)) || !stats || !out_bytes) return SSB_E_ARG;
    // large bodies are streamed through the device in coordinate pieces (bounded device memory, both directions of the host link busy)
    size_t piece = (size_t)1 << 30;
    if (const char *e = getenv("SSB_STREAM_BYTES")) { const size_t v = strtoull(e, NULL, 10); if (v >= 4096) piece = v; }
    if (n > piece + piece / 2 && !getenv("SSB_NO_STREAM"))
        return run_stream_host(sp, sam, n, out, out_cap, targets, n_targets, seed, results, stats, out_bytes, piece);
    return ssb_spike_run_shard_host(sp, NULL, NULL, sam, n, out, out_cap, targets, n_targets, seed, results, stats, out_bytes);
}

// Host helper: cut a coordinate-sorted SAM body into shards of about equal bytes (see ssb200.h).
extern "C" int ssb_spike_plan_shards(const uint8_t *sam, size_t n, const char *const *contig_names, int n_contigs, int count, int64_t halo_bases,
                                     ssb_spike_shard *shards, size_t *body_off, size_t *body_len)
{
    if ((!sam && n) || count < 1 || !shards || !body_off || !body_len || halo_bases < 0 || (n_contigs && !contig_names)) return SSB_E_ARG;
    auto line_start = [&](size_t p) -> size_t {                 // start of the first line that begins at or after p
        if (p == 0) return 0;
        const void *nl = memchr(sam + p - 1, '\n', n - (p - 1));
        return nl ? (size_t)((const uint8_t *)nl - sam) + 1 : n;
    };
    auto prev_line = [&](size_t p) -> size_t {                  // start of the line before the one starting at p
        if (p == 0) return 0;
        size_t q = p - 1;                                       // the newline that ends it
        while (q > 0 && sam[q - 1] != '\n') q--;
        return q;
    };
    // (tid, pos) of the line starting at p; false when the line has no usable position (unmapped, malformed): such lines never cut
    auto key_of = [&](size_t p, int &tid, int64_t &pos) -> bool {
        size_t e = p; int field = 0; size_t f0 = p;
        size_t rn0 = 0, rn1 = 0, ps0 = 0, ps1 = 0;
        while (e < n && sam[e] != '\n') {
            if (sam[e] == '\t') {
                if (field == 2) { rn0 = f0; rn1 = e; }
                if (field == 3) { ps0 = f0; ps1 = e; break; }
                field++; f0 = e + 1;
            }
            e++;
        }
        if (ps1 == 0 || rn1 <= rn0) return false;
        tid = -1;
        for (int c = 0; c < n_contigs; c++) if (strlen(contig_names[c]) == rn1 - rn0 && !memcmp(contig_names[c], sam + rn0, rn1 - rn0)) { tid = c; break; }
        if (tid < 0) return false;
        int64_t v = 0;
        for (size_t i = ps0; i < ps1; i++) { if (sam[i] < '0' || sam[i] > '9') return false; v = v * 10 + (sam[i] - '0'); if (v > 0x7fffffffll) return false; }
        if (v < 1) return false;
        pos = v - 1;
        return true;
    };
    int made = 0;
    size_t own_start = 0;                                       // first byte of the current shard's own lines
    int lo_tid = 0; int64_t lo_pos = 0;
    for (int g = 0; g < count && own_start <= n; g++) {
        // where the next shard's own lines begin: the first line at or after the byte target whose key differs from its predecessor's
        size_t cut = n; int ct = 0x7fffffff; int64_t cp = 0;
        if (g + 1 < count) {
            size_t p = line_start(own_start + (n - own_start) / (size_t)(count - g));
            while (p < n) {
                int t1, t0; int64_t p1, p0;
                if (key_of(p, t1, p1)) {
                    // reads with the same (tid, pos) must stay together: walk back to the first line of that key
                    size_t q = p;
                    while (q > own_start) { const size_t r = prev_line(q); if (key_of(r, t0, p0) && t0 == t1 && p0 == p1) q = r; else break; }
                    if (q > own_start) { cut = q; ct = t1; cp = p1; break; }
                }
                p = line_start(p + 1);
            }
        }
        ssb_spike_shard &sh = shards[made];
        memset(&sh, 0, sizeof sh);
        sh.index = made; sh.lo_tid = lo_tid; sh.lo_pos = lo_pos; sh.hi_tid = cut < n ? ct : 0x7fffffff; sh.hi_pos = cut < n ? cp : 0;
        // halo: lines before own_start on the same contig that start within halo_bases of lo
        size_t h0 = own_start;
        if (made > 0 && halo_bases > 0) {
            while (h0 > 0) {
                const size_t r = prev_line(h0); int t0; int64_t p0;
                if (!key_of(r, t0, p0)) { h0 = r; continue; }                 // lines without a position ride along
                if (t0 != lo_tid || p0 + halo_bases <= lo_pos) break;
                h0 = r;
            }
        }
        sh.halo_bytes = own_start - h0;
        body_off[made] = h0; body_len[made] = cut - h0;
        made++;
        if (cut >= n) break;
        own_start = cut; lo_tid = ct; lo_pos = cp;
    }
    for (int g = 0; g < made; g++) shards[g].count = made;
    return made;
}

// rand() #k0 .. #k0+n-1 of srand(seed) (glibc TYPE_3), generated by the same kernel the spike path uses.
extern "C" int ssb_spike_rand(ssb_spike *sp, unsigned seed, uint64_t k0, size_t n, int32_t *out_host)
{
    if (!sp || (!out_host && n)) return SSB_E_ARG;
    if (!n) return SSB_OK;
    ssb_ctx *ctx = sp->ctx;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    Arena ar(s);
    const unsigned long long M = (n + RNG_BLOCK - 1) / RNG_BLOCK * RNG_BLOCK;
    const size_t nblocks = (size_t)(M / RNG_BLOCK);
    std::vector<uint32_t> bp(nblocks * GLIBC_DEG);
    uint32_t stepb[GLIBC_DEG], cur[GLIBC_DEG], tmpb[GLIBC_DEG];
    glibc_poly_xpow(RNG_BLOCK, stepb);
    glibc_poly_xpow(310 + k0, cur);
    for (size_t b = 0; b < nblocks; b++) { memcpy(&bp[b * GLIBC_DEG], cur, sizeof cur); glibc_poly_mulmod(cur, stepb, tmpb); memcpy(cur, tmpb, sizeof cur); }
    uint32_t seedw[61];
    glibc_seed_window(seed, seedw);
    uint32_t *d_bp = ar.get<uint32_t>(bp.size()), *d_seedw = ar.get<uint32_t>(61); int32_t *R = ar.get<int32_t>(M);
    SPK_CHECK_ARENA(ar);
    SSB_CUDA(ctx, cudaMemcpyAsync(d_bp, bp.data(), bp.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    SSB_CUDA(ctx, cudaMemcpyAsync(d_seedw, seedw, sizeof seedw, cudaMemcpyHostToDevice, s));
    SSB_LAUNCH(ctx, rng_fill_kernel, (int)nblocks, RNG_TPB, 0, s, d_bp, sp->d_rng_tab, d_seedw, R, M, (uint32_t *)NULL, (uint32_t *)NULL, (uint32_t *)NULL);
    SSB_CUDA(ctx, cudaMemcpyAsync(out_host, R, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SSB_CUDA(ctx, cudaStreamSynchronize(s));
    return SSB_OK;
}

extern "C" int ssb_spike_seq_error_count(ssb_spike *sp, size_t *count)
{
    if (!sp || !count) return SSB_E_ARG;
    *count = sp->n_se;
    return SSB_OK;
}

extern "C" int ssb_spike_seq_errors(ssb_spike *sp, ssb_seq_error *dst, size_t cap)
{
    if (!sp || (!dst && cap)) return SSB_E_ARG;
    ssb_ctx *ctx = sp->ctx;
    size_t n = sp->n_se < cap ? sp->n_se : cap;
    if (sp->se_chunked) {
        SSB_CUDA(ctx, cudaSetDevice(ctx->device));
        size_t k = 0;
        for (auto &c : sp->se_chunks) {
            if (k >= n) break;
            const size_t m = c.second < n - k ? c.second : n - k;
            SSB_CUDA(ctx, cudaMemcpyAsync(dst + k, c.first, m * sizeof(ssb_seq_error), cudaMemcpyDeviceToHost, ctx->stream));
            k += m;
        }
        SSB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return SSB_OK;
    }
    if (n) {
        SSB_CUDA(ctx, cudaSetDevice(ctx->device));
        SSB_CUDA(ctx, cudaMemcpyAsync(dst, sp->d_se, n * sizeof(ssb_seq_error), cudaMemcpyDeviceToHost, ctx->stream));
        SSB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SSB_OK;
}

// test hook (host only): the optional-field check of the tokeniser on one TAG:TYPE:VALUE text
namespace { struct HostBytes { const char *p; __host__ __device__ uint8_t operator()(size_t i) const { return (uint8_t)p[i]; } }; }
extern "C" int ssb_test_aux_ok(const char *field, size_t n)
{
    const HostBytes at{field};
    const int rc = samparse::aux_ok_t(at, (size_t)0, n);
    return rc == samparse::AUX_FLOAT ? samparse::aux_float_ok_t(at, (size_t)0, n) : rc;
}
