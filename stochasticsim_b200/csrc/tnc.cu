// tnc.cu -- trinucleotide-context scan on B200 (hot path 2).
//
// Replaces the getline / 3-byte-window loop of tncCountsProfile.c:391-447 and the 64-way
// strncmp chain incCtx (tncCountsProfile.c:105-363).  Results are bit-exact with the
// reference, including its three quirks (SURVEY.md D11 / App. B):
//   * a record is KEPT unless empty, starting with '>' or free of upper-case G/C/A/T
//     (tncCountsProfile.c:398-407); non-kept records are invisible, contigs are joined;
//   * every window of three upper-case bases inside a kept record counts (:430-438);
//   * between two kept records exactly ONE straddling window (last(l), l'[0], l'[1]) counts,
//     the other one is lost to the newline slot (:409, :441-443).
//
// Decomposition (one streaming pass over the bytes, no inter-block dependency):
//   total = sum over byte positions p of
//             [b[p-2],b[p-1],b[p] upper-case bases]                         (in-line window)
//           + [b[p-2]=='\n', b[p-3],b[p-1],b[p] upper-case bases]           (straddle, optimistic)
//           - corrections at the (rare) places where the optimistic rule is wrong.
// The optimistic rule is wrong only around header records and where the record before a line
// start does not end in an upper-case base.  tnc_scan_kernel appends those positions to an
// exception list; tnc_fixup_kernel resolves each one exactly by walking back to the nearest kept
// record (one warp per exception).  In a 60-column genome FASTA that is a few thousand
// exceptions per 3 GB.
//
// tnc_scan_kernel: every thread takes 16 bytes per step.  A chunk whose bytes (and 2-byte halo) are all one of A C G T '\n' --
// checked exactly with one PRMT table lookup per word -- takes the fast path: bytes -> 3-bit symbols, the 4-mers at every second
// position -> base-6 bin by one dp4a -> a 1296-bin shared-memory histogram (8 shared atomics per 16 bytes), folded into the 64
// contexts once per block.  Anything else (N, lower case, '>', '\r', ragged end) takes the generic per-position path.  Newline
// positions are queued per warp and handled 32 at a time.  The per-segment "no upper-case base" counters that let the fix-up
// kernel jump over N blocks count 16-byte chunks (256 per 4 KiB segment).
#include "common.cuh"
#include <stdlib.h>
#include <type_traits>
#include <vector>

namespace {

constexpr int      TNC_BLOCK = 256;
constexpr int      TNC_BPT   = 16;            // bytes per thread per iteration
constexpr uint32_t EXC_HEADER = 0x80000000u;  // exception kind flag (positions stay < 2^31)
constexpr size_t   TNC_MAX_PIECE = (size_t)1 << 30;
// A piece this small can never overflow the exception list: at most one record per 2 bytes
// ("\n>" headers) = 65536 < tnc_exc_cap(131072) = 8192 + 65536.
constexpr size_t   TNC_SAFE_PIECE = (size_t)1 << 17;
constexpr int      TNC_SEG_SHIFT = 12;            // 4 KiB segments = 256 chunks of 16 bytes

struct TncDevState {                          // mirrors ssb_tnc_carry
    uint8_t started, prev[3], carry, frag_nonempty, frag_first, frag_has_base;
};
static_assert(sizeof(TncDevState) == sizeof(ssb_tnc_carry), "state layout");

__host__ __device__ inline bool is_base(uint8_t c) { const uint32_t d = (uint32_t)c - 0x41u; return d < 20u && ((0x80045u >> d) & 1u); }   // A C G T = 0x41 + {0, 2, 6, 19}
// reference index order A<C<G<T (tncCountsProfile.c:14-77)
__host__ __device__ inline int ref_code(uint8_t c) { const uint32_t s = ((uint32_t)c >> 1) & 3u; return (int)(s ^ (s >> 1)); }            // (c one of A C G T) bits 2..1: A 0, C 1, T 2, G 3

// ---- scan kernel ------------------------------------------------------------------------------
// Every thread takes 16 bytes per iteration.  Fast path (all bytes of the chunk and of its 2-byte halo are one of
// A C G T '\n', verified exactly with one PRMT table lookup per word): bytes become 3-bit symbols ((b >> 1) & 7:
// A 0, C 1, T 2, G 3, '\n' 5), and the 4-mers that start at every second position are binned base 6 (one integer dot
// product) into a 1296-bin shared-memory histogram -- one shared atomic per two windows.  When the block is done the histogram is
// folded: bin (s0,s1,s2,s3) feeds window (s0,s1,s2) and window (s1,s2,s3) when their symbols are bases.
// Anything else in a chunk (N, lower case, '>', '\r', the ragged end of the piece) takes the generic path, which
// looks at every position.  Newlines are not handled where they are found (that would make every warp execute the
// rare code for a few lanes): their positions go into a per-warp queue that is drained 32 at a time, one newline
// per lane: the straddling window (b[q-1], b[q+1], b[q+2]) is counted if its carry byte is a base, otherwise it
// becomes an exception for tnc_fixup_kernel; a '>' behind the newline becomes a header exception.
constexpr int TNC_WARPS = TNC_BLOCK / 32;
constexpr int TNC_SUB = 4;                        // 16-byte chunks per thread and warp iteration
constexpr int NLQ_CAP = 128;                      // >= 31 left over + 32 lanes * up to 2 newlines in 16 bytes... drained when >= 32

__device__ __forceinline__ uint32_t zero_bytes_mask(uint32_t d) { return ~(((d & 0x7f7f7f7fu) + 0x7f7f7f7fu) | d | 0x7f7f7f7fu); }

// Symbols: s = (byte >> 1) & 7 is distinct for the five bytes that matter -- A 0, C 1, T 2, G 3, '\n' 5 -- so it serves both as
// the 3-bit symbol and as the key of the exactness check: a byte is one of the five iff it equals TABLE[s].
__device__ __forceinline__ uint32_t symbols(uint32_t w) { return (w >> 1) & 0x07070707u; }
// non-zero iff some byte of w is not one of A C G T '\n' (sy = symbols(w))
__device__ __forceinline__ uint32_t not_acgtnl(uint32_t w, uint32_t sy)
{
    const uint32_t TLO = 0x47544341u, THI = 0x01010A01u;      // key 0->'A' 1->'C' 2->'T' 3->'G' | 4->01 5->'\n' 6->01 7->01
    const uint32_t e0 = __byte_perm(TLO, THI, sy), e1 = __byte_perm(TLO, THI, sy >> 16);
    return w ^ __byte_perm(e0, e1, 0x6420);
}
// bit k = the top bit of byte k (a byte flag mask as 4 bits)
__device__ __forceinline__ uint32_t msb4(uint32_t f) { return (((f >> 7) * 0x00204081u) >> 21) & 0xFu; }
// reference codes (A 0, C 1, G 2, T 3) of the four bytes of x, one per byte (meaningful where the byte is an upper-case base)
__device__ __forceinline__ uint32_t ref_codes4(uint32_t x) { const uint32_t sy = (x >> 1) & 0x03030303u; return sy ^ ((sy >> 1) & 0x01010101u); }
// per byte of (prev, cur) codes: the index 16 r[i-2] + 4 r[i-1] + r[i] of the window that ends at byte i of cur
__device__ __forceinline__ uint32_t win_index4(uint32_t prev, uint32_t cur) { return cur + 4u * __funnelshift_r(prev, cur, 24) + 16u * __funnelshift_r(prev, cur, 16); }
// 0x80 in every byte of w that is an upper-case A C G T
__device__ __forceinline__ uint32_t base_flags(uint32_t w) { return zero_bytes_mask(not_acgtnl(w, symbols(w))) & (w << 1); }
// four symbols [a,b,c,d] (one per byte, each 0..5) -> base-6 bin a + 6b + 36c + 216d: one integer dot product
__device__ __forceinline__ uint32_t pack4(uint32_t z) { return __dp4a(z, 0xD8240601u, 0u); }
constexpr int TNC_BINS = 1296;

__device__ __forceinline__ uint32_t ld_word(const uint8_t *b, size_t n, size_t off)
{
    // aligned 4-byte load with zero fill past the end (0x00 is "other")
    if (off + 4 <= n) return *reinterpret_cast<const uint32_t *>(b + off);
    uint32_t w = 0;
    for (int k = 0; k < 4; k++) if (off + k < n) w |= (uint32_t)b[off + k] << (8 * k);
    return w;
}

// one newline per lane: q = its position (q < n), or -1 / -2 for a newline that closes the 3-byte halo of the piece
__device__ __forceinline__ void handle_newline(const uint8_t *__restrict__ b, long n, const TncDevState &st, long q, uint32_t *hist3,
                                               uint32_t *__restrict__ exc_count, uint32_t *__restrict__ exc, uint32_t exc_cap)
{
    auto at = [&](long i) -> uint8_t { return i >= 0 ? b[i] : st.prev[3 + i]; };
    auto push = [&](uint32_t rec) { uint32_t slot = atomicAdd(exc_count, 1u); if (slot < exc_cap) exc[slot] = rec; };
    if (q + 1 >= 0 && q + 1 < n && b[q + 1] == '>') push((uint32_t)(q + 1) | EXC_HEADER);        // a header record starts here
    const long p = q + 2;
    if (p >= n) return;
    const uint8_t c1 = at(q + 1), c2 = b[p];
    if (!is_base(c1) || !is_base(c2)) return;
    // the straddling window needs the last byte of the record before the newline; when that byte is not a base, or lies
    // before this piece, the fix-up kernel finds the real carry
    if (q >= 1 && is_base(b[q - 1])) atomicAdd(&hist3[16 * ref_code(b[q - 1]) + 4 * ref_code(c1) + ref_code(c2)], 1u);
    else push((uint32_t)p);
}

__global__ void __launch_bounds__(TNC_BLOCK)
tnc_scan_kernel(const uint8_t *__restrict__ b, size_t n, const TncDevState *__restrict__ st_in, const uint8_t *__restrict__ prev3,
                unsigned long long *__restrict__ counts, uint32_t *__restrict__ exc_count,
                uint32_t *__restrict__ exc, uint32_t exc_cap, uint32_t *__restrict__ seg_nobase)
{
    __shared__ uint32_t hist4[TNC_BINS];
    __shared__ uint32_t hist3[64];
    __shared__ uint32_t nlq[TNC_WARPS][NLQ_CAP];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < TNC_BINS; i += TNC_BLOCK) hist4[i] = 0;
    if (threadIdx.x < 64) hist3[threadIdx.x] = 0;
    __syncthreads();
    // The scan needs only the three bytes in front of the piece from the state; for a piece behind another one in the same buffer they are
    // read from there (prev3), so that it need not wait for the previous piece's fix-up kernel, which is what writes the state.
    TncDevState st;
    if (prev3) { st.started = 1; st.prev[0] = prev3[0]; st.prev[1] = prev3[1]; st.prev[2] = prev3[2]; st.carry = 0; st.frag_nonempty = 0; st.frag_first = 0; st.frag_has_base = 0; }
    else st = *st_in;
    if (!st.started) { st.prev[0] = st.prev[1] = st.prev[2] = '\n'; }                 // start of file behaves like "\n\n\n"
    uint32_t qn = 0;                                                                   // entries in this warp's newline queue (warp uniform)
    uint32_t *q = nlq[wid];

    const size_t n_chunks = (n + TNC_BPT - 1) / TNC_BPT;
    // a warp iteration covers TNC_SUB * 32 consecutive chunks (lane l takes chunks l, l+32, ...): the loop overhead and the
    // newline queue are paid once per 2 KiB.  All lanes of a warp run the same number of iterations (the queue is warp collective).
    const size_t stride = ((size_t)gridDim.x * blockDim.x) * TNC_SUB;
    const size_t warp_first = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) - lane) * TNC_SUB;
    for (size_t cbase = warp_first; cbase < n_chunks; cbase += stride) {
      unsigned long long nl64 = 0;                                                     // bit 16*sub + i: byte i of sub-chunk `sub` is '\n'
      // a warp step whose 128 chunks are all whole and have their halo inside the piece runs without the edge tests (INTERIOR)
      auto warp_step = [&](auto interior_tag) {
      constexpr bool INTERIOR = decltype(interior_tag)::value;
#pragma unroll 1
      for (int sub = 0; sub < TNC_SUB; sub++) {
        const size_t chunk = cbase + (size_t)sub * 32 + lane;
        uint32_t nlmask = 0; bool nobase = false;
        const size_t p0 = chunk * TNC_BPT;
        if (INTERIOR || chunk < n_chunks) {
            uint32_t w[4];
            if (INTERIOR || p0 + TNC_BPT <= n) {
                const uint4 v = *reinterpret_cast<const uint4 *>(b + p0);
                w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) w[j] = ld_word(b, n, p0 + 4 * j);
            }
            uint32_t hw;                                                               // the 4 bytes before the chunk
            if (INTERIOR || p0) hw = *reinterpret_cast<const uint32_t *>(b + p0 - 4);
            else hw = (uint32_t)st.prev[0] << 8 | (uint32_t)st.prev[1] << 16 | (uint32_t)st.prev[2] << 24;
            const uint32_t s0 = symbols(w[0]), s1 = symbols(w[1]), s2 = symbols(w[2]), s3 = symbols(w[3]), sh = symbols(hw);
            const uint32_t bad = not_acgtnl(w[0], s0) | not_acgtnl(w[1], s1) | not_acgtnl(w[2], s2) | not_acgtnl(w[3], s3) | (not_acgtnl(hw, sh) & 0xFFFF0000u);
            if (bad == 0u && (INTERIOR || p0 + TNC_BPT <= n)) {
                // ---- fast path ----
                atomicAdd(&hist4[pack4(__funnelshift_r(sh, s0, 16))], 1u);       // windows ending at 0, 1
                atomicAdd(&hist4[pack4(s0)], 1u);                                // windows ending at 2, 3
                atomicAdd(&hist4[pack4(__funnelshift_r(s0, s1, 16))], 1u);
                atomicAdd(&hist4[pack4(s1)], 1u);
                atomicAdd(&hist4[pack4(__funnelshift_r(s1, s2, 16))], 1u);
                atomicAdd(&hist4[pack4(s2)], 1u);
                atomicAdd(&hist4[pack4(__funnelshift_r(s2, s3, 16))], 1u);
                atomicAdd(&hist4[pack4(s3)], 1u);
                const uint32_t f0 = s0 & 0x04040404u, f1 = s1 & 0x04040404u, f2 = s2 & 0x04040404u, f3 = s3 & 0x04040404u;   // symbol 5 = newline
                if (f0 | f1 | f2 | f3) {                                             // a newline in these 16 bytes (one chunk in four)
                    nlmask = ((((f0 >> 2) * 0x00204081u) >> 21) & 0xFu) | (((((f1 >> 2) * 0x00204081u) >> 21) & 0xFu) << 4) |
                             (((((f2 >> 2) * 0x00204081u) >> 21) & 0xFu) << 8) | (((((f3 >> 2) * 0x00204081u) >> 21) & 0xFu) << 12);
                }
            } else {
                // ---- generic path: exact flags per byte, windows from SWAR codes ----
                // upper-case base flags (bit 7 per byte) and newline flags of the four words, exactly
                uint32_t bf[4], nf[4], anyb = 0, anyn = 0;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const uint32_t z = zero_bytes_mask(not_acgtnl(w[j], symbols(w[j])));   // 0x80 where the byte is A C G T or newline
                    bf[j] = z & (w[j] << 1);                                        // bit 6 set: a base
                    nf[j] = z & ~(w[j] << 1);
                    anyb |= bf[j]; anyn |= nf[j];
                }
                if (anyn) {
#pragma unroll
                    for (int j = 0; j < 4; j++) nlmask |= msb4(nf[j]) << (4 * j);
                    if (!INTERIOR && p0 + TNC_BPT > n) nlmask &= (1u << (n - p0)) - 1u;
                }
                if (!anyb) nobase = true;
                else {
                    // base flags of positions -2 .. 15 as a bit mask (bit i+2 <-> position i); a window ends where three in a row are set
                    const uint32_t hz = base_flags(hw);
                    uint32_t bm = msb4(hz) >> 2;                                                      // positions -2, -1 -> bits 0, 1
#pragma unroll
                    for (int j = 0; j < 4; j++) bm |= msb4(bf[j]) << (2 + 4 * j);
                    uint32_t win = bm & (bm >> 1) & (bm >> 2);                                        // bit i: window ending at position i
                    if (!INTERIOR && p0 + TNC_BPT > n) win &= (1u << (n - p0)) - 1u;
                    if (win) {
                        // reference codes (A 0, C 1, G 2, T 3) of every byte, then per byte the index 16 r[i-2] + 4 r[i-1] + r[i] of the window that ends there
                        const uint32_t rh = ref_codes4(hw), r0 = ref_codes4(w[0]), r1 = ref_codes4(w[1]), r2 = ref_codes4(w[2]), r3 = ref_codes4(w[3]);
                        const uint32_t xw[4] = {win_index4(rh, r0), win_index4(r0, r1), win_index4(r1, r2), win_index4(r2, r3)};
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            uint32_t wj = (win >> (4 * j)) & 0xFu;
                            while (wj) { const int k = __ffs(wj) - 1; wj &= wj - 1; atomicAdd(&hist3[(xw[j] >> (8 * k)) & 63u], 1u); }
                        }
                    }
                }
            }
            if (!INTERIOR && chunk == 0) {
                // newlines that close the halo of the piece (positions -2 and -1) are handled right here
                if (st.prev[1] == '\n') handle_newline(b, (long)n, st, -2, hist3, exc_count, exc, exc_cap);
                if (st.prev[2] == '\n') handle_newline(b, (long)n, st, -1, hist3, exc_count, exc, exc_cap);
            }
        }
        {   // chunks without an upper-case base, counted per 4 KiB segment: the 32 chunks of a warp step lie in one segment -> one atomic
            const unsigned nb = __ballot_sync(0xffffffffu, nobase);
            if (nb && lane == 0) atomicAdd(&seg_nobase[((cbase + (size_t)sub * 32) * TNC_BPT) >> TNC_SEG_SHIFT], (uint32_t)__popc(nb));
        }
        nl64 |= (unsigned long long)nlmask << (16 * sub);
      }
      };
      if (cbase > 0 && (cbase + (size_t)TNC_SUB * 32) * TNC_BPT <= n) warp_step(std::true_type{}); else warp_step(std::false_type{});
        // ---- queue the newline positions of this warp iteration, drain 32 at a time ----
        const unsigned has_nl = __ballot_sync(0xffffffffu, nl64 != 0ull);
        if (has_nl) {
            const uint32_t cnt = __popcll(nl64);
            auto pos_of = [&](int bit) -> size_t { return (cbase + (size_t)(bit >> 4) * 32 + lane) * TNC_BPT + (bit & 15); };
            uint32_t incl, total;
            if (__ballot_sync(0xffffffffu, cnt > 1u) == 0u) {                       // the usual case: at most one newline per lane
                incl = __popc(has_nl & (0xffffffffu >> (31 - lane))); total = __popc(has_nl);
            } else {
                incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
                total = __shfl_sync(0xffffffffu, incl, 31);
            }
            if (qn + total <= NLQ_CAP) {
                uint32_t slot = qn + incl - cnt; unsigned long long m = nl64;
                while (m) { const int bit = __ffsll((long long)m) - 1; m &= m - 1; q[slot++] = (uint32_t)pos_of(bit); }
                qn += total;
            } else {
                // (pathological: more than two newlines per 16 bytes across the warp) handle them in place
                unsigned long long m = nl64;
                while (__ballot_sync(0xffffffffu, m != 0ull)) {
                    if (m) { const int bit = __ffsll((long long)m) - 1; m &= m - 1; handle_newline(b, (long)n, st, (long)pos_of(bit), hist3, exc_count, exc, exc_cap); }
                }
            }
            __syncwarp();
            while (qn >= 32) {
                qn -= 32;
                handle_newline(b, (long)n, st, (long)q[qn + lane], hist3, exc_count, exc, exc_cap);
                __syncwarp();
            }
        }
    }
    __syncwarp();
    if ((uint32_t)lane < qn) handle_newline(b, (long)n, st, (long)q[lane], hist3, exc_count, exc, exc_cap);
    __syncthreads();
    // ---- fold the 4-mer histogram into the 64 contexts (reference index order A<C<G<T) ----
    for (int bin = threadIdx.x; bin < TNC_BINS; bin += TNC_BLOCK) {
        const uint32_t v = hist4[bin];
        if (!v) continue;
        const uint32_t s0 = bin % 6, s1 = (bin / 6) % 6, s2 = (bin / 36) % 6, s3 = bin / 216;
        // symbol -> reference code: A0 C1 T2 G3 -> A0 C1 G2 T3
        const uint32_t r0 = s0 ^ (s0 >> 1), r1 = s1 ^ (s1 >> 1), r2 = s2 ^ (s2 >> 1), r3 = s3 ^ (s3 >> 1);
        if (s0 < 4 && s1 < 4 && s2 < 4) atomicAdd(&hist3[16 * r0 + 4 * r1 + r2], v);
        if (s1 < 4 && s2 < 4 && s3 < 4) atomicAdd(&hist3[16 * r1 + 4 * r2 + r3], v);
    }
    __syncthreads();
    if (threadIdx.x < 64 && hist3[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)hist3[threadIdx.x]);
}

// ---- exception resolution ----------------------------------------------------------------
// All helpers below are called by a full warp with identical arguments.

__device__ __forceinline__ uint8_t byte_at(const uint8_t *b, const TncDevState &st, long i)
{
    return i >= 0 ? b[i] : st.prev[3 + i];       // i in [-3,-1] reads the bytes before the piece
}

// Looks backwards from index e-1 for the nearest '\n'.  a = its index + 1, or -1 when the
// record began before the piece.  has_base: an upper-case base lies in [max(a,0), e).
__device__ void scan_back(const uint8_t *b, long e, long &a, bool &has_base)
{
    const int lane = threadIdx.x & 31;
    has_base = false;
    long hi = e;
    a = -1;
    while (hi > 0) {
        long idx = hi - 1 - lane;
        uint8_t c = idx >= 0 ? b[idx] : (uint8_t)0xFF;
        unsigned m_nl = __ballot_sync(0xffffffffu, c == '\n');
        unsigned m_b  = __ballot_sync(0xffffffffu, is_base(c));
        if (m_nl) {
            int l = __ffs(m_nl) - 1;
            has_base |= (m_b & ((1u << l) - 1u)) != 0;
            a = hi - l;
            return;
        }
        has_base |= m_b != 0;
        hi -= 32;
    }
}

// Looks forwards from index q for the nearest '\n'; returns n when there is none.
__device__ long scan_fwd_newline(const uint8_t *b, long n, long q)
{
    const int lane = threadIdx.x & 31;
    for (long lo = q; lo < n; lo += 32) {
        long idx = lo + lane;
        unsigned m = __ballot_sync(0xffffffffu, idx < n && b[idx] == '\n');
        if (m) return lo + __ffs(m) - 1;
    }
    return n;
}

// Last byte of the nearest kept, newline-terminated record that ends before line start q
// (0 when there is none): the reference's 1-byte carry (tncCountsProfile.c:441-443).
// every 16-byte chunk of segment s is free of upper-case bases
__device__ __forceinline__ bool seg_free(const uint32_t *seg, long n, long s)
{
    const long left = n - (s << TNC_SEG_SHIFT);
    const uint32_t chunks = left >= (1L << TNC_SEG_SHIFT) ? (1u << (TNC_SEG_SHIFT - 4)) : (uint32_t)((left + 15) >> 4);
    return seg[s] == chunks;
}

__device__ uint8_t resolve_carry(const uint8_t *b, long n, const uint32_t *seg, const TncDevState &st, long q)
{
    long e = q - 1;                               // the newline that terminates the previous record
    for (;;) {
        if (e < 0) return st.carry;               // that newline lies before this piece
        // records that lie completely inside a base-free stretch cannot be kept: jump to the record that straddles its start
        if (seg && e >= (2L << TNC_SEG_SHIFT)) {
            long s = (e - 1) >> TNC_SEG_SHIFT;
            if (seg_free(seg, n, s) && seg_free(seg, n, s - 1)) {
                while (s > 0 && seg_free(seg, n, s - 1)) s--;
                const long z0 = s << TNC_SEG_SHIFT;
                const long f = scan_fwd_newline(b, n, z0);      // first newline inside the stretch (e itself at the latest)
                if (f < e) e = f;
            }
        }
        long a; bool hb;
        scan_back(b, e, a, hb);
        if (a >= 0) {
            if (e > a && b[a] != '>' && hb) return b[e - 1];
            e = a - 1;
        } else {
            bool nonempty = st.frag_nonempty || e > 0;
            uint8_t first = st.frag_nonempty ? st.frag_first : b[0];
            hb = hb || st.frag_has_base;
            uint8_t last = e > 0 ? b[e - 1] : st.prev[2];
            if (nonempty && first != '>' && hb) return last;
            return st.carry;
        }
    }
}

__device__ __forceinline__ void bump(unsigned long long *counts, uint8_t x, uint8_t y, uint8_t z, long long delta)
{
    atomicAdd(&counts[16 * ref_code(x) + 4 * ref_code(y) + ref_code(z)], (unsigned long long)delta);
}

// A header record occupies [q, f) (q may be -1: it began before the piece).  Undo what the scan
// counted optimistically inside and right after it.
__device__ void fix_header(const uint8_t *b, long n, const uint32_t *seg, const TncDevState &st, unsigned long long *counts, long q)
{
    const int lane = threadIdx.x & 31;
    long f = scan_fwd_newline(b, n, q < 0 ? 0 : q);
    // (1) windows inside the header were counted as in-line windows
    for (long lo = (q < 0 ? 0 : q); lo < f; lo += 32) {
        long i = lo + lane;
        if (i < f) {
            uint8_t c0 = byte_at(b, st, i - 2), c1 = byte_at(b, st, i - 1), c2 = b[i];
            if (is_base(c0) && is_base(c1) && is_base(c2)) bump(counts, c0, c1, c2, -1);
        }
    }
    // (2) the record after the header: the scan used the header's last byte as the carry
    if (f + 2 < n && f - 1 >= 0 && is_base(b[f - 1]) && is_base(b[f + 1]) && is_base(b[f + 2])) {
        uint8_t carry = resolve_carry(b, n, seg, st, f + 1);
        if (lane == 0) {
            bump(counts, b[f - 1], b[f + 1], b[f + 2], -1);
            if (is_base(carry)) bump(counts, carry, b[f + 1], b[f + 2], +1);
        }
    }
}

__global__ void __launch_bounds__(128)
tnc_fixup_kernel(const uint8_t *__restrict__ b, size_t n_, const TncDevState *__restrict__ st_in,
                 TncDevState *__restrict__ st_out, unsigned long long *__restrict__ counts,
                 const uint32_t *__restrict__ exc_count, uint32_t *__restrict__ ovf,
                 const uint32_t *__restrict__ exc, uint32_t exc_cap, const uint32_t *__restrict__ seg)
{
    const long n = (long)n_;
    TncDevState st = *st_in;
    if (!st.started) { st.prev[0] = st.prev[1] = st.prev[2] = '\n'; st.carry = 0; st.frag_nonempty = 0; st.frag_first = 0; st.frag_has_base = 0; }
    const int lane = threadIdx.x & 31;
    const long warps = ((long)gridDim.x * blockDim.x) >> 5;
    uint32_t nexc = *exc_count;
    if (nexc > exc_cap || *ovf) {                 // list overflowed: flag it, the host redoes the call in smaller pieces
        if (blockIdx.x == 0 && threadIdx.x == 0) *ovf = 1;
        return;
    }
    // tasks: [0, nexc) exceptions, nexc = implicit header at the start of the piece, nexc+1 = state out
    for (long task = (((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5); task < (long)nexc + 2; task += warps) {
        if (task < nexc) {
            uint32_t rec = exc[task];
            long p = (long)(rec & ~EXC_HEADER);
            if (rec & EXC_HEADER) fix_header(b, n, seg, st, counts, p);
            else {
                uint8_t carry = resolve_carry(b, n, seg, st, p - 1);
                if (lane == 0 && is_base(carry)) bump(counts, carry, byte_at(b, st, p - 1), b[p], +1);
            }
        } else if (task == nexc) {
            if (st.frag_nonempty && st.frag_first == '>') fix_header(b, n, seg, st, counts, -1);
        } else if (st_out) {
            long a; bool hb;
            scan_back(b, n, a, hb);
            TncDevState o;
            o.started = 1;
            if (a >= 0) {
                o.carry = resolve_carry(b, n, seg, st, a);
                o.frag_nonempty = n > a;
                o.frag_first = n > a ? b[a] : 0;
                o.frag_has_base = hb;
            } else {
                o.carry = st.carry;
                o.frag_nonempty = st.frag_nonempty || n > 0;
                o.frag_first = st.frag_nonempty ? st.frag_first : (n > 0 ? b[0] : 0);
                o.frag_has_base = st.frag_has_base || hb;
            }
            for (int k = 0; k < 3; k++) o.prev[k] = byte_at(b, st, n - 3 + k < -3 ? -3 : n - 3 + k);
            if (n < 3) {                           // fewer than 3 new bytes: slide the old ones
                uint8_t all[6] = {st.prev[0], st.prev[1], st.prev[2], 0, 0, 0};
                for (long k = 0; k < n; k++) all[3 + k] = b[k];
                for (int k = 0; k < 3; k++) o.prev[k] = all[n + k];
            }
            if (lane == 0) *st_out = o;
        }
    }
}

// reverse complement folding order of the reference's printf block (tncCountsProfile.c:452-483)
const char *const OUT_ORDER[32] = {
    "ACA","ACC","ACG","ACT","ATA","ATC","ATG","ATT","CCA","CCC","CCG","CCT","CTA","CTC","CTG","CTT",
    "GCA","GCC","GCG","GCT","GTA","GTC","GTG","GTT","TCA","TCC","TCG","TCT","TTA","TTC","TTG","TTT"};

// device scratch: scanner state (ping-pong), per-call accumulators, overflow flag, exception list
struct TncScratch {
    TncDevState        *st[2];
    uint32_t           *exc_count;
    uint32_t           *ovf;         // set by the fix-up kernel when the exception list overflowed
    unsigned long long *acc;         // 64 per-call accumulators
    uint32_t           *exc;
    uint32_t            exc_cap;
    uint32_t           *seg;         // per 4 KiB segment: number of 16-byte chunks without an upper-case base
    size_t              seg_words;
    uint32_t           *exc_count2, *exc2, *seg2;   // second set (device-resident runs: piece i+1 is scanned while piece i is fixed up); NULL otherwise
    uint8_t            *tail;        // first byte after the scratch arrays (256-byte aligned)
};

size_t tnc_exc_cap(size_t piece_bytes) { return piece_bytes / 16 + (1u << 16); }

int tnc_scratch(ssb_ctx *ctx, size_t piece_bytes, size_t extra_bytes, TncScratch *s, bool two_sets = false)
{
    size_t cap = tnc_exc_cap(piece_bytes);
    size_t seg_words = (piece_bytes >> TNC_SEG_SHIFT) + 2;
    size_t head = 1024 + cap * sizeof(uint32_t);
    head = (head + 255) & ~(size_t)255;
    const size_t seg_off = head;
    head += seg_words * sizeof(uint32_t);
    head = (head + 255) & ~(size_t)255;
    const size_t exc2_off = head;
    if (two_sets) { head += cap * sizeof(uint32_t); head = (head + 255) & ~(size_t)255; }
    const size_t seg2_off = head;
    if (two_sets) { head += seg_words * sizeof(uint32_t); head = (head + 255) & ~(size_t)255; }
    int r = ssb_scratch_reserve(ctx, head + extra_bytes);
    if (r) return r;
    uint8_t *base = (uint8_t *)ctx->scratch;
    s->st[0] = (TncDevState *)(base);
    s->st[1] = (TncDevState *)(base + 64);
    s->exc_count = (uint32_t *)(base + 128);
    s->ovf = (uint32_t *)(base + 192);
    s->acc = (unsigned long long *)(base + 256);
    s->exc = (uint32_t *)(base + 1024);
    s->exc_cap = (uint32_t)cap;
    s->seg = (uint32_t *)(base + seg_off);
    s->seg_words = seg_words;
    s->exc_count2 = two_sets ? (uint32_t *)(base + 136) : NULL;      // (inside the range tnc_begin clears)
    s->exc2 = two_sets ? (uint32_t *)(base + exc2_off) : NULL;
    s->seg2 = two_sets ? (uint32_t *)(base + seg2_off) : NULL;
    s->tail = base + head;
    return SSB_OK;
}

__global__ void tnc_final_kernel(const unsigned long long *__restrict__ acc, const uint32_t *__restrict__ ovf,
                                 unsigned long long *__restrict__ counts)
{
    if (*ovf == 0) counts[threadIdx.x] += acc[threadIdx.x];
}

// One piece (n <= TNC_MAX_PIECE) already in HBM; state flows st_in -> st_out on the device.
int tnc_piece(ssb_ctx *ctx, cudaStream_t stream, const uint8_t *d, size_t n, const TncScratch &s,
              TncDevState *st_in, TncDevState *st_out)
{
    SSB_CUDA(ctx, cudaMemsetAsync(s.exc_count, 0, sizeof(uint32_t), stream));
    SSB_CUDA(ctx, cudaMemsetAsync(s.seg, 0, ((n >> TNC_SEG_SHIFT) + 2) * sizeof(uint32_t), stream));
    size_t n_chunks = (n + TNC_BPT - 1) / TNC_BPT;
    int grid = (int)((n_chunks + (size_t)TNC_BLOCK * TNC_SUB - 1) / ((size_t)TNC_BLOCK * TNC_SUB));
    int max_grid = ctx->sm_count * 8;            // persistent: every block folds its 1296-bin histogram once
    if (grid > max_grid) grid = max_grid;
    if (grid < 1) grid = 1;
    SSB_LAUNCH_P(ctx, SSB_K_TNC_SCAN, tnc_scan_kernel, grid, TNC_BLOCK, 0, stream, d, n, st_in, (const uint8_t *)NULL, s.acc, s.exc_count, s.exc, s.exc_cap, s.seg);
    int fgrid = ctx->sm_count * 4;
    SSB_LAUNCH_P(ctx, SSB_K_TNC_FIXUP, tnc_fixup_kernel, fgrid, 128, 0, stream, d, n, st_in, st_out, s.acc, s.exc_count, s.ovf, s.exc, s.exc_cap, s.seg);
    return SSB_OK;
}

int tnc_begin(ssb_ctx *ctx, cudaStream_t stream, const TncScratch &s, const ssb_tnc_carry *carry_in)
{
    static const ssb_tnc_carry zero = {0, {0, 0, 0}, 0, 0, 0, 0};
    SSB_CUDA(ctx, cudaMemsetAsync(s.exc_count, 0, 128 + 64 * sizeof(unsigned long long), stream));   // count, ovf, acc
    SSB_CUDA(ctx, cudaMemcpyAsync(s.st[0], carry_in ? carry_in : &zero, sizeof(ssb_tnc_carry), cudaMemcpyHostToDevice, stream));
    return SSB_OK;
}

// Device-resident buffer of any size, cut into pieces of at most `piece` bytes.  The scan of piece i+1 does not depend on the fix-up of piece i
// (see tnc_scan_kernel: prev3), so the scans run back to back on the compute stream and the fix-ups, which carry the state from piece to piece,
// follow on the second stream; two sets of exception lists alternate.
int tnc_run_device(ssb_ctx *ctx, const uint8_t *d, size_t n, size_t piece, const TncScratch &s, int *cur_io)
{
    int cur = *cur_io;
    size_t off = 0;
    cudaStream_t sS = ctx->stream, sF = s.exc2 ? ctx->copy_stream : ctx->stream;
    int i = 0;
    do {
        const size_t len = n - off < piece ? n - off : piece;
        const int k = s.exc2 ? (i & 1) : 0;
        uint32_t *exc_count = k ? s.exc_count2 : s.exc_count, *exc = k ? s.exc2 : s.exc, *seg = k ? s.seg2 : s.seg;
        if (s.exc2 && i >= 2) SSB_CUDA(ctx, cudaStreamWaitEvent(sS, ctx->ev[2 + k], 0));           // set k: fixed up and free again
        SSB_CUDA(ctx, cudaMemsetAsync(exc_count, 0, sizeof(uint32_t), sS));
        SSB_CUDA(ctx, cudaMemsetAsync(seg, 0, ((len >> TNC_SEG_SHIFT) + 2) * sizeof(uint32_t), sS));
        const size_t n_chunks = (len + TNC_BPT - 1) / TNC_BPT;
        int grid = (int)((n_chunks + (size_t)TNC_BLOCK * TNC_SUB - 1) / ((size_t)TNC_BLOCK * TNC_SUB));
        const int max_grid = ctx->sm_count * 8;            // persistent: every block folds its 1296-bin histogram once
        if (grid > max_grid) grid = max_grid;
        if (grid < 1) grid = 1;
        const uint8_t *prev3 = (s.exc2 && off >= 3) ? d + off - 3 : NULL;
        if (s.exc2 && !prev3 && i > 0) SSB_CUDA(ctx, cudaStreamWaitEvent(sS, ctx->ev[2 + ((i - 1) & 1)], 0));  // (cannot happen with pieces of >= 32 bytes: the state itself)
        SSB_LAUNCH_P(ctx, SSB_K_TNC_SCAN, tnc_scan_kernel, grid, TNC_BLOCK, 0, sS, d + off, len, s.st[cur], prev3, s.acc, exc_count, exc, s.exc_cap, seg);
        if (s.exc2) { SSB_CUDA(ctx, cudaEventRecord(ctx->ev[k], sS)); SSB_CUDA(ctx, cudaStreamWaitEvent(sF, ctx->ev[k], 0)); }
        SSB_LAUNCH_P(ctx, SSB_K_TNC_FIXUP, tnc_fixup_kernel, ctx->sm_count * 4, 128, 0, sF, d + off, len, s.st[cur], s.st[cur ^ 1], s.acc, exc_count, s.ovf, exc, s.exc_cap, seg);
        if (s.exc2) SSB_CUDA(ctx, cudaEventRecord(ctx->ev[2 + k], sF));
        cur ^= 1;
        off += len;
        i++;
    } while (off < n);
    if (s.exc2) {                                           // the compute stream goes on when the last fix-ups are done
        SSB_CUDA(ctx, cudaStreamWaitEvent(sS, ctx->ev[2 + ((i - 1) & 1)], 0));
        if (i >= 2) SSB_CUDA(ctx, cudaStreamWaitEvent(sS, ctx->ev[2 + (i & 1)], 0));
    }
    *cur_io = cur;
    return SSB_OK;
}

} // namespace

// ---- C ABI ---------------------------------------------------------------------------------

extern "C" int ssb_tnc_count_device(ssb_ctx *ctx, const uint8_t *d_fasta, size_t n, const ssb_tnc_carry *carry_in,
                                    ssb_tnc_carry *carry_out, int64_t *d_counts64)
{
    if (!ctx || (!d_fasta && n) || !d_counts64) return SSB_E_ARG;
    if (((uintptr_t)d_fasta & 15) != 0) return SSB_E_ARG;          // 16-byte vector loads
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    size_t piece = n < TNC_MAX_PIECE ? n : TNC_MAX_PIECE;
    if (const char *e = getenv("SSB_TNC_PIECE")) { const size_t v = strtoull(e, NULL, 10) & ~(size_t)15; if (v >= 32 && v < piece) piece = v; }     // (tests: many pieces on a small input)
    for (int attempt = 0; attempt < 2; attempt++) {
        TncScratch s;
        int r = tnc_scratch(ctx, piece, 0, &s, n > piece);       // several pieces: two sets, the scans run ahead of the fix-ups
        if (r) return r;
        // attempt 1 (after an overflow): pieces so small that the list holds their worst case
        size_t use = attempt == 0 ? piece : TNC_SAFE_PIECE;
        if ((r = tnc_begin(ctx, ctx->stream, s, carry_in))) return r;
        int cur = 0;
        if ((r = tnc_run_device(ctx, d_fasta, n, use, s, &cur))) return r;
        SSB_LAUNCH(ctx, tnc_final_kernel, 1, 64, 0, ctx->stream, s.acc, s.ovf, (unsigned long long *)d_counts64);
        uint32_t ovf = 0;
        ssb_tnc_carry out;
        SSB_CUDA(ctx, cudaMemcpyAsync(&ovf, s.ovf, sizeof ovf, cudaMemcpyDeviceToHost, ctx->stream));
        SSB_CUDA(ctx, cudaMemcpyAsync(&out, s.st[cur], sizeof out, cudaMemcpyDeviceToHost, ctx->stream));
        SSB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (!ovf) { if (carry_out) *carry_out = out; return SSB_OK; }
    }
    snprintf(ctx->err, sizeof ctx->err, "tnc: exception list overflow in safe mode");
    return SSB_E_FORMAT;
}

extern "C" int ssb_tnc_count_host(ssb_ctx *ctx, const uint8_t *fasta, size_t n, const ssb_tnc_carry *carry_in,
                                  ssb_tnc_carry *carry_out, int64_t counts64[64])
{
    if (!ctx || (!fasta && n) || !counts64) return SSB_E_ARG;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    size_t chunk = (size_t)64 << 20;
    if (const char *e = getenv("SSB_TNC_CHUNK")) { size_t v = strtoull(e, NULL, 10); if (v >= 64) chunk = v; }
    chunk &= ~(size_t)31;
    if (chunk > TNC_MAX_PIECE) chunk = TNC_MAX_PIECE;
    if (chunk > n) chunk = (n + 31) & ~(size_t)31;
    if (chunk < 32) chunk = 32;
    // is the caller's buffer already pinned?  then copy straight out of it
    cudaPointerAttributes attr;
    bool pinned_src = cudaPointerGetAttributes(&attr, fasta) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    for (int attempt = 0; attempt < 2; attempt++) {
        TncScratch s;
        int r = tnc_scratch(ctx, chunk, 2 * chunk, &s);
        if (r) return r;
        uint8_t *dbuf[2] = {s.tail, s.tail + chunk};
        if (!pinned_src) { r = ssb_pinned_reserve(ctx, 2 * chunk); if (r) return r; }
        uint8_t *hbuf[2] = {(uint8_t *)ctx->pinned, (uint8_t *)ctx->pinned + chunk};
        if ((r = tnc_begin(ctx, ctx->stream, s, carry_in))) return r;
        int cur = 0;
        size_t n_chunks = n ? (n + chunk - 1) / chunk : 1;
        // ev[k]: chunk copied into buffer k (copy stream -> compute); ev[2+k]: buffer k consumed (compute -> copy)
        for (size_t i = 0; i < n_chunks; i++) {
            int k = (int)(i & 1);
            size_t off = i * chunk, len = n - off < chunk ? n - off : chunk;
            if (i >= 2) SSB_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev[2 + k], 0));
            const uint8_t *src = fasta + off;
            if (!pinned_src && len) {
                if (i >= 2) SSB_CUDA(ctx, cudaEventSynchronize(ctx->ev[k]));      // staging buffer k is free again
                memcpy(hbuf[k], src, len);
                src = hbuf[k];
            }
            if (len) SSB_CUDA(ctx, cudaMemcpyAsync(dbuf[k], src, len, cudaMemcpyHostToDevice, ctx->copy_stream));
            SSB_CUDA(ctx, cudaEventRecord(ctx->ev[k], ctx->copy_stream));
            SSB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev[k], 0));
            if ((r = tnc_piece(ctx, ctx->stream, dbuf[k], len, s, s.st[cur], s.st[cur ^ 1]))) return r;
            cur ^= 1;
            SSB_CUDA(ctx, cudaEventRecord(ctx->ev[2 + k], ctx->stream));
        }
        uint32_t ovf = 0;
        ssb_tnc_carry out;
        SSB_CUDA(ctx, cudaMemcpyAsync(counts64, s.acc, 64 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        SSB_CUDA(ctx, cudaMemcpyAsync(&ovf, s.ovf, sizeof ovf, cudaMemcpyDeviceToHost, ctx->stream));
        SSB_CUDA(ctx, cudaMemcpyAsync(&out, s.st[cur], sizeof out, cudaMemcpyDeviceToHost, ctx->stream));
        SSB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (!ovf) { if (carry_out) *carry_out = out; return SSB_OK; }
        // adversarial input (a header every few bytes): redo with chunks whose worst case fits the list
        chunk = TNC_SAFE_PIECE;
    }
    snprintf(ctx->err, sizeof ctx->err, "tnc: exception list overflow in safe mode");
    return SSB_E_FORMAT;
}

// ---- BED-restricted scan (BASELINE config 3, SURVEY 8d C3) ---------------------------------------------------------------------
// The reference has no BED input; the semantics are those of running it on the FASTA `bedtools getfasta` would make: per interval,
// in BED order, a header line and the interval's bases on ONE line.  That FASTA is built here on the device (a gather over the
// genome text through a .fai-style index) and scanned by the exact kernels above, so every quirk of the reference -- which records
// are kept, the single straddling window between consecutive kept records -- is inherited rather than restated.
namespace {
__global__ void bed_len_kernel(const ssb_bed_interval *__restrict__ iv, size_t first, size_t n_own, long long ctx_iv, unsigned long long *__restrict__ len)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_own) return;
    // slot 0 = the context record (the nearest earlier interval that holds an upper-case base; empty when there is none), then the own ones
    const long long k = i == 0 ? ctx_iv : (long long)(first + i - 1);
    len[i] = k < 0 ? 0ull : (unsigned long long)(iv[k].end - iv[k].start) + 3ull;        // ">\n" + bases + "\n"
}
__device__ __forceinline__ size_t fasta_byte(const ssb_fasta_contig &c, int64_t p) { return (size_t)c.seq_off + (size_t)p + (size_t)(p / c.line_bases) * (size_t)(c.line_bytes - c.line_bases); }
// the interval lies inside its contig
__host__ __device__ inline bool bed_iv_ok(const ssb_bed_interval &v, const ssb_fasta_contig *contigs, size_t n_contigs)
{
    return v.contig >= 0 && (size_t)v.contig < n_contigs && v.start >= 0 && v.end >= v.start && v.end <= contigs[v.contig].len;
}
// a byte the index places at a base position cannot be a line end or a header: then the index does not describe this file
__device__ __forceinline__ bool not_a_sequence_byte(uint8_t ch) { return ch == '\n' || ch == '>'; }
// one warp per record
__global__ void bed_gather_kernel(const uint8_t *__restrict__ fa, size_t n, const ssb_fasta_contig *__restrict__ contigs, size_t n_contigs, const ssb_bed_interval *__restrict__ iv,
                                  size_t first, size_t n_own, long long ctx_iv, const unsigned long long *__restrict__ off, uint8_t *__restrict__ out, unsigned int *__restrict__ bad)
{
    const int lane = threadIdx.x & 31;
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i > n_own) return;
    const long long k = i == 0 ? ctx_iv : (long long)(first + i - 1);
    if (k < 0) return;
    const ssb_bed_interval v = iv[k];
    if (!bed_iv_ok(v, contigs, n_contigs)) { if (lane == 0) atomicOr(bad, 1u); return; }
    const ssb_fasta_contig c = contigs[v.contig];
    uint8_t *o = out + off[i];
    if (lane == 0) { o[0] = '>'; o[1] = '\n'; o[2 + (v.end - v.start)] = '\n'; }
    for (int64_t p = v.start + lane; p < v.end; p += 32) {
        const size_t b = fasta_byte(c, p);
        const uint8_t ch = b < n ? fa[b] : (uint8_t)'\n';
        if (not_a_sequence_byte(ch)) atomicOr(bad, 2u);
        o[2 + (p - v.start)] = ch;
    }
}
// nearest interval before `first` that holds an upper-case base (its last base is what the reference would carry into the next record)
__global__ void bed_context_kernel(const uint8_t *__restrict__ fa, size_t n, const ssb_fasta_contig *__restrict__ contigs, size_t n_contigs, const ssb_bed_interval *__restrict__ iv,
                                   size_t first, long long *__restrict__ ctx_iv)
{
    const int lane = threadIdx.x;
    for (long long k = (long long)first - 1; k >= 0; k--) {
        const ssb_bed_interval v = iv[k];
        if (!bed_iv_ok(v, contigs, n_contigs)) continue;
        const ssb_fasta_contig c = contigs[v.contig];
        bool any = false;
        for (int64_t p0 = v.start; p0 < v.end && !any; p0 += 32) {
            const int64_t p = p0 + lane;
            uint8_t ch = 0;
            if (p < v.end) { const size_t b = fasta_byte(c, p); ch = b < n ? fa[b] : 0; }
            any = __ballot_sync(0xffffffffu, is_base(ch)) != 0u;
        }
        if (any) { if (lane == 0) *ctx_iv = k; return; }
    }
    if (lane == 0) *ctx_iv = -1;
}
__global__ void sub_counts_kernel(unsigned long long *__restrict__ a, const unsigned long long *__restrict__ b) { a[threadIdx.x] -= b[threadIdx.x]; }
} // namespace

extern "C" int ssb_tnc_count_bed_device(ssb_ctx *ctx, const uint8_t *d_fasta, size_t n, const ssb_fasta_contig *contigs, size_t n_contigs,
                                        const ssb_bed_interval *intervals, size_t n_intervals, size_t first, size_t last, int64_t *d_counts64)
{
    if (!ctx || (!d_fasta && n) || !d_counts64 || (n_contigs && !contigs) || (n_intervals && !intervals) || first > last || last > n_intervals) return SSB_E_ARG;
    if (first == last) return SSB_OK;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t n_own = last - first;
    size_t own_bytes = 0, max_len = 0;
    for (size_t i = 0; i < n_intervals; i++) {
        if (intervals[i].end < intervals[i].start) return SSB_E_ARG;
        const size_t l = (size_t)(intervals[i].end - intervals[i].start);
        if (i < first && l > max_len) max_len = l;
        if (i >= first && i < last) own_bytes += l + 3;
    }
    struct Bufs { void *p[8]; int k = 0; ~Bufs() { for (int i = 0; i < k; i++) cudaFree(p[i]); } } bufs;
    auto dev = [&](size_t bytes) -> void * { void *q = NULL; if (cudaMalloc(&q, bytes ? bytes : 1) != cudaSuccess) return NULL; bufs.p[bufs.k++] = q; return q; };
    ssb_fasta_contig *d_contigs = (ssb_fasta_contig *)dev(n_contigs * sizeof *contigs);
    ssb_bed_interval *d_iv = (ssb_bed_interval *)dev(n_intervals * sizeof *intervals);
    unsigned long long *d_len = (unsigned long long *)dev((n_own + 2) * 8), *d_off = (unsigned long long *)dev((n_own + 2) * 8);
    const size_t out_cap = own_bytes + max_len + 3 + 64;
    uint8_t *d_out = (uint8_t *)dev(out_cap);
    long long *d_ctx = (long long *)dev(64);                     // [0] context interval, [1] flags, [2..] 64 counters follow in their own buffer
    unsigned long long *d_tmp = (unsigned long long *)dev(64 * 8);
    if (!d_contigs || !d_iv || !d_len || !d_off || !d_out || !d_ctx || !d_tmp) { snprintf(ctx->err, sizeof ctx->err, "tnc/bed: device allocation failed"); return SSB_E_NOMEM; }
    SSB_CUDA(ctx, cudaMemcpyAsync(d_contigs, contigs, n_contigs * sizeof *contigs, cudaMemcpyHostToDevice, s));
    SSB_CUDA(ctx, cudaMemcpyAsync(d_iv, intervals, n_intervals * sizeof *intervals, cudaMemcpyHostToDevice, s));
    SSB_CUDA(ctx, cudaMemsetAsync(d_ctx, 0, 64, s));
    SSB_LAUNCH(ctx, bed_context_kernel, 1, 32, 0, s, d_fasta, n, d_contigs, n_contigs, d_iv, first, d_ctx);
    long long h_ctx = -1;
    SSB_CUDA(ctx, cudaMemcpyAsync(&h_ctx, d_ctx, 8, cudaMemcpyDeviceToHost, s));
    SSB_CUDA(ctx, cudaStreamSynchronize(s));
    SSB_LAUNCH(ctx, bed_len_kernel, (int)((n_own + 1 + 255) / 256), 256, 0, s, d_iv, first, n_own, h_ctx, d_len);
    // offsets: host prefix sums (a few hundred thousand intervals)
    std::vector<unsigned long long> off(n_own + 2);
    off[0] = 0; off[1] = h_ctx < 0 ? 0 : (unsigned long long)(intervals[h_ctx].end - intervals[h_ctx].start) + 3;
    for (size_t i = 0; i < n_own; i++) off[i + 2] = off[i + 1] + (unsigned long long)(intervals[first + i].end - intervals[first + i].start) + 3;
    const size_t total = (size_t)off[n_own + 1], ctx_bytes = (size_t)off[1];
    if (total > out_cap) return SSB_E_STATE;
    SSB_CUDA(ctx, cudaMemcpyAsync(d_off, off.data(), (n_own + 2) * 8, cudaMemcpyHostToDevice, s));
    unsigned int *d_bad = (unsigned int *)(d_ctx + 1);
    SSB_LAUNCH(ctx, bed_gather_kernel, (int)(((n_own + 1) * 32 + 127) / 128), 128, 0, s, d_fasta, n, d_contigs, n_contigs, d_iv, first, n_own, h_ctx, d_off, d_out, d_bad);
    unsigned int h_bad = 0;
    SSB_CUDA(ctx, cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, s));
    SSB_CUDA(ctx, cudaStreamSynchronize(s));
    if (h_bad) { snprintf(ctx->err, sizeof ctx->err, "tnc/bed: %s", (h_bad & 1) ? "an interval lies outside its contig" : "the FASTA index does not describe the file (line widths)"); return SSB_E_FORMAT; }
    // the built FASTA through the exact scan; then take the context record's own windows off again
    int rc = ssb_tnc_count_device(ctx, d_out, total, NULL, NULL, d_counts64);
    if (rc) return rc;
    if (ctx_bytes) {
        SSB_CUDA(ctx, cudaMemsetAsync(d_tmp, 0, 64 * 8, s));
        if ((rc = ssb_tnc_count_device(ctx, d_out, ctx_bytes, NULL, NULL, (int64_t *)d_tmp))) return rc;
        SSB_LAUNCH(ctx, sub_counts_kernel, 1, 64, 0, s, (unsigned long long *)d_counts64, (const unsigned long long *)d_tmp);
    }
    SSB_CUDA(ctx, cudaStreamSynchronize(s));
    return SSB_OK;
}

// ---- Per-interval counts ---------------------------------------------------------------------------------------------------------------
// Row i = what the reference counts on the FASTA that holds interval i alone (a header line, the bases on one line).  For one line the
// reference's rules reduce to: a window counts at every p in [start, end-2) where bases p, p+1, p+2 are all upper-case A/C/G/T.  So the
// genome text is read in place through the index -- no extracted FASTA.
//
// Work: an item is (interval, segment of at most IV_T windows); an interval of 1 or 2 bases is one item without windows, so that its
// bytes are checked against the index like any other.  Every warp of a persistent grid takes one contiguous range of the item list
// (equal item counts; the host finds where each range starts).  Per item the warp stages the segment's bases plus the 2-base halo into
// shared memory with the line terminators removed (aligned 4-byte loads, 128 bytes per warp step), then takes the windows four at a time
// from SWAR codes as the generic path of tnc_scan_kernel does, counting into a lane-private 64-bin shared histogram (column = lane:
// no atomics, no bank conflicts).  The histogram is flushed when the warp leaves an interval: with plain adds when the warp covered the
// whole interval (every short interval), with 64 global atomics when the interval is split between warps (long intervals, whole-genome bins).
namespace {
constexpr int IV_T = 2048;                        // windows per item
constexpr int IV_WARPS = 4;                       // warps per block: 4 x (8 KiB histogram + 2 KiB stage) of static shared memory
constexpr int IV_STAGE_WORDS = (4 + IV_T + 2 + 3) / 4 + 1;   // a zero word, then the segment's IV_T + 2 bases, then zero fill

struct IvTask { unsigned long long iv, item, count; };   // a warp's range: `count` items from item `item` of interval `iv`

__host__ __device__ inline unsigned long long iv_items(int64_t len) { return len <= 0 ? 0ull : len <= 2 ? 1ull : (unsigned long long)(len - 2 + IV_T - 1) / IV_T; }

// the warp's histogram is added to `row` (plain adds when this warp owns the whole row, atomics otherwise) and zeroed
__device__ __forceinline__ void iv_flush(uint32_t *h, int lane, int64_t *row, bool whole)
{
    __syncwarp();
    uint32_t t0 = 0, t1 = 0;
#pragma unroll 8
    for (int j = 0; j < 32; j++) {                       // lane takes bins lane and lane + 32; (j + lane) & 31 spreads the banks
        const int c = (j + lane) & 31;
        t0 += h[lane * 32 + c]; h[lane * 32 + c] = 0;
        t1 += h[(lane + 32) * 32 + c]; h[(lane + 32) * 32 + c] = 0;
    }
    if (whole) { if (t0) row[lane] += t0; if (t1) row[lane + 32] += t1; }
    else {
        if (t0) atomicAdd((unsigned long long *)&row[lane], (unsigned long long)t0);
        if (t1) atomicAdd((unsigned long long *)&row[lane + 32], (unsigned long long)t1);
    }
    __syncwarp();
}

__global__ void __launch_bounds__(IV_WARPS * 32)
tnc_intervals_kernel(const uint8_t *__restrict__ fa, size_t n, const ssb_fasta_contig *__restrict__ contigs, const ssb_bed_interval *__restrict__ iv,
                     const IvTask *__restrict__ tasks, size_t n_tasks, int64_t *__restrict__ rows, unsigned int *__restrict__ bad)
{
    __shared__ uint32_t hist[IV_WARPS][64 * 32];
    __shared__ uint32_t stage[IV_WARPS][IV_STAGE_WORDS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const size_t gw = (size_t)blockIdx.x * IV_WARPS + wid;
    if (gw >= n_tasks) return;
    uint32_t *h = hist[wid], *st = stage[wid];
    uint8_t *stb = reinterpret_cast<uint8_t *>(st) + 4;   // base j of the segment; st[0] stays 0 (no window ends before base 2)
    for (int i = lane; i < 64 * 32; i += 32) h[i] = 0;
    if (lane == 0) st[0] = 0;
    const IvTask t = tasks[gw];
    size_t i = (size_t)t.iv;
    unsigned long long k = t.item, left = t.count;
    bool whole = k == 0, counted = false;
    while (left) {
        const ssb_bed_interval v = iv[i];
        const unsigned long long ni = iv_items(v.end - v.start);
        if (ni == 0) { i++; continue; }
        const ssb_fasta_contig c = contigs[v.contig];
        const int64_t s = v.start + (int64_t)k * IV_T, e = min(s + IV_T + 2, v.end);
        const uint32_t m = (uint32_t)(e - s);
        const size_t tbs = fasta_byte(c, s), tbe = fasta_byte(c, e - 1);
        if (tbe >= n) { if (lane == 0) atomicOr(bad, 2u); }
        else {
            // ---- stage bases [s, e) into stb[0, m): text byte a >= tbs sits in column (col0 + a - tbs) mod line_bytes of line
            //      (col0 + a - tbs) / line_bytes, counted from s's line; it is a base when that column is < line_bases
            __syncwarp();                                                 // the previous item's windows are counted
            if (lane == 0) st[(m + 3) / 4] = 0;                           // zero the bytes after base m - 1 in its word
            __syncwarp();
            const uint32_t lb = c.line_bases, lbytes = c.line_bytes, col0 = (uint32_t)(s % lb);
            const size_t a_end = tbe + 1;
            bool badc = false;
            for (size_t w0 = (tbs & ~(size_t)3) + 4 * lane; w0 < a_end; w0 += 4 * 128) {
                uint32_t wd[4];
#pragma unroll
                for (int u = 0; u < 4; u++) { const size_t wa = w0 + 128 * u; wd[u] = wa < a_end ? ld_word(fa, n, wa) : 0u; }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const size_t wa = w0 + 128 * u;
                    if (wa >= a_end) break;
                    const uint32_t j0 = wa < tbs ? (uint32_t)(tbs - wa) : 0u;          // first byte of this word at or after s
                    const uint32_t c0 = col0 + (uint32_t)(wa + j0 - tbs);
                    uint32_t dl = c0 / lbytes, col = c0 - dl * lbytes;
#pragma unroll
                    for (uint32_t j = 0; j < 4; j++) {
                        if (j < j0 || wa + j >= a_end) continue;
                        const uint8_t ch = (uint8_t)(wd[u] >> (8 * j));
                        const uint32_t d = dl * lb + col - col0;                    // (< m whenever the index is consistent)
                        if (col < lb && d < m) { stb[d] = ch; badc |= not_a_sequence_byte(ch); }
                        if (++col == lbytes) { col = 0; dl++; }
                    }
                }
            }
            if (badc) atomicOr(bad, 2u);
            __syncwarp();
            // ---- windows ending at bases 4(w-1) .. 4(w-1)+3, from the words w-1 and w of the stage
            bool any = false;
            for (uint32_t w = 1 + lane; w <= (m + 3) / 4; w += 32) {
                const uint32_t prev = st[w - 1], cur = st[w];
                const uint32_t bm = (msb4(base_flags(prev)) >> 2) | (msb4(base_flags(cur)) << 2);
                uint32_t win = bm & (bm >> 1) & (bm >> 2) & 0xFu;
                if (win) {
                    const uint32_t x = win_index4(ref_codes4(prev), ref_codes4(cur));
                    any = true;
                    while (win) { const int b = __ffs(win) - 1; win &= win - 1; h[((x >> (8 * b)) & 63u) * 32 + lane]++; }
                }
            }
            counted |= __any_sync(0xffffffffu, any);
        }
        left--;
        if (++k == ni) {
            if (counted) iv_flush(h, lane, rows + 64 * i, whole);
            i++; k = 0; whole = true; counted = false;
        }
    }
    if (counted) iv_flush(h, lane, rows + 64 * i, false);            // the range ends inside interval i: other warps share its row
}
} // namespace

extern "C" int ssb_tnc_count_intervals_device(ssb_ctx *ctx, const uint8_t *d_fasta, size_t n, const ssb_fasta_contig *contigs, size_t n_contigs,
                                              const ssb_bed_interval *intervals, size_t n_intervals, size_t first, size_t last, int64_t *d_rows)
{
    if (!ctx || (!d_fasta && n) || !d_rows || (n_contigs && !contigs) || (n_intervals && !intervals) || first > last || last > n_intervals) return SSB_E_ARG;
    if (((uintptr_t)d_fasta & 15) != 0) return SSB_E_ARG;
    if (first == last) return SSB_OK;
    const size_t n_own = last - first;
    const ssb_bed_interval *own = intervals + first;
    unsigned long long total = 0;
    bool outside = false;
    for (size_t i = 0; i < n_own; i++) {
        const ssb_bed_interval &v = own[i];
        if (v.end < v.start) return SSB_E_ARG;
        if (!bed_iv_ok(v, contigs, n_contigs)) { outside = true; continue; }
        const ssb_fasta_contig &c = contigs[v.contig];
        if (v.end > v.start && (c.line_bases == 0 || c.line_bytes < c.line_bases)) outside = true;   // no geometry to read it by
        total += iv_items(v.end - v.start);
    }
    if (outside) { snprintf(ctx->err, sizeof ctx->err, "tnc/intervals: an interval lies outside its contig"); return SSB_E_FORMAT; }
    if (total == 0) return SSB_OK;
    SSB_CUDA(ctx, cudaSetDevice(ctx->device));
    int per_sm = 0;
    SSB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tnc_intervals_kernel, IV_WARPS * 32, 0));
    unsigned long long n_warps = (unsigned long long)ctx->sm_count * (per_sm > 0 ? per_sm : 1) * IV_WARPS;
    if (n_warps > total) n_warps = total;
    // warp w takes items [total w / n_warps, total (w + 1) / n_warps)
    std::vector<IvTask> tasks((size_t)n_warps);
    unsigned long long before = 0, w = 0, lo = 0;
    for (size_t i = 0; i < n_own && w < n_warps; i++) {
        const unsigned long long ni = iv_items(own[i].end - own[i].start);
        while (w < n_warps && lo < before + ni) {
            const unsigned long long hi = (unsigned long long)((unsigned __int128)total * (w + 1) / n_warps);
            tasks[w] = IvTask{i, lo - before, hi - lo};
            lo = hi; w++;
        }
        before += ni;
    }
    // device copies of the index, this range's intervals and the ranges, in the context's scratch
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t o_iv = up(n_contigs * sizeof *contigs), o_task = o_iv + up(n_own * sizeof *intervals), o_bad = o_task + up(tasks.size() * sizeof(IvTask));
    int r = ssb_scratch_reserve(ctx, o_bad + 256);
    if (r) return r;
    uint8_t *base = (uint8_t *)ctx->scratch;
    cudaStream_t st = ctx->stream;
    SSB_CUDA(ctx, cudaMemcpyAsync(base, contigs, n_contigs * sizeof *contigs, cudaMemcpyHostToDevice, st));
    SSB_CUDA(ctx, cudaMemcpyAsync(base + o_iv, own, n_own * sizeof *intervals, cudaMemcpyHostToDevice, st));
    SSB_CUDA(ctx, cudaMemcpyAsync(base + o_task, tasks.data(), tasks.size() * sizeof(IvTask), cudaMemcpyHostToDevice, st));
    SSB_CUDA(ctx, cudaMemsetAsync(base + o_bad, 0, sizeof(unsigned int), st));
    const int grid = (int)((n_warps + IV_WARPS - 1) / IV_WARPS);
    SSB_LAUNCH_P(ctx, SSB_K_TNC_INTERVALS, tnc_intervals_kernel, grid, IV_WARPS * 32, 0, st, d_fasta, n, (const ssb_fasta_contig *)base,
                 (const ssb_bed_interval *)(base + o_iv), (const IvTask *)(base + o_task), tasks.size(), d_rows, (unsigned int *)(base + o_bad));
    unsigned int h_bad = 0;
    SSB_CUDA(ctx, cudaMemcpyAsync(&h_bad, base + o_bad, sizeof h_bad, cudaMemcpyDeviceToHost, st));
    SSB_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_bad) { snprintf(ctx->err, sizeof ctx->err, "tnc/intervals: the FASTA index does not describe the file (line widths)"); return SSB_E_FORMAT; }
    return SSB_OK;
}

// .fai-style index of a FASTA text (host): one entry per '>' record, in file order.  names[i] points into the text (not NUL
// terminated).  Like faidx it takes the line geometry from a record's first sequence line and refuses (SSB_E_FORMAT) a record
// in which another line but the last has a different width; blank lines after the last sequence line are allowed ('>' cannot
// occur inside a sequence line, so the next record is found by a byte search, not line by line).
extern "C" int ssb_fasta_index(const uint8_t *fa, size_t n, ssb_fasta_contig *out, const char **names, uint32_t *name_lens, size_t cap, size_t *n_out)
{
    if ((!fa && n) || !n_out) return SSB_E_ARG;
    size_t k = 0, p = 0;
    while (p < n) {
        if (fa[p] != '>') {                                   // text before the first header: skip the line
            const uint8_t *nl = (const uint8_t *)memchr(fa + p, '\n', n - p);
            if (!nl) break;
            p = (size_t)(nl - fa) + 1;
            continue;
        }
        const uint8_t *nl = (const uint8_t *)memchr(fa + p, '\n', n - p);
        const size_t e = nl ? (size_t)(nl - fa) : n;          // end of the header line
        const size_t s0 = e < n ? e + 1 : n;                  // first sequence byte
        size_t end = n;                                       // start of the next record
        for (size_t r = s0; r < n;) {
            const uint8_t *g = (const uint8_t *)memchr(fa + r, '>', n - r);
            if (!g) break;
            const size_t gp = (size_t)(g - fa);
            if (gp == s0 || fa[gp - 1] == '\n') { end = gp; break; }
            r = gp + 1;
        }
        ssb_fasta_contig c; c.seq_off = s0; c.len = 0; c.line_bases = 0; c.line_bytes = 0;
        const size_t bytes = end - s0;
        if (bytes) {
            const uint8_t *nl2 = (const uint8_t *)memchr(fa + s0, '\n', bytes);
            const size_t l_bytes = nl2 ? (size_t)(nl2 - (fa + s0)) + 1 : bytes;            // first line incl. its newline
            size_t term = nl2 ? 1 : 0; if (nl2 && l_bytes >= 2 && fa[s0 + l_bytes - 2] == '\r') term = 2;
            c.line_bytes = (uint32_t)l_bytes; c.line_bases = (uint32_t)(l_bytes - term);
            if (c.line_bases) {
                // up to the last byte that is not a line terminator: blank lines after the last sequence line hold no base
                size_t t = bytes;
                while (t && (fa[s0 + t - 1] == '\n' || fa[s0 + t - 1] == '\r')) t--;
                const size_t full = term ? t / l_bytes : 0, rest = term ? t % l_bytes : t;      // (term 0: one unterminated line)
                // every line but the last ends where the first one does, with the same terminator, and the last is no longer: any
                // other record (a blank line inside it, a ragged line) would put bases where the geometry does not look for them
                bool uniform = rest <= c.line_bases && !memchr(fa + s0 + full * l_bytes, '\n', rest);
                for (size_t j = 1; uniform && j <= full; j++) {
                    const uint8_t *x = fa + s0 + j * l_bytes;
                    uniform = x[-1] == '\n' && (x[-2] == '\r') == (term == 2);
                }
                if (!uniform) return SSB_E_FORMAT;
                c.len = (int64_t)(full * c.line_bases + rest);
            }
        }
        if (k < cap && out) {
            size_t q = p + 1; while (q < e && fa[q] != ' ' && fa[q] != '\t' && fa[q] != '\r') q++;
            if (names) names[k] = (const char *)fa + p + 1;
            if (name_lens) name_lens[k] = (uint32_t)(q - p - 1);
            out[k] = c;
        }
        k++;
        p = end;
    }
    *n_out = k;
    return SSB_OK;
}

// Host restatement of the *state transition only* (no counting): lets a caller cut a FASTA into
// shards for several GPUs.  Mirrors the state-out task of tnc_fixup_kernel.
extern "C" int ssb_tnc_carry_after(const uint8_t *b, size_t n_, const ssb_tnc_carry *carry_in, ssb_tnc_carry *out)
{
    if (!out || (!b && n_)) return SSB_E_ARG;
    ssb_tnc_carry st;
    if (carry_in && carry_in->started) st = *carry_in;
    else { memset(&st, 0, sizeof st); st.prev[0] = st.prev[1] = st.prev[2] = '\n'; }
    long n = (long)n_;
    auto scan_back_h = [&](long e, long &a, bool &hb) {
        hb = false; a = -1;
        for (long i = e - 1; i >= 0; i--) { if (b[i] == '\n') { a = i + 1; return; } if (is_base(b[i])) hb = true; }
    };
    auto resolve = [&](long q) -> uint8_t {
        long e = q - 1;
        for (;;) {
            if (e < 0) return st.carry;
            long a; bool hb; scan_back_h(e, a, hb);
            if (a >= 0) { if (e > a && b[a] != '>' && hb) return b[e - 1]; e = a - 1; }
            else {
                bool nonempty = st.frag_nonempty || e > 0;
                uint8_t first = st.frag_nonempty ? st.frag_first : b[0];
                hb = hb || st.frag_has_base;
                uint8_t last = e > 0 ? b[e - 1] : st.prev[2];
                return (nonempty && first != '>' && hb) ? last : st.carry;
            }
        }
    };
    ssb_tnc_carry o; memset(&o, 0, sizeof o);
    o.started = 1;
    long a; bool hb; scan_back_h(n, a, hb);
    if (a >= 0) { o.carry = resolve(a); o.frag_nonempty = n > a; o.frag_first = n > a ? b[a] : 0; o.frag_has_base = hb; }
    else {
        o.carry = st.carry; o.frag_nonempty = st.frag_nonempty || n > 0;
        o.frag_first = st.frag_nonempty ? st.frag_first : (n > 0 ? b[0] : 0);
        o.frag_has_base = st.frag_has_base || hb;
    }
    uint8_t all[6] = {st.prev[0], st.prev[1], st.prev[2], 0, 0, 0};
    if (n >= 3) { o.prev[0] = b[n - 3]; o.prev[1] = b[n - 2]; o.prev[2] = b[n - 1]; }
    else { for (long k = 0; k < n; k++) all[3 + k] = b[k]; for (int k = 0; k < 3; k++) o.prev[k] = all[n + k]; }
    *out = o;
    return SSB_OK;
}

extern "C" void ssb_tnc_fold32(const int64_t counts64[64], int64_t out32[32])
{
    for (int i = 0; i < 32; i++) {
        const char *s = OUT_ORDER[i];
        const int fwd = 16 * ref_code(s[0]) + 4 * ref_code(s[1]) + ref_code(s[2]);
        const int rev = 16 * (3 - ref_code(s[2])) + 4 * (3 - ref_code(s[1])) + (3 - ref_code(s[0]));
        out32[i] = counts64[fwd] + counts64[rev];
    }
}

extern "C" int ssb_tnc_format(const int64_t counts64[64], char *dst, size_t cap)
{
    if (!counts64 || !dst) return SSB_E_ARG;
    int64_t o[32];
    ssb_tnc_fold32(counts64, o);
    size_t used = 0;
    for (int i = 0; i < 32; i++) {
        int w = snprintf(dst + used, cap - used, "%s\t%ld\n", OUT_ORDER[i], (long)o[i]);
        if (w < 0 || (size_t)w >= cap - used) return SSB_E_ARG;
        used += (size_t)w;
    }
    return (int)used;
}
