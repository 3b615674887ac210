// sam_parse.cuh -- one streaming pass over SAM text: find lines, parse the fields the spike path
// needs, apply the reference's read filter.  (Stands in for htslib's sam_read1 + read_bam,
// stochasticSpike.c:243-268, for SAM text input.)
//
// Shape: persistent blocks (exactly the resident ones) pull 32 KiB tiles of the body in order (atomic ticket).  A block
//   1. asks the tile it is likely to draw next into L2 and stages its own tile (+ an overhang for the line that runs past
//      the end) in shared memory with ONE bulk asynchronous copy (cp.async.bulk = TMA, completion on an mbarrier; SASS: UBLKCP);
//   2. finds newlines byte-parallel: SWAR zero-byte test per 32-bit word; the few chunks that hold one note its position, warp ballots
//      count them per (iteration, warp) cell and a 64-cell scan orders the line starts (tiles that do not look like SAM -- two newlines
//      within 16 bytes -- and the ragged last tiles take the general path: 16-bit mask per chunk, block-wide scan of popcounts);
//   3. publishes its line count at once; warp 0 then finds the end of the tile's last line and learns the global index of
//      the first one from a decoupled look-back over per-tile line counts (single pass, no separate counting kernel)
//      WHILE
//   4. warps 1..3 parse the heads (QNAME .. TLEN) of one line per thread, lanes kept together (parse_head_conv);
//   5. all threads stage the reference window under the tile's reads; warps 1..3 then check SEQ, QUAL and the reference
//      in one pass (long_fields), list the exceptional bases and write the 64-byte SamRecs.
// Two line parsers: the fast one of steps 4-5 (parse_head_conv + long_fields) for lines of the common shape, and the careful
// parse_line() for the lines the fast one objects to, the lines beyond the first 96 of a tile, and the lines that end past the
// staged window (those it reads from global memory).  They share the read filter (read_bam_filter) and the CIGAR ops (cigar_op).
// Shared-memory regions change hands inside a tile (newline masks -> reference window, line starts -> exception buffer).
// HBM traffic: the text is read once; 64 B per line and 8 B per exceptional base are written.
#pragma once
#include "common.cuh"
#include "spike_types.cuh"

namespace samparse {

constexpr int TILE      = 32768;
constexpr int OVERHANG  = 3072;
constexpr int THREADS   = 128;
constexpr int MAX_LINES = 2048;                 // a valid SAM line has >= 22 bytes -> <= 1490 per tile
constexpr int CHUNKS    = TILE / 16;            // 16-byte chunks per tile
constexpr int CPT       = CHUNKS / THREADS;     // chunks per thread (a multiple of 8)
static_assert(CPT * (THREADS / 32) == 64, "the one-pass newline search scans 64 (iteration, warp) cells, two per lane");
constexpr int REFW      = 4096;                 // reference window staged per tile for the base-vs-reference comparison
constexpr int EXC_BUF   = 1024;                 // exceptional bases of one tile, kept in shared memory until the tile is done
// shared memory of a block: the staged text, then two regions that change hands inside a tile:
//   A: newline masks (steps 2-3)  ->  reference window (steps 4-5);   B: line starts (steps 3-4a)  ->  exception buffer (steps 4b-5)
constexpr int REGION_A  = (CHUNKS * 2 > REFW + 64 ? CHUNKS * 2 : REFW + 64);
constexpr int REGION_B  = (MAX_LINES * 2 > EXC_BUF * 4 ? MAX_LINES * 2 : EXC_BUF * 4);
constexpr int SMEM_BYTES = TILE + OVERHANG + REGION_A + REGION_B + 64;

// tile_state word: bits 63..62 = status (0 none, 1 aggregate, 2 inclusive prefix), low 62 bits = line count
constexpr unsigned long long ST_AGG = 1ull << 62, ST_INC = 2ull << 62, ST_MASK = 3ull << 62;

struct ContigNames {          // device: concatenated names + offsets, for RNAME -> tid
    const char *text;
    const uint32_t *off;      // n + 1 offsets
    int n;
    // reference sequences (ASCII, case preserved) for the base-vs-reference comparison of kept simple reads
    const uint8_t *const *seq; const int64_t *len;
    // exceptional bases found while tokenising: (global line index << 16) | query offset.  The tally stage resolves them.
    unsigned long long *exc; unsigned long long *exc_count; unsigned long long exc_cap;
    // shard support: a read whose last base lies before keep_lo = (tid << 32 | pos) belongs to an earlier shard's pileups only
    // (it is one of the halo lines in front of this shard's own) and is not kept; n_keep counts the kept lines.
    unsigned long long keep_lo; unsigned long long *n_keep;
    unsigned long long *n_float;      // lines flagged REC_AUX_F
    unsigned long long *max_end;      // largest end coordinate of a kept line (the output-order sort packs its keys with it)
    // per line, next to the record: kept? and the sortedness key of a pushed read ((tid + 1) << 32 | pos, 0 otherwise) -- what the
    // compaction scans need, so that nobody has to read the 64-byte records again just for two fields
    uint32_t *keep_flag; unsigned long long *pkey;
};

__device__ __forceinline__ void line_keys(const ContigNames &names, unsigned long long g, const SamRec &r)
{
    names.keep_flag[g] = (r.bits & REC_KEEP) ? 1u : 0u;
    // bam_plp_push compares (tid, pos) of every pushed read with the running maximum
    names.pkey[g] = (r.bits & REC_PUSHED) ? (((unsigned long long)(uint32_t)(r.tid + 1) << 32) | (uint32_t)r.pos) : 0ull;
}

// applies the shard's lower bound to a parsed record
__device__ __forceinline__ void shard_keep(SamRec &r, const ContigNames &names)
{
    if ((r.bits & REC_KEEP) && ((((unsigned long long)(uint32_t)r.tid << 32) | (uint32_t)r.end) - 1 < names.keep_lo)) r.bits &= (uint8_t)~REC_KEEP;
}

// The end of every line: a refused line (rc != 0) leaves an empty record and, if it is the first error, its code and offset;
// the shard's lower bound applies; the record and its keys go to line g.
__device__ __forceinline__ void store_line(SamRec &r, int rc, size_t s, unsigned long long g, const ContigNames &names,
                                           SamRec *__restrict__ recs, size_t rec_cap, SpikeErr *__restrict__ err)
{
    if (rc) { if (atomicCAS(&err->code, 0, rc) == 0) err->where = s; memset(&r, 0, sizeof r); r.line_off = s; r.tid = -1; }
    shard_keep(r, names);
    if (g < rec_cap) { recs[g] = r; line_keys(names, g, r); }
    else if (atomicCAS(&err->code, 0, SSB_E_NOMEM) == 0) err->where = s;
}

__device__ __forceinline__ uint32_t nl_mask16(uint4 v)
{
    // 16-bit mask of '\n' bytes in 16 bytes
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        uint32_t d = w[j] ^ 0x0A0A0A0Au;
        uint32_t t = (d & 0x7f7f7f7fu) + 0x7f7f7f7fu;
        uint32_t z = ~(t | d | 0x7f7f7f7fu);                   // 0x80 per '\n'
        m |= ((((z >> 7) * 0x00204081u) >> 21) & 0xFu) << (4 * j);
    }
    return m;
}

// read_bam (stochasticSpike.c:253-263) + bam_plp_push's tid test, on a parsed record
__device__ __forceinline__ void read_bam_filter(SamRec &r)
{
    const bool pass = !(r.flag & (4 | 256 | 512 | 1024)) && r.mapq >= 30 && !((r.flag & 1) && !(r.flag & 2));
    if (pass && r.tid >= 0) r.bits |= (r.end > r.pos) ? (REC_PUSHED | REC_KEEP) : REC_PUSHED;
}

// The class of a CIGAR op byte, branch free: CIG_OK for the nine ops (MIDNSHP=X), CIG_REF if it consumes the reference,
// CIG_QRY if it consumes the query, CIG_M for M, = and X.  0 for any other byte.
constexpr uint32_t CIG_REF = 1, CIG_QRY = 2, CIG_M = 4, CIG_OK = 8;
__host__ __device__ constexpr uint32_t cig_bit(char op) { return 1u << (op - '='); }      // one bit per byte '=' .. 'X'
__device__ __forceinline__ uint32_t cigar_op(uint32_t c)
{
    constexpr uint32_t M = cig_bit('M') | cig_bit('=') | cig_bit('X');
    constexpr uint32_t REF = M | cig_bit('D') | cig_bit('N'), QRY = M | cig_bit('I') | cig_bit('S');
    constexpr uint32_t OK = REF | QRY | cig_bit('H') | cig_bit('P');
    const uint32_t i = c - '=', b = i <= (uint32_t)('X' - '=') ? 1u << i : 0u;
    return ((b & REF) ? CIG_REF : 0u) | ((b & QRY) ? CIG_QRY : 0u) | ((b & M) ? CIG_M : 0u) | ((b & OK) ? CIG_OK : 0u);
}

__device__ __forceinline__ bool seq_char_ok(uint8_t c)
{
    // the bytes htslib's 4-bit round trip maps to themselves: "=ACMGRSVTWYHKDBN"
    if (c == '=') return true;
    if (c < 'A' || c > 'Z') return false;
    return ((0x16e34cfu >> (c - 'A')) & 1u) != 0;          // A B C D G H K M N R S T V W Y
}

// RNAME / RNEXT lookup: index of the first @SQ named by the len bytes at p, -1 if none
__device__ __forceinline__ int name_lookup(const uint8_t *p, uint32_t len, const ContigNames &names, int hint)
{
    auto same = [&](int c) {
        uint32_t a = names.off[c], b = names.off[c + 1];
        if (b - a != len) return false;
        for (uint32_t i = 0; i < len; i++) if ((uint8_t)names.text[a + i] != p[i]) return false;
        return true;
    };
    if (hint >= 0 && hint < names.n && same(hint)) {
        // the hint is only valid if no EARLIER @SQ carries the same name (sam_hdr_name2tid returns the first)
        for (int c = 0; c < hint; c++) if (same(c)) return c;
        return hint;
    }
    for (int c = 0; c < names.n; c++) if (same(c)) return c;
    return -1;
}

// Float text that htslib prints back unchanged: it parses the value into a 32-bit float and prints it with "%g" (six
// significant digits, trailing zeros dropped, exponent form outside 1e-4 .. 1e6).  A decimal of at most six significant
// digits survives the trip through a float (FLT_DIG = 6), so the text is its own "%g" image exactly when it has the shape
// "%g" produces: [-]ddd[.ddd] without superfluous zeros for exponents -4 .. 5, [-]d[.ddddd]e[+-]XX otherwise (normal range
// only), or inf / nan.
template <typename AT>
__host__ __device__ __noinline__ bool canon_float_t(const AT &at, size_t a, size_t b)
{
    if (a < b && at(a) == '-') a++;
    if (a >= b) return false;
    if (b - a == 3 && ((at(a) == 'i' && at(a + 1) == 'n' && at(a + 2) == 'f') || (at(a) == 'n' && at(a + 1) == 'a' && at(a + 2) == 'n'))) return true;
    size_t e = a; while (e < b && at(e) != 'e') e++;                       // mantissa [a, e), exponent text (e, b)
    size_t dot = a; while (dot < e && at(dot) != '.') dot++;
    const size_t ni = dot - a, nf = dot < e ? e - dot - 1 : 0;             // integer / fraction digits
    if (ni == 0 || (dot < e && nf == 0)) return false;
    for (size_t i = a; i < e; i++) { if (i == dot) continue; const uint8_t c = at(i); if (c < '0' || c > '9') return false; }
    if (ni > 1 && at(a) == '0') return false;
    if (nf && at(e - 1) == '0') return false;                              // "%g" drops trailing zeros
    if (e == b) {
        // fixed notation: decimal exponent X in [-4, 6)
        if (at(a) != '0') return ni <= 6 && ni + nf <= 6;
        if (nf == 0) return true;                                          // "0", "-0"
        size_t z = 0; while (z < nf && at(dot + 1 + z) == '0') z++;
        return z < nf && z <= 3 && nf - z <= 6;
    }
    // exponent notation: one non-zero digit before the point, sign, at least two exponent digits
    if (ni != 1 || at(a) == '0' || 1 + nf > 6) return false;
    size_t x = e + 1;
    if (x >= b || (at(x) != '+' && at(x) != '-')) return false;
    const bool neg = at(x) == '-'; x++;
    if (b - x != 2) return false;
    if (at(x) < '0' || at(x) > '9' || at(x + 1) < '0' || at(x + 1) > '9') return false;
    const int X = (at(x) - '0') * 10 + (at(x + 1) - '0');
    if (X > 37) return false;                                              // keep clear of overflow / denormals
    return neg ? X >= 5 : X >= 6;                                          // inside -4 .. 5 "%g" would have used fixed notation
}

// One optional field [p, q): TAG:TYPE:VALUE in the form htslib prints back unchanged.
// Float-typed fields (TAG:f:..., TAG:B:f,...) are not judged while tokenising (their check is long and would cost every line
// registers): the tokeniser answers AUX_FLOAT, the line is flagged REC_AUX_F, and aux_float_kernel judges the flagged lines.
constexpr int AUX_FLOAT = 1;
template <typename AT>       // at(i): byte i of the body
__host__ __device__ __forceinline__ int aux_ok_t(const AT at, size_t p, size_t q)
{
    if (q - p < 5 || at(p + 2) != ':' || at(p + 4) != ':') return SSB_E_FORMAT;
    uint8_t ty = at(p + 3);
    size_t v = p + 5;
    auto canon_int = [&](size_t a, size_t b) {
        if (a < b && at(a) == '-') a++;
        if (a >= b) return false;
        if (b - a > 1 && at(a) == '0') return false;
        if (b - a > 10) return false;
        for (size_t i = a; i < b; i++) { uint8_t c = at(i); if (c < '0' || c > '9') return false; }
        return !(b - a == 1 && at(a) == '0' && a > v && at(a - 1) == '-');      // "-0"
    };
    switch (ty) {
    case 'f': return AUX_FLOAT;
    case 'A': return (q - v == 1 && at(v) >= '!' && at(v) <= '~') ? 0 : SSB_E_FORMAT;
    case 'i': return canon_int(v, q) ? 0 : SSB_E_FORMAT;
    case 'Z': for (size_t i = v; i < q; i++) { uint8_t c = at(i); if (c < ' ' || c > '~') return SSB_E_FORMAT; } return 0;
    case 'H': if ((q - v) & 1) return SSB_E_FORMAT;
              for (size_t i = v; i < q; i++) { uint8_t c = at(i); if (!((c >= '0' && c <= '9') || (c >= 'A' && c <= 'F'))) return SSB_E_FORMAT; } return 0;
    case 'B': {
        if (q - v < 1) return SSB_E_FORMAT;
        uint8_t st = at(v);
        if (st == 'f') return AUX_FLOAT;
        if (st != 'c' && st != 'C' && st != 's' && st != 'S' && st != 'i' && st != 'I') return SSB_E_FORMAT;
        size_t a = v + 1;
        while (a < q) {
            if (at(a) != ',') return SSB_E_FORMAT;
            size_t b = a + 1; while (b < q && at(b) != ',') b++;
            size_t s0 = a + 1;
            if (s0 < b && at(s0) == '-') s0++;
            if (s0 >= b || (b - s0 > 1 && at(s0) == '0')) return SSB_E_FORMAT;
            for (size_t i = s0; i < b; i++) { uint8_t c = at(i); if (c < '0' || c > '9') return SSB_E_FORMAT; }
            a = b;
        }
        return 0;
    }
    default: return SSB_E_FORMAT;      // unknown types are outside the byte-exact pass-through envelope
    }
}

// the float-typed field [p, q) in full: TAG:f:<float> or TAG:B:f,<float>,...
template <typename AT>
__host__ __device__ int aux_float_ok_t(const AT &at, size_t p, size_t q)
{
    if (q - p < 6 || at(p + 2) != ':' || at(p + 4) != ':') return SSB_E_FORMAT;
    if (at(p + 3) == 'f') return canon_float_t(at, p + 5, q) ? 0 : SSB_E_FORMAT;
    if (at(p + 3) != 'B' || at(p + 5) != 'f') return SSB_E_FORMAT;
    size_t a = p + 6;
    while (a < q) {
        if (at(a) != ',') return SSB_E_FORMAT;
        size_t b = a + 1; while (b < q && at(b) != ',') b++;
        if (!canon_float_t(at, a + 1, b)) return SSB_E_FORMAT;
        a = b;
    }
    return 0;
}

// L = first byte of the line, offsets relative to it
__device__ int aux_ok(const uint8_t *L, uint32_t p, uint32_t q)
{
    return aux_ok_t([=](size_t i) -> uint8_t { return L[i]; }, (size_t)p, (size_t)q);
}

// ---- SWAR helpers for the long fields (SEQ, QUAL) ----

__device__ __forceinline__ uint32_t zero_bytes(uint32_t d)          // 0x80 in every byte of d that is zero (exact)
{
    return ~(((d & 0x7f7f7f7fu) + 0x7f7f7f7fu) | d | 0x7f7f7f7fu);
}
// bytes of the word that are NOT printable ('!'..'~'): 0x80 flags
__device__ __forceinline__ uint32_t nonprint_bytes(uint32_t w)
{
    return (w | ~(w + 0x5f5f5f5fu) | (w + 0x01010101u)) & 0x80808080u;     // >= 0x80, < 0x21, > 0x7e  (the adds cannot carry across bytes once w < 0x80)
}
// bytes of the word that are not one of A C G T N (low three bits 1 3 7 4 6 select the only candidate): 0x80 flags
__device__ __forceinline__ uint32_t non_acgtn_bytes(uint32_t w)
{
    const uint32_t TLO = 0x43014101u, THI = 0x474E0154u;       // index: 0->01 1->'A' 2->01 3->'C' 4->'T' 5->01 6->'N' 7->'G'
    const uint32_t sidx = w & 0x07070707u;
    const uint32_t e0 = __byte_perm(TLO, THI, sidx), e1 = __byte_perm(TLO, THI, sidx >> 16);
    const uint32_t e = __byte_perm(e0, e1, 0x6420);
    return ~zero_bytes(w ^ e) & 0x80808080u;
}
__device__ __forceinline__ uint64_t mix64(uint64_t x)
{
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
    return x;
}

// ---- the careful parser: any line, in the staged tile or in global memory ----

// Canonical decimal field ending at '\t' (what htslib prints back): digits only, no leading zero unless the value is 0,
// value <= maxv.  On success p sits on the terminating tab.
__device__ __forceinline__ int udec(const uint8_t *L, uint32_t &p, uint32_t len, uint32_t maxv, uint32_t &out)
{
    const uint32_t p0 = p; uint32_t v = 0;
    while (p < len) {
        const uint32_t c = L[p];
        if (c == '\t') break;
        const uint32_t d = c - '0';
        if (d > 9u) return SSB_E_FORMAT;
        if (p - p0 >= 10) return SSB_E_FORMAT;                     // more than 10 digits cannot fit
        if (v > 214748364u || (v == 214748364u && d > 7u)) return SSB_E_FORMAT;
        v = v * 10u + d;
        p++;
    }
    if (p >= len || p == p0 || v > maxv) return SSB_E_FORMAT;
    if (p - p0 > 1 && L[p0] == '0') return SSB_E_FORMAT;
    out = v;
    return 0;
}

// words of the field [a, a+n) of the line: `bad` accumulates the flagged bytes.  CHECK(x) returns 0x80 flags.  Only aligned
// words inside the field are loaded, so the line may lie in shared or in global memory.
template <typename CHECK>
__device__ __forceinline__ uint32_t check_field(const uint8_t *L, uint32_t a, uint32_t n, uint32_t filler, CHECK check)
{
    uint32_t bad = 0, i = 0;
    // bytes up to the first 4-byte aligned address, then aligned words, then the tail
    const uint32_t mis = (uint32_t)((4u - ((uint32_t)(uintptr_t)(L + a) & 3u)) & 3u);
    if (mis) {
        const uint32_t take = mis < n ? mis : n;
        uint32_t x = filler;
        for (uint32_t k = 0; k < take; k++) x = (x & ~(0xffu << (8 * k))) | ((uint32_t)L[a + k] << (8 * k));
        bad |= check(x);
        i = take;
    }
    const uint32_t *W = reinterpret_cast<const uint32_t *>(L + a + i);
    const uint32_t nw = (n - i) >> 2;
    for (uint32_t w = 0; w < nw; w++) bad |= check(W[w]);
    i += nw << 2;
    if (i < n) {
        uint32_t x = filler;
        for (uint32_t k = 0; i + k < n; k++) x = (x & ~(0xffu << (8 * k))) | ((uint32_t)L[a + i + k] << (8 * k));
        bad |= check(x);
    }
    return bad;
}

// Parses the line of len bytes at L (without its newline; has_nl: one follows) that starts at body offset s.  L points into the
// staged tile or into the body in global memory; every read is at an offset < len, so nothing past the line is touched.
// Returns 0 or an SSB_E_* code.  A line is accepted only if htslib's parse -> format round trip (sam_read1 + sam_write1,
// stochasticSpike.c:248,273) reproduces it byte for byte, so that the emit stage can pass the original bytes through
// (DESIGN.md "pass-through envelope").
__device__ int parse_line(const uint8_t *L, uint32_t len, size_t s, bool has_nl, const ContigNames &names, int &tid_cache, SamRec &r)
{
    uint32_t p = 0, v;
    r.line_off = s;
    r.line_len = len + (has_nl ? 1u : 0u);
    r.bits = has_nl ? 0 : REC_NO_NL;
    for (int k = 0; k < 6; k++) r.pad[k] = 0;
    // QNAME: printable, hashed with two 32-bit FNV-1a streams
    uint32_t h1 = 2166136261u, h2 = 0x9747b28cu;
    while (p < len) { const uint32_t c = L[p]; if (c == '\t') break; if (c - '!' > (uint32_t)('~' - '!')) return SSB_E_FORMAT; h1 = (h1 ^ c) * 16777619u; h2 = (h2 + c) * 0x85ebca6bu; p++; }
    if (p >= len || p == 0 || p > 254) return SSB_E_FORMAT;
    r.qhash = ((uint64_t)h1 << 32) | (h2 ^ (h2 >> 15)); r.qname_len = (uint16_t)p;
    p++;
    if (udec(L, p, len, 65535u, v)) return SSB_E_FORMAT;
    r.flag = (uint16_t)v; p++;
    // RNAME
    uint32_t p0 = p;
    while (p < len && L[p] != '\t') p++;
    if (p >= len || p == p0) return SSB_E_FORMAT;
    if (p - p0 == 1 && L[p0] == '*') r.tid = -1;
    else {
        r.tid = name_lookup(L + p0, p - p0, names, tid_cache);
        if (r.tid < 0) return SSB_E_FORMAT;          // htslib would warn and print '*': not a pass-through
        tid_cache = r.tid;
    }
    p++;
    if (udec(L, p, len, 0x7fffffffu, v)) return SSB_E_FORMAT;
    r.pos = (int32_t)v - 1; p++;
    if (udec(L, p, len, 255u, v)) return SSB_E_FORMAT;
    r.mapq = (uint8_t)v; p++;
    // CIGAR
    p0 = p;
    uint32_t rlen = 0, qlen = 0; bool has_cigar = true, simple = true;
    if (p + 1 < len && L[p] == '*' && L[p + 1] == '\t') { has_cigar = false; simple = false; p++; }
    else {
        uint32_t num = 0; int nd = 0; uint32_t first = 0;
        while (p < len) {
            const uint32_t c = L[p];
            if (c == '\t') break;
            const uint32_t d = c - '0';
            if (d <= 9u) { if (!nd) first = c; num = num * 10u + d; nd++; if (nd > 9 || num > 0x0fffffffu) return SSB_E_FORMAT; }
            else {
                if (!nd || (nd > 1 && first == '0')) return SSB_E_FORMAT;
                const uint32_t k = cigar_op(c);
                if (!(k & CIG_OK)) return SSB_E_FORMAT;
                if (k & CIG_REF) rlen += num;
                if (k & CIG_QRY) qlen += num;
                if (!(k & CIG_M)) simple = false;
                if (rlen > 0x7ffffff0u || qlen > 0x7ffffff0u) return SSB_E_FORMAT;
                num = 0; nd = 0;
            }
            p++;
        }
        if (nd) return SSB_E_FORMAT;
    }
    if (simple) r.bits |= REC_SIMPLE;
    if (p >= len || p == p0 || p - p0 > 65535 || p0 > 65535) return SSB_E_FORMAT;
    r.cigar_off = (uint16_t)p0; r.cigar_len = has_cigar ? (uint16_t)(p - p0) : 0;
    if (r.pos < 0 && rlen) return SSB_E_FORMAT;
    if ((uint64_t)(r.pos < 0 ? 0 : r.pos) + rlen > 0x7ffffff0ull) return SSB_E_FORMAT;
    r.end = r.pos + (int32_t)rlen;
    p++;
    // RNEXT: '*', '=' or another @SQ name (the same name spelled out would be printed back as '=')
    p0 = p;
    while (p < len && L[p] != '\t') p++;
    if (p >= len || p == p0) return SSB_E_FORMAT;
    if (!(p - p0 == 1 && (L[p0] == '*' || L[p0] == '='))) {
        const int mt = name_lookup(L + p0, p - p0, names, -1);
        if (mt < 0 || mt == r.tid) return SSB_E_FORMAT;
    } else if (L[p0] == '=' && r.tid < 0) return SSB_E_FORMAT;
    p++;
    if (udec(L, p, len, 0x7fffffffu, v)) return SSB_E_FORMAT;   // PNEXT
    p++;
    if (p < len && L[p] == '-') { p++; if (p < len && L[p] == '0') return SSB_E_FORMAT; }
    if (udec(L, p, len, 0x7fffffffu, v)) return SSB_E_FORMAT;   // TLEN
    p++;
    // SEQ
    r.seq_off = p;
    p0 = p;
    if (p < len && L[p] == '*' && p + 1 < len && L[p + 1] == '\t') { r.l_seq = 0; p++; }
    else if (has_cigar && qlen > 0 && p + qlen < len) {
        const uint32_t bad = check_field(L, p, qlen, 0x41414141u, [](uint32_t x) { return non_acgtn_bytes(x); });
        if (bad) for (uint32_t i = 0; i < qlen; i++) if (!seq_char_ok(L[p + i])) return SSB_E_FORMAT;    // other IUPAC codes, '='
        p += qlen;
        if (L[p] != '\t') return SSB_E_FORMAT;                      // htslib: "CIGAR and query sequence are of different length"
        r.l_seq = qlen;
    } else {
        while (p < len) { const uint8_t c = L[p]; if (c == '\t') break; if (!seq_char_ok(c)) return SSB_E_FORMAT; p++; }
        r.l_seq = p - p0;
        if (has_cigar && qlen != r.l_seq) return SSB_E_FORMAT;
    }
    if (p >= len || p == p0) return SSB_E_FORMAT;
    p++;
    // QUAL
    r.qual_off = p;
    if (p >= len) return SSB_E_FORMAT;
    uint32_t qend;
    if (L[p] == '*' && (p + 1 == len || L[p + 1] == '\t')) { r.bits |= REC_QUALSTAR; qend = p + 1; }
    else {
        qend = p + r.l_seq;
        if (r.l_seq == 0 || qend > len) return SSB_E_FORMAT;
        if (qend < len && L[qend] != '\t') return SSB_E_FORMAT;     // htslib: "SEQ and QUAL are of different length"
        if (check_field(L, p, r.l_seq, 0x21212121u, [](uint32_t x) { return nonprint_bytes(x); })) return SSB_E_FORMAT;
    }
    // optional fields
    for (uint32_t q = qend; q < len;) {
        uint32_t a = q + 1, b = a;
        while (b < len && L[b] != '\t') b++;
        { const int ar = aux_ok(L, a, b); if (ar == AUX_FLOAT) r.bits |= REC_AUX_F; else if (ar) return SSB_E_FORMAT; }
        q = b;
    }
    read_bam_filter(r);
    if ((r.bits & REC_KEEP) && r.l_seq == 0) return SSB_E_FORMAT;  // a kept read without SEQ makes the reference read outside its buffer
    return 0;
}

// ---- the fast parser: the common shape of a line, parsed so that the lanes of a warp stay together ----
//
// The tokeniser has two line parsers: the careful parse_line() above, which decides every line, and this one
// (parse_head_conv + long_fields) for the first lines of a tile that end inside the staged window.  parse_line() leaves a
// loop the moment it meets a byte it does not like; with those exits inside the loops the lanes of a warp no longer
// reconverge after a field whose length differs from lane to lane, and everything behind it -- SEQ, QUAL, the comparison
// with the reference -- runs a few lanes at a time.  The functions below accept exactly the lines of the common shape
// (mapped RNAME, a CIGAR, RNEXT '=' or '*', SEQ of the CIGAR's query length) and collect every objection in one flag
// instead of leaving; a line that raises the flag is handed to parse_line(), which decides.  Every loop has one exit, and
// the lanes meet again (__syncwarp) after each field.  Both share read_bam_filter() and cigar_op().

__device__ __forceinline__ uint32_t udec_conv(const uint8_t *L, uint32_t &p, uint32_t len, uint32_t maxv, uint32_t &out)
{
    const uint32_t p0 = p; uint32_t v = 0, bad = 0;
    while (p < len) {
        const uint32_t c = L[p];
        if (c == '\t') break;
        const uint32_t d = c - '0';
        bad |= (uint32_t)(d > 9u);
        v = v * 10u + d;
        p++;
    }
    // up to nine digits cannot overflow; a longer field (a position beyond 999,999,999) is left to the careful parser, which checks the range digit by digit
    bad |= (uint32_t)(p >= len) | (uint32_t)(p == p0) | (uint32_t)(p - p0 > 9u) | (uint32_t)(v > maxv);
    bad |= (uint32_t)(p - p0 > 1u && L[p0] == '0');
    out = v;
    return bad;
}

// QNAME .. QUAL bounds of the line [L, L+len).  Returns 0 when the line has the common shape and its head is valid; then
// r holds everything but the verdict on the SEQ / QUAL / optional-field bytes, and qend is the end of QUAL.
__device__ __forceinline__ uint32_t parse_head_conv(const uint8_t *L, uint32_t len, size_t s, bool has_nl,
                                                    const ContigNames &names, int tid_cache, SamRec &r, uint32_t &qend, unsigned mask)
{
    uint32_t p = 0, v = 0, bad = 0;
    r.line_off = s;
    r.line_len = len + (has_nl ? 1u : 0u);
    r.bits = has_nl ? 0 : REC_NO_NL;
    for (int k = 0; k < 6; k++) r.pad[k] = 0;
    uint32_t h1 = 2166136261u, h2 = 0x9747b28cu;
    while (p < len) { const uint32_t c = L[p]; if (c == '\t') break; bad |= (uint32_t)(c - '!' > (uint32_t)('~' - '!')); h1 = (h1 ^ c) * 16777619u; h2 = (h2 + c) * 0x85ebca6bu; p++; }
    bad |= (uint32_t)(p >= len) | (uint32_t)(p == 0) | (uint32_t)(p > 254u);
    r.qhash = ((uint64_t)h1 << 32) | (h2 ^ (h2 >> 15)); r.qname_len = (uint16_t)p;
    p++;
    __syncwarp(mask);
    bad |= udec_conv(L, p, len, 65535u, v);
    r.flag = (uint16_t)v; p++;
    __syncwarp(mask);
    uint32_t p0 = p;
    while (p < len && L[p] != '\t') p++;
    bad |= (uint32_t)(p >= len) | (uint32_t)(p == p0);
    __syncwarp(mask);
    r.tid = -1;
    if (!bad && !(p - p0 == 1 && L[p0] == '*')) r.tid = name_lookup(L + p0, p - p0, names, tid_cache);
    bad |= (uint32_t)(r.tid < 0);
    p++;
    __syncwarp(mask);
    bad |= udec_conv(L, p, len, 0x7fffffffu, v);
    r.pos = (int32_t)v - 1; p++;
    bad |= udec_conv(L, p, len, 255u, v);
    r.mapq = (uint8_t)v; p++;
    __syncwarp(mask);
    p0 = p;
    uint32_t rlen = 0, qlen = 0, num = 0, nd = 0, first = 0; bool simple = true;
    while (p < len) {
        const uint32_t c = L[p];
        if (c == '\t') break;
        const uint32_t d = c - '0';
        if (d <= 9u) { if (!nd) first = c; num = num * 10u + d; nd++; bad |= (uint32_t)(nd > 8u); }           // (eight digits < 2^28; longer: the careful parser decides)
        else {
            bad |= (uint32_t)(!nd) | (uint32_t)(nd > 1u && first == '0');
            const uint32_t k = cigar_op(c);
            if (k & CIG_REF) rlen += num;
            if (k & CIG_QRY) qlen += num;
            if (!(k & CIG_M)) simple = false;
            bad |= (uint32_t)!(k & CIG_OK) | (uint32_t)(rlen > 0x7ffffff0u) | (uint32_t)(qlen > 0x7ffffff0u);
            num = 0; nd = 0;
        }
        p++;
    }
    bad |= (uint32_t)(nd != 0) | (uint32_t)(p >= len) | (uint32_t)(p == p0) | (uint32_t)(p - p0 > 65535u) | (uint32_t)(p0 > 65535u);
    if (simple) r.bits |= REC_SIMPLE;
    r.cigar_off = (uint16_t)p0; r.cigar_len = (uint16_t)(p - p0);
    bad |= (uint32_t)(r.pos < 0 && rlen) | (uint32_t)((uint64_t)(r.pos < 0 ? 0 : r.pos) + rlen > 0x7ffffff0ull);
    r.end = r.pos + (int32_t)rlen;
    p++;
    __syncwarp(mask);
    p0 = p;
    while (p < len && L[p] != '\t') p++;
    bad |= (uint32_t)(p >= len) | (uint32_t)(p - p0 != 1u);
    if (!bad) bad |= (uint32_t)(L[p0] != '=' && L[p0] != '*');
    p++;
    __syncwarp(mask);
    bad |= udec_conv(L, p, len, 0x7fffffffu, v);
    p++;
    if (p < len && L[p] == '-') { p++; bad |= (uint32_t)(p < len && L[p] == '0'); }
    bad |= udec_conv(L, p, len, 0x7fffffffu, v);
    p++;
    __syncwarp(mask);
    r.seq_off = p; r.l_seq = qlen;
    bad |= (uint32_t)(qlen == 0) | (uint32_t)(p >= len) | (uint32_t)((uint64_t)p + qlen >= len);
    if (!bad) bad |= (uint32_t)(L[p + qlen] != '\t');
    p += qlen + 1;
    r.qual_off = p;
    bad |= (uint32_t)(p >= len);
    qend = p;
    if (!bad) {
        if (L[p] == '*' && (p + 1 == len || L[p + 1] == '\t')) { r.bits |= REC_QUALSTAR; qend = p + 1; }
        else { qend = p + qlen; bad |= (uint32_t)(qend > len); if (!bad && qend < len) bad |= (uint32_t)(L[qend] != '\t'); }
    }
    read_bam_filter(r);
    return bad;
}

// SEQ and QUAL of one line in a single pass over aligned SEQ words (QUAL, and the reference under the read, are shifted
// into place).  CMP: the read aligns 1:1 to the staged reference window `ref` (bytes that are not A/C/G/T/N replaced by
// 0xff there, so "equal to the reference" implies "valid SEQ byte"); every base that differs from the reference or has
// BQ 0 goes to the tile's exception buffer.  Returns nonzero if a byte is outside what htslib prints back unchanged.
template <bool CMP>
__device__ __forceinline__ uint32_t long_fields(const uint8_t *L, uint32_t seq_off, uint32_t l_seq, uint32_t qual_off, bool qstar,
                                                const uint8_t *ref, const uint8_t *ref_raw, uint32_t line_in_tile,
                                                uint32_t *excbuf, unsigned int *s_nexc)
{
    const uint8_t *As = L + seq_off;
    const uint32_t sh = (uint32_t)((uintptr_t)As & 3u);
    const uint32_t *Ws = reinterpret_cast<const uint32_t *>(As - sh);
    const uint32_t nw = (sh + l_seq + 3u) >> 2;
    const uint8_t *Aq = L + qual_off - sh;
    const uint32_t shq = (uint32_t)((uintptr_t)Aq & 3u) * 8u;
    const uint32_t *Wq = reinterpret_cast<const uint32_t *>(Aq - (shq >> 3));
    uint32_t qprev = qstar ? 0u : Wq[0];
    const uint8_t *Ar = CMP ? ref - sh : L;
    const uint32_t shr = (uint32_t)((uintptr_t)Ar & 3u) * 8u;
    const uint32_t *Wr = reinterpret_cast<const uint32_t *>(Ar - (shr >> 3));
    uint32_t rprev = CMP ? Wr[0] : 0u;
    const uint32_t m_first = 0x80808080u << (8 * sh);
    const uint32_t tail = (sh + l_seq) & 3u;
    const uint32_t m_last = tail ? (0x80808080u >> (8 * (4 - tail))) : 0x80808080u;
    uint32_t bad = 0;                                   // bit 0: a byte outside the envelope, bit 1: the exception buffer is full
    // flags of word j (0x80 per byte that needs a closer look); sq/ql/rf = the word's SEQ, QUAL and reference bytes
    auto flags = [&](uint32_t j, uint32_t &sq, uint32_t &ql, uint32_t &rf) -> uint32_t {
        sq = Ws[j]; ql = 0x7e7e7e7eu; rf = 0;
        if (!qstar) { const uint32_t nx = Wq[j + 1]; ql = __funnelshift_r(qprev, nx, shq); qprev = nx; }
        if (CMP) {
            const uint32_t nx = Wr[j + 1]; rf = __funnelshift_r(rprev, nx, shr); rprev = nx;
            const uint32_t d = sq ^ rf;
            return ((((d & 0x7f7f7f7fu) + 0x7f7f7f7fu) | d | sq) | (ql | ~(ql + 0x5e5e5e5eu) | (ql + 0x01010101u))) & 0x80808080u;   // differs | >= 0x80 | BQ outside '"'..'~'
        }
        return (non_acgtn_bytes(sq) | nonprint_bytes(ql)) & 0x80808080u;
    };
    auto look = [&](uint32_t j, uint32_t fl, uint32_t sq, uint32_t ql, uint32_t rf) {
        while (fl) {
            const uint32_t k = (uint32_t)(__ffs(fl) - 1) >> 3; fl &= fl - 1;
            const uint32_t sb = (sq >> (8 * k)) & 0xffu, qb = (ql >> (8 * k)) & 0xffu;
            if (!seq_char_ok((uint8_t)sb) || qb < '!' || qb > '~') { bad |= 1u; continue; }
            if (CMP) {
                const uint32_t q = 4 * j + k - sh;
                uint32_t rb = (rf >> (8 * k)) & 0xffu;
                if (rb == 0xffu) rb = ref_raw[q];                          // not A/C/G/T: the tally compares with the byte as it is
                // a read N is never a reference base, not even over a reference N (reads through the N runs of a real reference)
                if (sb != rb || qb == '!' || sb == 'N') {
                    const unsigned int slot = atomicAdd(s_nexc, 1u);
                    if (slot < (unsigned int)EXC_BUF) excbuf[slot] = (line_in_tile << 16) | q;
                    else bad |= 2u;
                }
            }
        }
    };
    uint32_t sq, ql, rf;
    {   // first word (its low bytes may belong to the field before)
        uint32_t fl = flags(0, sq, ql, rf) & m_first;
        if (nw == 1) fl &= m_last;
        if (fl) look(0, fl, sq, ql, rf);
    }
    uint32_t j = 1;
    for (; j + 2 < nw; j += 2) {                        // whole words, two at a time
        uint32_t sq2, ql2, rf2;
        const uint32_t f1 = flags(j, sq, ql, rf), f2 = flags(j + 1, sq2, ql2, rf2);
        if (f1 | f2) { look(j, f1, sq, ql, rf); look(j + 1, f2, sq2, ql2, rf2); }
    }
    for (; j < nw; j++) {                               // the rest; the last word's high bytes may belong to the next field
        uint32_t fl = flags(j, sq, ql, rf);
        if (j == nw - 1) fl &= m_last;
        if (fl) look(j, fl, sq, ql, rf);
    }
    return bad;
}

// Decoupled look-back (one warp): lines in all tiles before `tile`.  Every tile publishes its own line count at once (ST_AGG) and its
// inclusive prefix when it knows it (ST_INC).  The frontier of known inclusive prefixes moves one window per L2 round trip, so the
// window is wide: the warp inspects 256 predecessors per hop, all loads of a hop in flight.  Publishes this tile's inclusive prefix.
__device__ __forceinline__ unsigned long long tile_lookback(unsigned long long *__restrict__ tile_state, size_t tile, uint32_t n_here, int lane)
{
    unsigned long long excl = 0;
    volatile unsigned long long *ts = tile_state;
    if (tile != 0) {
        long long j = (long long)tile - 1;
        for (;;) {
            const long long hi = j - 8 * lane;                     // this lane looks at tiles hi, hi-1, .. hi-7
            unsigned long long v[8];
#pragma unroll
            for (int k = 0; k < 8; k++) { v[k] = 2ull << 62; if (hi - k >= 0) v[k] = ts[hi - k]; }     // before tile 0: inclusive prefix 0
            unsigned long long sum = 0; bool has_inc = false;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (has_inc) continue;
                while ((v[k] & ST_MASK) == 0) v[k] = ts[hi - k];                      // not published yet
                sum += v[k] & ~ST_MASK;
                has_inc = (v[k] & ST_MASK) == ST_INC;
            }
            const unsigned inc = __ballot_sync(0xffffffffu, has_inc);
            const int first = inc ? __ffs(inc) - 1 : 31;           // nearest lane that met an inclusive prefix
            unsigned long long c = lane <= first ? sum : 0ull;
#pragma unroll
            for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            excl += c;
            if (inc) break;
            j -= 256;
        }
        if (lane == 0) atomicExch(&tile_state[tile], ST_INC | (excl + n_here));
    }
    return excl;
}

// ---- bulk asynchronous copy (TMA, 1-D) of a tile into shared memory, completion on an mbarrier ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_load_tile(void *dst_smem, const void *src_global, uint32_t bytes, unsigned long long *bar)
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");                       // earlier generic-proxy accesses to the buffer are ordered before the copy
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_global), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}

#ifndef SSB_PARSE_MINBLOCKS
#define SSB_PARSE_MINBLOCKS 5      // 5 blocks of 128 threads per SM: at most 96 registers, against 112 and 4 blocks
#endif
__global__ void __launch_bounds__(THREADS, SSB_PARSE_MINBLOCKS)
parse_kernel(const uint8_t *__restrict__ body, size_t n, ContigNames names, SamRec *__restrict__ recs, size_t rec_cap,
             unsigned long long *__restrict__ tile_state, unsigned int *__restrict__ ticket,
             unsigned long long *__restrict__ n_lines_out, SpikeErr *__restrict__ err)
{
    extern __shared__ __align__(16) uint8_t sm[];
    uint8_t  *text   = sm;                                            // TILE + OVERHANG
    uint16_t *masks  = reinterpret_cast<uint16_t *>(sm + TILE + OVERHANG);                  // region A
    uint8_t  *refwin = sm + TILE + OVERHANG + 16;                                           // region A (16 bytes in front: words are read from 3 bytes before a read's first base)
    uint16_t *starts = reinterpret_cast<uint16_t *>(sm + TILE + OVERHANG + REGION_A);       // region B: MAX_LINES, tile-relative (<= TILE)
    uint32_t *excbuf = reinterpret_cast<uint32_t *>(sm + TILE + OVERHANG + REGION_A);       // region B: EXC_BUF
    __shared__ unsigned int s_tile;
    __shared__ unsigned int s_warp_tot[THREADS / 32];
    __shared__ unsigned long long s_base;
    __shared__ unsigned int s_first;
    __shared__ unsigned long long s_last_end;
    __shared__ int4 s_wkey[THREADS / 32];
    __shared__ unsigned int s_nexc;
    __shared__ unsigned int s_cell[CPT * (THREADS / 32)];            // line starts per (iteration, warp) of the one-pass newline search
    __shared__ __align__(8) unsigned long long s_mbar;          // completion of the tile's bulk copy

    const size_t n_tiles = (n + TILE - 1) / TILE;
    const int tid_ = threadIdx.x, lane = tid_ & 31, wid = tid_ >> 5;
    int tid_cache = -1;
    int end_max = 0;                                                   // largest end of a kept line this thread has seen
    uint32_t mbar_phase = 0;
    if (tid_ == 0) { s_nexc = 0; mbar_init(&s_mbar, 1); }

    for (;;) {
        __syncthreads();
        if (tid_ == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const size_t tile = s_tile;
        if (tile >= n_tiles) break;
        const size_t T0 = tile * TILE;
        const size_t stage_end = (T0 + TILE + OVERHANG < n) ? T0 + TILE + OVERHANG : n;
        // the tile this block is likely to draw next (one round of the resident blocks ahead) is asked into L2 now
        {
            const size_t P0 = T0 + (size_t)gridDim.x * TILE;
#pragma unroll
            for (int q = 0; q < TILE / 128 / THREADS; q++) {
                const size_t a = P0 + ((size_t)q * THREADS + tid_) * 128;
                if (a < n) asm volatile("prefetch.global.L2 [%0];" ::"l"(body + a));
            }
        }
        // 1. stage: ONE bulk asynchronous copy (TMA) of the tile and its overhang, issued by one thread; everybody waits on the mbarrier
        if (T0 + TILE + OVERHANG <= n && ((uintptr_t)body & 15u) == 0) {
            if (tid_ == 0) bulk_load_tile(text, body + T0, (uint32_t)(TILE + OVERHANG), &s_mbar);
            mbar_wait(&s_mbar, mbar_phase);
            mbar_phase ^= 1u;
        } else {
            for (size_t o = (size_t)tid_ * 16; T0 + o < stage_end; o += THREADS * 16) {
                if (T0 + o + 16 <= n && ((uintptr_t)body & 15u) == 0) *reinterpret_cast<uint4 *>(text + o) = *reinterpret_cast<const uint4 *>(body + T0 + o);
                else for (int k = 0; k < 16; k++) text[o + k] = (T0 + o + k < n) ? body[T0 + o + k] : (uint8_t)'\n';
            }
        }
        if (tid_ == 0) s_first = (T0 == 0) ? 1u : (body[T0 - 1] == '\n');
        __syncthreads();
        // 2'. the usual tile (full, SAM-like: never two newlines within 16 bytes, a thread meets at most NL_KEEP of them): one pass.  Chunk
        //     c = 128 it + tid; a chunk with a newline is rare (one in ~20), so only the zero-byte test runs for every chunk and the position
        //     is worked out where one was found.  Line starts are ordered by chunk: the warp ballots count them per (iteration, warp) cell,
        //     and a scan over the 64 cells gives every cell its first slot.  Anything else falls through to the general steps 2-3 below.
        uint32_t n_here = 0, first = s_first;
        bool lines_done = false;
        if (T0 + TILE + OVERHANG <= n) {
            // pass 1, branch free: which of this thread's chunks hold a newline (bit it of `anym`), and its rank among the lanes of the warp
            // that found one in the same iteration (5 bits each, six to a word)
            uint32_t anym = 0, rk[3] = {0u, 0u, 0u};
#pragma unroll
            for (int it = 0; it < CPT; it++) {
                const uint4 v = *reinterpret_cast<const uint4 *>(text + (it * THREADS + tid_) * 16);
                const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
                uint32_t z = 0;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    uint32_t zj = ~((((w4[j] ^ 0x0A0A0A0Au) & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w4[j]) & 0x80808080u;      // 0x80 per '\n'
                    if (it == CPT - 1 && j == 3 && tid_ == THREADS - 1) zj &= 0x00ffffffu;     // newline on the last byte of the tile: the next tile's line
                    z |= zj;
                }
                const bool any = z != 0u;
                const unsigned bal = __ballot_sync(0xffffffffu, any);
                anym |= (any ? 1u : 0u) << it;
                rk[it / 6] |= (uint32_t)__popc(bal & ((1u << lane) - 1u)) << (5 * (it % 6));
                if (lane == 0) s_cell[it * (THREADS / 32) + wid] = (uint32_t)__popc(bal);
            }
            __syncthreads();
            // every warp scans the 64 cells for itself (two per lane)
            const uint32_t c0 = s_cell[2 * lane], c1 = s_cell[2 * lane + 1];
            uint32_t incl = c0 + c1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
            const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
            const uint32_t ex0 = incl - c0 - c1;                        // first slot of cell 2 lane; cell 2 lane + 1 starts c0 later
            bool odd = first + total > (uint32_t)MAX_LINES;             // (block uniform)
            // pass 2, only where a newline was seen (about one chunk in twenty): its position; two in one chunk make the tile odd
            const unsigned act = __ballot_sync(0xffffffffu, anym != 0u && !odd);
            for (unsigned left = act; left;) {                          // (the shuffles need every lane: warp uniform loop over the lanes' turns)
                const bool mine = anym != 0u && !odd;
                const int it = mine ? __ffs(anym) - 1 : 0;
                const uint32_t cell = (uint32_t)it * (THREADS / 32) + wid;
                const uint32_t pa = __shfl_sync(0xffffffffu, ex0, cell >> 1), pb = __shfl_sync(0xffffffffu, c0, cell >> 1);
                if (mine) {
                    anym &= anym - 1u;
                    const uint4 v = *reinterpret_cast<const uint4 *>(text + (it * THREADS + tid_) * 16);
                    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
                    uint32_t m = 0;
#pragma unroll
                    for (int j = 0; j < 4; j++) m |= (((~((((w4[j] ^ 0x0A0A0A0Au) & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w4[j]) & 0x80808080u) * 0x00204081u) >> 28) << (4 * j);
                    if (it == CPT - 1 && tid_ == THREADS - 1) m &= 0x7fffu;
                    if (m & (m - 1u)) odd = true;
                    else starts[first + pa + ((cell & 1u) ? pb : 0u) + (((it < 6 ? rk[0] : it < 12 ? rk[1] : rk[2]) >> (5 * (it < 6 ? it : it < 12 ? it - 6 : it - 12))) & 31u)] = (uint16_t)((it * THREADS + tid_) * 16 + __ffs(m));
                }
                left = __ballot_sync(0xffffffffu, anym != 0u && !odd);
            }
            if (!__syncthreads_or(odd)) {
                n_here = first + total;
                if (tid_ == 0) { atomicExch(&tile_state[tile], (tile == 0 ? ST_INC : ST_AGG) | (unsigned long long)n_here); if (first) starts[0] = 0; }
                lines_done = true;
            }
        }
        if (!lines_done) {
            // 2. newline masks per 16-byte chunk (chunk c covers tile bytes [16c, 16c+16))
            const size_t tile_bytes = (T0 + TILE <= n) ? TILE : n - T0;
            for (int c = tid_; c < CHUNKS; c += THREADS) {
                uint32_t m = 0;
                if ((size_t)c * 16 < tile_bytes) {
                    m = nl_mask16(*reinterpret_cast<const uint4 *>(text + c * 16));
                    size_t rem = tile_bytes - (size_t)c * 16;
                    if (rem < 16) m &= (1u << rem) - 1u;
                }
                masks[c] = (uint16_t)m;
            }
            __syncthreads();
            // a line starts after every newline except one sitting on the last byte of the tile (or of the body)
            // thread t owns chunks [CPT t, CPT t + CPT)
            uint32_t mym[CPT]; uint32_t cnt = 0;
            {
#pragma unroll
                for (int q = 0; q < CPT / 8; q++) {
                    const uint4 mm = *reinterpret_cast<const uint4 *>(masks + CPT * tid_ + 8 * q);
                    const uint32_t w4[4] = {mm.x, mm.y, mm.z, mm.w};
#pragma unroll
                    for (int k = 0; k < 4; k++) { mym[8 * q + 2 * k] = w4[k] & 0xFFFFu; mym[8 * q + 2 * k + 1] = w4[k] >> 16; }
                }
                if (tid_ == THREADS - 1) mym[CPT - 1] &= 0x7FFFu;        // newline on the last byte of a full tile: next tile's line
                // drop a newline that is the very last byte of the body: nothing starts after it
                if (n - T0 <= (size_t)TILE) {
#pragma unroll
                    for (int k = 0; k < CPT; k++) {
                        const size_t cb = T0 + (size_t)(CPT * tid_ + k) * 16;
                        if (n > cb && n - cb <= 16) mym[k] &= ~(1u << (n - cb - 1));
                    }
                }
#pragma unroll
                for (int k = 0; k < CPT; k++) cnt += __popc(mym[k]);
            }
            // block exclusive scan of cnt
            uint32_t incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
            if (lane == 31) s_warp_tot[wid] = incl;
            __syncthreads();
            uint32_t warp_base = 0, total = 0;
#pragma unroll
            for (int w = 0; w < THREADS / 32; w++) { uint32_t t = s_warp_tot[w]; if (w < wid) warp_base += t; total += t; }
            uint32_t my_base = first + warp_base + incl - cnt;
            n_here = first + total;
            // 3a. this tile's line count is published at once; the look-back itself (3b) runs on warp 0 while the other warps parse
            if (tid_ == 0) atomicExch(&tile_state[tile], (tile == 0 ? ST_INC : ST_AGG) | (unsigned long long)n_here);
            if (n_here > MAX_LINES) {                                      // > 2048 lines in 32 KiB cannot be SAM
                if (tid_ == 0 && atomicCAS(&err->code, 0, SSB_E_FORMAT) == 0) err->where = T0;
                // 3b. the global index of this tile's first line (warp 0)
                if (wid == 0) {
                    const unsigned long long excl = tile_lookback(tile_state, tile, n_here, lane);
                    if (lane == 0) { s_base = excl; if (tile == n_tiles - 1) *n_lines_out = excl + n_here; }
                }
                __syncthreads();
                continue;
            }
            if (tid_ == 0 && first) starts[0] = 0;
            if (cnt) {
#pragma unroll
                for (int k = 0; k < CPT; k++) {
                    uint32_t m = mym[k];
                    while (m) {
                        int b = __ffs(m) - 1; m &= m - 1;
                        starts[my_base++] = (uint16_t)((CPT * tid_ + k) * 16 + b + 1);
                    }
                }
            }
        }
        __syncthreads();
        // 4. one line per thread of warps 1..3.  The last line of the tile ends in the overhang (or beyond): warp 0 finds its newline.
        if (wid == 0 && n_here > 0) {
            size_t e = T0 + starts[n_here - 1] + lane;
            for (;;) {
                const bool hit = e >= n || (e < stage_end ? text[e - T0] : body[e]) == '\n';
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                if (m) { e = e - lane + (__ffs(m) - 1); break; }
                e += 32;
            }
            if (lane == 0) s_last_end = e > n ? n : e;
        }
        __syncthreads();
        // 3b. the global index of this tile's first line (warp 0, while the other warps parse)
        if (wid == 0) {
            const unsigned long long excl = tile_lookback(tile_state, tile, n_here, lane);
            if (lane == 0) { s_base = excl; if (tile == n_tiles - 1) *n_lines_out = excl + n_here; }
        }
        // 4a. heads.  The threads of warps 1..3 take one line each; the lanes of a warp stay together (parse_head_conv).  A line that
        //     is not of the common shape, or does not end inside the staged window, is parsed by the careful parser at once.
        constexpr uint32_t PARSERS = THREADS - 32;                         // warp 0 serves (look-back, last newline); the others parse.  (Giving warp 0 a
        // quarter of the lines after its service was measured: 12.6 ms instead of 11.7 -- its lines start late whenever the look-back has to wait.)
        const uint32_t li = wid ? (uint32_t)(lane * (THREADS / 32 - 1) + (wid - 1)) : 0xffffffffu;   // consecutive lines go to different warps
        const bool have = li < n_here;
        const unsigned wmask = __ballot_sync(0xffffffffu, have);
        SamRec r; int rc = 0; bool fast = false; uint32_t qend = 0, lo = 0, len = 0; size_t ls = 0;
        if (have) {
            lo = starts[li]; ls = T0 + lo;
            const size_t e = (li + 1 < n_here) ? T0 + starts[li + 1] - 1 : (size_t)s_last_end;
            const bool insm = e <= stage_end;
            const unsigned fmask = __ballot_sync(wmask, insm);
            len = (uint32_t)(e - ls);
            if (insm) fast = parse_head_conv(text + lo, len, ls, e < n, names, tid_cache, r, qend, fmask) == 0;
            if (!fast) rc = e - ls > 0x7fffffffull ? SSB_E_FORMAT : parse_line(insm ? text + lo : body + ls, len, ls, e < n, names, tid_cache, r);
            if (!rc && r.tid >= 0) tid_cache = r.tid;
        }
        // the reference window under the tile's reads: lowest (tid, pos) among the reads that align 1:1
        const bool elig = fast && names.exc && (r.bits & REC_KEEP) && (r.bits & REC_SIMPLE) && r.l_seq < 65536u &&
                          names.seq[r.tid] && (int64_t)r.end <= names.len[r.tid];
        if (names.exc) {
            const int tmin = __reduce_min_sync(0xffffffffu, elig ? r.tid : 0x7fffffff);
            const int pmin = __reduce_min_sync(0xffffffffu, (elig && r.tid == tmin) ? r.pos : 0x7fffffff);
            const int emax = __reduce_max_sync(0xffffffffu, (elig && r.tid == tmin) ? r.end : 0);
            if (lane == 0) s_wkey[wid] = make_int4(tmin, pmin, emax, 0);
        }
        __syncthreads();
        const unsigned long long gbase = s_base;                           // warp 0 finished the look-back before this barrier
        const unsigned long long gi = gbase + li;
        // tiles of very short lines: the lines beyond the first PARSERS take the careful path, one per thread (before the line starts give way to the exception buffer)
        for (uint32_t i = wid ? li + PARSERS : 0xffffffffu; i < n_here; i += PARSERS) {
            const size_t s = T0 + starts[i];
            const size_t e = (i + 1 < n_here) ? T0 + starts[i + 1] - 1 : (size_t)s_last_end;
            SamRec r2;
            const int rc2 = e - s > 0x7fffffffull ? SSB_E_FORMAT
                                                  : parse_line(e <= stage_end ? text + (s - T0) : body + s, (uint32_t)(e - s), s, e < n, names, tid_cache, r2);
            store_line(r2, rc2, s, gbase + i, names, recs, rec_cap, err);
            if (r2.bits & REC_KEEP) { atomicAdd(names.n_keep, 1ull); if (r2.end > end_max) end_max = r2.end; }
            if (r2.bits & REC_AUX_F) atomicAdd(names.n_float, 1ull);
        }
        bool in_win = false; int32_t w_lo = 0; int wtid = -1;
        if (names.exc) {
            int emax = 0; int pmin = 0x7fffffff; wtid = 0x7fffffff;
#pragma unroll
            for (int w = 0; w < THREADS / 32; w++) { const int4 k = s_wkey[w]; if (k.x < wtid) wtid = k.x; }
#pragma unroll
            for (int w = 0; w < THREADS / 32; w++) { const int4 k = s_wkey[w]; if (k.x == wtid) { if (k.y < pmin) pmin = k.y; if (k.z > emax) emax = k.z; } }
            if (wtid != 0x7fffffff) {
                w_lo = pmin;
                int32_t w_hi = emax; if (w_hi > w_lo + REFW) w_hi = w_lo + REFW;
                const uint8_t *ref = names.seq[wtid] + w_lo;
                const uint32_t ra = (uint32_t)((uintptr_t)ref & 3u);
                const uint32_t *rw = reinterpret_cast<const uint32_t *>(ref - ra);
                uint32_t *dw = reinterpret_cast<uint32_t *>(refwin);
                const int nwords = ((w_hi - w_lo + 3) >> 2) + 1;
                for (int w = tid_; w < nwords; w += THREADS) {
                    const uint32_t x = __funnelshift_r(__ldg(rw + w), __ldg(rw + w + 1), ra * 8);
                    // anything but A C G T can never equal a valid SEQ byte; N too, so that a read over a reference N is always looked at
                    dw[w] = x | (((non_acgtn_bytes(x) | zero_bytes(x ^ 0x4E4E4E4Eu)) >> 7) * 0xffu);
                }
                in_win = elig && gi < rec_cap && gi < (1ull << 47) && r.tid == wtid && r.pos >= w_lo && r.end <= w_lo + REFW;
            } else wtid = -1;
        }
        __syncthreads();
        // 4b. SEQ, QUAL (and the reference under the read) in one pass; optional fields; the record
        if (have) {
            if (fast) {
                const uint8_t *L = text + lo;
                const bool qstar = (r.bits & REC_QUALSTAR) != 0;
                uint32_t bad;
                if (in_win) {
                    bad = long_fields<true>(L, r.seq_off, r.l_seq, r.qual_off, qstar, refwin + (r.pos - w_lo), names.seq[wtid] + r.pos, li, excbuf, &s_nexc);
                    if (!(bad & 2u)) r.bits |= REC_EXC_DONE;               // buffer full: the generic tally takes this read
                    bad &= 1u;
                } else bad = long_fields<false>(L, r.seq_off, r.l_seq, r.qual_off, qstar, NULL, NULL, li, excbuf, &s_nexc);
                for (uint32_t q = qend; q < len;) {                      // optional fields, straight from shared memory
                    uint32_t a = q + 1, b = a;
                    while (b < len && L[b] != '\t') b++;
                    { const int ar = aux_ok(L, a, b); if (ar == AUX_FLOAT) r.bits |= REC_AUX_F; else if (ar) bad = 1; }
                    q = b;
                }
                if (bad) rc = SSB_E_FORMAT;
            }
            store_line(r, rc, ls, gi, names, recs, rec_cap, err);
            if ((r.bits & REC_KEEP) && r.end > end_max) end_max = r.end;
        }
        {   // kept lines of this tile: one atomic per warp
            const unsigned km = __ballot_sync(0xffffffffu, have && (r.bits & REC_KEEP));
            if (lane == 0 && km) atomicAdd(names.n_keep, (unsigned long long)__popc(km));
            if (have && (r.bits & REC_AUX_F)) atomicAdd(names.n_float, 1ull);            // rare: only inputs with float-typed tags
        }
        // 5. hand the tile's exceptional bases over: one reservation per tile, coalesced stores
        if (names.exc) {
            __syncthreads();
            if (wid == 0) {
                unsigned int cnt = s_nexc; if (cnt > (unsigned int)EXC_BUF) cnt = EXC_BUF;
                unsigned long long slot = 0;
                if (lane == 0 && cnt) slot = atomicAdd(names.exc_count, (unsigned long long)cnt);
                slot = __shfl_sync(0xffffffffu, slot, 0);
                for (unsigned int k = lane; k < cnt; k += 32) {
                    const uint32_t v = excbuf[k];
                    if (slot + k < names.exc_cap) names.exc[slot + k] = ((gbase + (v >> 16)) << 16) | (v & 0xffffu);
                }
                __syncwarp();
                if (lane == 0) s_nexc = 0;
            }
        }
    }
    {   // one atomic per warp and kernel
        const int em = __reduce_max_sync(0xffffffffu, end_max);
        if (lane == 0 && em > 0) atomicMax(names.max_end, (unsigned long long)em);
    }
}

// Judges the float-typed optional fields of the lines the tokeniser flagged (REC_AUX_F): one thread per line.
__global__ void aux_float_kernel(const uint8_t *__restrict__ body, size_t n, const SamRec *__restrict__ recs, size_t N, SpikeErr *__restrict__ err)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const SamRec r = recs[i];
    if (!(r.bits & REC_AUX_F)) return;
    const uint8_t *L = body + r.line_off;
    const size_t len = r.line_len - ((r.bits & REC_NO_NL) ? 0 : 1);
    size_t q = r.qual_off;                                        // walk from QUAL to its end, then field by field
    while (q < len && L[q] != '\t') q++;
    auto at = [=](size_t k) -> uint8_t { return L[k]; };
    while (q < len) {
        size_t a = q + 1, b = a;
        while (b < len && L[b] != '\t') b++;
        if (b - a >= 6 && (L[a + 3] == 'f' || (L[a + 3] == 'B' && L[a + 5] == 'f')) && aux_float_ok_t(at, a, b)) {
            if (atomicCAS(&err->code, 0, SSB_E_FORMAT) == 0) err->where = r.line_off;
            return;
        }
        q = b;
    }
}

} // namespace samparse
