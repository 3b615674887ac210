"""Seeded FASTA inputs in the shapes real genome files have and fasta_cases' generators never make: unwrapped contigs and
lines wider than a 4 KiB segment, base-free stretches of 4 KiB to 1 MB placed on and next to segment boundaries, long lines
whose only upper-case base sits at an edge, headers from 1 byte to 70 kB (some full of ACGT runs), CRLF and lone '\\r', IUPAC
codes, bytes >= 0x80, and runs of 10 000 blank or 1-base lines.

Every family returns (data, bounds, placed): the FASTA bytes, the sorted boundary offsets (line starts and ends, header
starts and ends, run starts and ends, and the middle of every "\\r\\n"), and a Counter of the shapes it placed.  The tests
cut the file at every boundary offset +-0..3.  Runs of thousands of identical lines mark only their ends and first and last
lines, so that those cuts stay in the hundreds.

Alignments are to the buffer start.  The GPU tests cut device pieces at multiples of 4 KiB as well, so the same alignments
hold relative to those piece starts."""
import functools
import random
from collections import Counter

import numpy as np

SEG = 4096                                   # tnc.cu: per-segment "no upper-case base" counters (TNC_SEG_SHIFT)
STRETCH_LENGTHS = (4095, 4096, 8191, 8192, 8193, 12289)
LONG_STRETCH_LENGTHS = (100_000, 1_000_000)
WIDTHS = (50, 60, 61, 80, 100, 1000, 2047, 2048, 2049, 4095, 4096, 4097, 65536)
HEADER_SIZES = (1, 40, 3000, 5000, 70_000)
IUPAC = b"ACGTRYKMSWBDHVNacgtrykmswbdhvn"

# shapes each family must place (the CPU test asserts every count is non-zero)
FAMILY_SHAPES = {
    "unwrapped": ["unwrapped_contig", "masked_run_in_unwrapped", "n_run_in_unwrapped", "short_last_line", "no_final_newline"]
                 + ["width_%d" % w for w in WIDTHS],
    "stretches": ["stretch_%d" % L for L in STRETCH_LENGTHS]
                 + ["stretch_%s" % k for k in ("lower", "N", "mixed")]
                 + ["stretch_newlines", "stretch_one_line", "align_on", "align_before", "align_after",
                    "carry_base", "carry_not_base", "lone_base_line_in_stretch"],
    "long_stretches": ["stretch_%d" % L for L in LONG_STRETCH_LENGTHS]
                      + ["stretch_%s" % k for k in ("lower", "N", "mixed")]
                      + ["stretch_newlines", "stretch_one_line", "carry_base", "carry_not_base"],
    "single_base_lines": ["single_base_first", "single_base_last", "single_base_before_seg", "single_base_at_seg",
                          "single_base_line_over_64k"],
    "headers": ["header_%d" % s for s in HEADER_SIZES]
               + ["header_acgt_runs", "header_over_seg", "consecutive_headers", "gt_in_sequence", "gt_last_byte",
                  "semicolon_comment", "header_last_no_newline"],
    "line_ends": ["crlf_contig", "mixed_crlf_lf", "lone_cr", "trailing_blanks", "blank_lines_10000",
                  "one_base_lines_10000", "iupac", "high_bytes"],
}
FAMILIES = tuple(FAMILY_SHAPES)


class _Builder:
    def __init__(self, seed):
        self.rng = random.Random(seed)
        self.buf = bytearray()
        self.bounds = set()
        self.placed = Counter()

    def mark(self, off=None):
        self.bounds.add(len(self.buf) if off is None else off)

    def bases(self, k, alph=b"ACGT"):
        return bytes(self.rng.choices(alph, k=k))

    def line(self, body, end=b"\n", mark=True):
        if mark:
            self.mark()
        self.buf += body
        if mark:
            self.mark()
            if end == b"\r\n":
                self.mark(len(self.buf) + 1)
        self.buf += end
        if mark:
            self.mark()

    def pad_to(self, target, reserve=0):
        """A kept filler line such that the byte `reserve` bytes further on lies at `target` modulo SEG."""
        need = (target - len(self.buf) - reserve) % SEG
        if need:
            self.line(self.bases(need - 1))

    def done(self):
        self.bounds.add(len(self.buf))
        return bytes(self.buf), sorted(self.bounds), self.placed


def _wrap(seq, width, end=b"\n"):
    return [seq[i:i + width] for i in range(0, len(seq), width)], end


def unwrapped(seed=1):
    """Contigs written as one line (10 kB to 500 kB, with soft-masked and N runs), then one contig per line width from 50 to
    65536 with a short last line; the file ends without a final newline."""
    b = _Builder(seed)
    for k, size in enumerate((10_000, 200_000, 500_000)):
        b.line(b">u%d unwrapped" % k)
        seq = bytearray(b.bases(size))
        a = b.rng.randrange(size // 4)
        seq[a:a + 5000] = seq[a:a + 5000].lower()
        c = b.rng.randrange(size // 2, size - 3000)
        seq[c:c + 2500] = b"N" * 2500
        start = len(b.buf)
        for off in (a, a + 5000, c, c + 2500):
            b.mark(start + off)
        b.line(bytes(seq))
        b.placed.update(["unwrapped_contig", "masked_run_in_unwrapped", "n_run_in_unwrapped"])
    for w in WIDTHS:
        b.line(b">w%d" % w)
        n = 2 * w + b.rng.randrange(1, w) if w < 65536 else w + 1000
        lines, _ = _wrap(b.bases(n), w)
        for i, l in enumerate(lines):
            b.line(l, mark=i < 2 or i >= len(lines) - 2)
        b.placed["width_%d" % w] += 1
        b.placed["short_last_line"] += 1
    b.line(b">tail")
    b.line(b.bases(1000))
    b.mark()
    b.buf += b.bases(77)                                 # last line without a newline
    b.placed["no_final_newline"] += 1
    return b.done()


def _stretch_bytes(rng, L, kind, newlines):
    alph = {"lower": b"acgtn", "N": b"N", "mixed": b"acgtnN"}[kind]
    s = bytearray(rng.choices(alph, k=L))
    if newlines:
        s[60::61] = b"\n" * len(range(60, L, 61))
        if kind == "mixed":                             # and blank lines
            for i in range(61 * 3, L, 61 * 7):
                s[i] = 10
    return s


def _framed_stretch(b, L, kind, newlines, align, carry_base):
    """A kept line whose last byte is an upper-case base (or 'n'), the stretch starting at `align` modulo SEG, and a line that
    starts with two bases: the one straddling window it gets takes its first byte from the kept line."""
    frame = b.bases(20) + (b.bases(1) if carry_base else b"n")
    b.pad_to(align, reserve=len(frame) + 1)
    b.line(frame)
    s = _stretch_bytes(b.rng, L, kind, newlines)
    start = len(b.buf)
    nl = [i for i in (s.find(b"\n"), s.rfind(b"\n")) if i >= 0]
    for i in nl:
        b.mark(start + i)
        b.mark(start + i + 1)
    b.line(bytes(s))
    b.line(b.bases(30))
    b.placed.update(["stretch_%d" % L, "stretch_" + kind, "stretch_newlines" if newlines else "stretch_one_line",
                     "carry_base" if carry_base else "carry_not_base"])


ALIGNS = {"align_on": 0, "align_before": SEG - 1, "align_after": 1}


def stretches(seed=2):
    """Base-free stretches of 4095..12289 bytes (lower case, N, or both with blank lines; with and without newlines inside),
    starting on, one byte before and one byte after a 4 KiB boundary, framed so that the carry into the next kept line is a base
    or is not.  Also the case the segment jump must not take: one kept line, whose only base is its last byte, inside a stretch
    that covers several whole segments on both sides of it."""
    b = _Builder(seed)
    b.line(b">stretches")
    i = 0
    for L in STRETCH_LENGTHS:
        for kind in ("lower", "N", "mixed"):
            for newlines in (True, False):
                name = list(ALIGNS)[i % 3]
                _framed_stretch(b, L, kind, newlines, ALIGNS[name], carry_base=(i // 3) % 2 == 0)
                b.placed[name] += 1
                i += 1
    for seg_of_base in (1, 2):
        frame = b.bases(21)
        b.pad_to(0, reserve=len(frame) + 1)
        b.line(frame)
        start = len(b.buf)
        s = _stretch_bytes(b.rng, 5 * SEG, "lower", True)
        j = s.index(b"\n", seg_of_base * SEG + 100)      # the last byte of a line in that segment is the only upper-case base
        s[j - 1] = ord(b.rng.choice([c for c in "ACGT" if ord(c) != frame[-1]]))
        for off in (j - 1, j, j + 1):
            b.mark(start + off)
        b.line(bytes(s))
        b.line(b.bases(30))
        b.placed["lone_base_line_in_stretch"] += 1
    return b.done()


def long_stretches(seed=3):
    """Base-free stretches of 100 kB and 1 MB."""
    b = _Builder(seed)
    b.line(b">long stretches")
    i = 0
    for kind in ("lower", "N", "mixed"):
        for newlines in (True, False):
            _framed_stretch(b, LONG_STRETCH_LENGTHS[0], kind, newlines, list(ALIGNS.values())[i % 3], carry_base=i % 2 == 0)
            i += 1
    _framed_stretch(b, LONG_STRETCH_LENGTHS[1], "mixed", True, 0, carry_base=True)
    return b.done()


def single_base_lines(seed=4):
    """Long lower-case lines whose only upper-case base is the first byte, the last byte, or one byte before or at a 4 KiB
    boundary: that one base decides whether the line is kept.  The line in front ends in a base and the line behind starts
    with two, so a wrong decision changes the straddling window.  One line is longer than the 64 KiB device piece."""
    b = _Builder(seed)
    b.line(b">single base")
    for name, L in (("single_base_first", 20_000), ("single_base_last", 20_000), ("single_base_before_seg", 20_000),
                    ("single_base_at_seg", 20_000), ("single_base_line_over_64k", 70_000)):
        b.line(b.bases(21))
        start = len(b.buf)
        s = bytearray(b.bases(L, b"acgtn"))
        if name in ("single_base_first", "single_base_line_over_64k"):
            k = 0
        elif name == "single_base_last":
            k = L - 1
        else:
            k = (-start) % SEG + SEG - (1 if name == "single_base_before_seg" else 0)
        s[k] = ord(b.rng.choice("ACGT"))
        b.mark(start + k)
        b.mark(start + k + 1)
        b.line(bytes(s))
        b.line(b.bases(30))
        b.placed[name] += 1
    return b.done()


def _header_text(rng, size, runs):
    if size == 1:
        return b">"
    out = bytearray(b">")
    while len(out) < size:
        if runs:
            out += bytes(rng.choices(b"ACGT", k=rng.randint(3, 300))) + rng.choice([b" ", b"|", b"n", b":"])
        else:
            out += rng.choice([b"chr", b" len=", b"|", b"Homo sapiens ", b"%d" % rng.randrange(10 ** 6)])
    return bytes(out[:size])


def headers(seed=5):
    """Headers of 1 byte to 70 kB, some full of ACGT runs, each between a line ending in a base and a line starting with two;
    a 3 kB header across a 4 KiB boundary; consecutive headers; '>' inside and at the end of a sequence line; ';' lines that
    hold GATTACA (the reference keeps and counts them); and a header as the last line, without a newline."""
    b = _Builder(seed)
    b.line(_header_text(b.rng, 40, True))
    for size in HEADER_SIZES:
        for runs in ((False, True) if size > 1 else (False,)):
            b.line(b.bases(50))
            b.line(_header_text(b.rng, size, runs))
            b.line(b.bases(50))
            b.placed["header_%d" % size] += 1
            b.placed["header_acgt_runs"] += runs
    b.line(b.bases(61))
    b.pad_to(SEG - 1000)
    b.line(_header_text(b.rng, 3000, True))
    b.line(b.bases(61))
    b.placed["header_over_seg"] += 1
    for k in range(3):
        b.line(_header_text(b.rng, b.rng.choice([1, 5, 40]), k == 1))
    b.line(b.bases(61))
    b.placed["consecutive_headers"] += 1
    b.line(b.bases(20) + b">" + b.bases(20))
    b.line(b.bases(20) + b">")
    b.line(b.bases(10))
    b.placed.update(["gt_in_sequence", "gt_last_byte"])
    b.line(b";comment GATTACA GATTACA")
    b.line(b.bases(10))
    b.line(b";GATTACA")
    b.placed["semicolon_comment"] += 2
    b.line(b.bases(40))
    b.mark()
    b.buf += _header_text(b.rng, 300, True)
    b.placed["header_last_no_newline"] += 1
    return b.done()


def line_ends(seed=6):
    """CRLF throughout a contig, mixed CRLF/LF, lone '\\r', trailing tabs and spaces, 10 000 blank lines and 10 000 one-base lines
    (more newlines per 2 KiB than the scan's per-warp newline queue takes), IUPAC codes in both cases, bytes 0x80-0xFF."""
    b = _Builder(seed)
    b.line(b">crlf", b"\r\n")
    for i in range(100):
        b.line(b.bases(60 if i < 99 else 17), b"\r\n")
    b.placed["crlf_contig"] += 1
    b.line(b">mixed", b"\r\n")
    for i in range(100):
        b.line(b.bases(b.rng.choice([1, 2, 3, 60])), b.rng.choice([b"\n", b"\r\n"]))
    b.placed["mixed_crlf_lf"] += 1
    for body in (b"AC\rGT", b"\rACGT", b"ACGT\r\r", b"\r", b"ACG\rT", b"TT\r\rAA"):
        b.line(body)
        b.line(b.bases(5))
        b.placed["lone_cr"] += 1
    for tail in (b" ", b"\t", b" \t ", b"\t\t"):
        b.line(b.bases(40) + tail)
        b.line(b.bases(40))
        b.placed["trailing_blanks"] += 1
    for name, unit in (("blank_lines_10000", lambda: b""), ("one_base_lines_10000", lambda: b.bases(1))):
        b.line(b.bases(33))
        for i in range(10_000):
            b.line(unit(), mark=i < 3 or i >= 9_997)
        b.line(b.bases(33))
        b.placed[name] += 1
    for _ in range(20):
        b.line(b.bases(b.rng.randint(2, 120), IUPAC))
        b.placed["iupac"] += 1
    high = bytes(range(0x80, 0x100))
    for _ in range(20):
        b.line(bytes(b.rng.choices(b"ACGT" * 8 + high, k=b.rng.randint(2, 120))))
        b.placed["high_bytes"] += 1
    b.line(b"ACGT" + high + b"ACGT")
    return b.done()


BUILDERS = {"unwrapped": unwrapped, "stretches": stretches, "long_stretches": long_stretches,
            "single_base_lines": single_base_lines, "headers": headers, "line_ends": line_ends}


@functools.lru_cache(maxsize=None)
def family(name):
    return BUILDERS[name]()


def cuts(bounds, n, reach=3):
    """Every boundary offset +-0..reach, inside [0, n]."""
    return sorted({c for x in bounds for c in range(x - reach, x + reach + 1) if 0 <= c <= n})


# ---------------------------------------------------------------------------------------------------------------- byte sweep
SWEEP_SLOT, SWEEP_PIECE = 64, 64 * 18          # a slot is 4 chunks; the pieces of one device call are SWEEP_PIECE bytes


def byte_sweep(v, seed=7):
    """ACGT and '\\n' everywhere except byte v, which sits at each of the 16 positions of a chunk (slot k: position k of the
    slot's second chunk) and at the two bytes in front of a device piece of SWEEP_PIECE bytes (the halo the scan takes from
    the bytes before the piece).  Returns (data, offsets of v)."""
    rng = random.Random(seed * 256 + v)
    slots = 3 * SWEEP_PIECE // SWEEP_SLOT
    buf = bytearray(rng.choices(b"ACGT", k=slots * SWEEP_SLOT))
    buf[SWEEP_SLOT - 1::SWEEP_SLOT] = b"\n" * slots       # 63-base lines; v stays inside a line
    where = [k * SWEEP_SLOT + 16 + k for k in range(16)]
    where += [SWEEP_PIECE - 2, 2 * SWEEP_PIECE - 1]       # halo -2 of piece 1, halo -1 of piece 2
    buf[SWEEP_PIECE - 1] = ord("G")                      # the lines run on across both piece starts
    for w in where:
        buf[w] = v
    return bytes(buf), where


# ---------------------------------------------------------------------------------------------------------------- index inputs
def index_files(seed=8):
    """Small FASTA texts for the .fai-style index and the BED gather: CRLF, unwrapped, one width per contig (50..4097),
    no final newline, and blank lines between records (LF and CRLF).  [(name, data)]"""
    rng = random.Random(seed)

    def contig(name, n, width, end=b"\n", blank_after=0):
        seq = bytes(rng.choices(b"ACGTacgtN", weights=[8, 8, 8, 8, 1, 1, 1, 1, 1], k=n))
        body = b"".join(seq[i:i + width] + end for i in range(0, n, width))
        return b">" + name + b" desc" + end + body + end * blank_after

    out = [
        ("crlf", b"".join(contig(b"c%d" % k, rng.randint(500, 5000), 60, b"\r\n") for k in range(3))),
        ("unwrapped", b"".join(contig(b"u%d" % k, n, n) for k, n in enumerate((3000, 70_000, 12_289)))),
        ("mixed_widths", b"".join(contig(b"w%d" % w, rng.randint(3 * w, 5 * w), w) for w in (50, 61, 80, 1000, 4097))),
        ("blank_lines_lf", b"".join(contig(b"b%d" % k, rng.randint(300, 3000), 60, b"\n", k + 1) for k in range(3))),
        ("blank_lines_crlf", b"".join(contig(b"r%d" % k, rng.randint(300, 3000), 60, b"\r\n", k + 1) for k in range(3))),
    ]
    nf = b"".join(contig(b"n%d" % k, rng.randint(300, 3000), 70) for k in range(3))
    out.append(("no_final_newline", nf.rstrip(b"\n")))
    out.append(("crlf_unwrapped_no_final_newline", contig(b"x", 9000, 9000, b"\r\n").rstrip(b"\r\n")))
    return out


# Records whose lines do not share the first line's width.  The index once read positions after a blank line inside a record
# from the wrong bytes (the CRLF case gave 'A' for a 'G' at base 6), so it must refuse them.  [(name, data)]
UNEVEN_RECORDS = [
    ("blank_line_inside_crlf", b">r desc\r\nACGT\r\n\r\nACGT\r\nGG\r\n>s\r\nTTGCA\r\n"),
    ("blank_line_inside_lf", b">r desc\nACGT\n\nACGT\nGG\n>s\nTTGCA\n"),
    ("short_line_inside", b">r\nACGT\nAC\nACGT\n>s\nTTGCA\n"),
    ("last_line_longer", b">s\nTTGCA\n>r\nACGT\nACGTA\n"),
    ("two_short_last_lines", b">r\nACGT\nA\nC\n"),
    ("lf_then_crlf", b">r\nACGT\nACGT\r\nAC\n"),
]


# ---------------------------------------------------------------------------------------------------------------- GRCh38 shape
def grch38_like(seed=9, mb=64):
    """A `mb` MB genome in GRCh38's layout: 60-column contigs and one contig written as one line; 10 kb N blocks at every contig
    end and an N block of 1-5 Mb in the middle; soft-masked runs of 300-50 000 bases; one 10 kB header.  Returns
    (data, cuts): a handful of offsets inside the long runs."""
    rng = np.random.default_rng(seed)
    total = mb << 20
    sizes = [int(total * f) for f in (0.45, 0.2, 0.3)]         # 60-col, unwrapped, 60-col (the header lines are extra)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    parts, cut_at, off = [], [], 0
    for k, n in enumerate(sizes):
        seq = lut[rng.integers(0, 4, n, dtype=np.uint8)]
        seq[:10_000] = ord("N")
        seq[-10_000:] = ord("N")
        nb = int(rng.integers(1_000_000, 5_000_001)) if k != 1 else 1_000_000
        a = n // 2 - nb // 2
        seq[a:a + nb] = ord("N")
        masked = []
        pos = 20_000
        while pos < n - 80_000:
            ln = int(rng.integers(300, 50_001))
            if not (a - ln <= pos <= a + nb):
                seq[pos:pos + ln] |= 0x20
                masked.append((pos, ln))
            pos += ln + int(rng.integers(1000, 200_000))
        hdr = b">chr%d  AC:CM0006%02d.2  gi|568336%03d|gb|CM0006%02d.2| Homo sapiens chromosome %d, GRCh38 reference primary assembly\n" % (
            k + 1, k, k, k, k + 1)
        if k == 2:
            hdr = hdr[:-1] + b" " + bytes(rng.choice(lut, 10_000 - len(hdr))) + b"\n"
        parts.append(hdr)
        off += len(hdr)
        if k == 1:
            body = seq.tobytes() + b"\n"
            to_byte = lambda p: off + p
        else:
            rows = -(-n // 60)
            arr = np.full(rows * 61, ord("\n"), dtype=np.uint8).reshape(rows, 61)
            flat = np.full(rows * 60, 0, dtype=np.uint8)
            flat[:n] = seq
            arr[:, :60] = flat.reshape(rows, 60)
            body = arr.reshape(-1)[:n + (n - 1) // 60].tobytes() + b"\n"
            to_byte = lambda p: off + p + p // 60
        m = masked[len(masked) // 2]
        for p in (a + 17, a + nb // 2, a + nb - 5, m[0] + m[1] // 2, 5_000):
            cut_at.append(to_byte(p))
        parts.append(body)
        off += len(body)
    return b"".join(parts), sorted(cut_at)
