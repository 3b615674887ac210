"""Numpy restatement of the per-interval trinucleotide counts (ssb_tnc_count_intervals_device), shared by the tests and
tools/tnc_intervals_probe.py.

Row i is what the reference counts on the FASTA `bedtools getfasta` writes for interval i alone (one header line, the bases on
one line).  For one line that reduces to a closed form: a window counts at every position p in [start, end-2) where bases p, p+1
and p+2 are all upper-case A/C/G/T.  test_tnc_intervals.py pins this form to the oracle; the large GPU cases then check against it."""
import numpy as np

_CODE = np.full(256, -1, dtype=np.int8)
_CODE[np.frombuffer(b"ACGT", dtype=np.uint8)] = np.arange(4)


def contig_bases(text, c, start, end):
    """Bases [start, end) of contig `c` (a FastaContig) read from the genome text (uint8 array) through its line geometry."""
    p = np.arange(start, end, dtype=np.int64)
    return text[c.seq_off + p + (p // max(1, c.line_bases)) * (c.line_bytes - c.line_bases)]


def window_index(bases):
    """Per window start p: 16a + 4b + c of bases p, p+1, p+2 (A<C<G<T), or -1 when one of them is not an upper-case A/C/G/T."""
    k = _CODE[np.asarray(bases, dtype=np.uint8)]
    if len(k) < 3:
        return np.zeros(0, dtype=np.int8)
    a, b, c = k[:-2], k[1:-1], k[2:]
    return np.where((a >= 0) & (b >= 0) & (c >= 0), 16 * a + 4 * b + c, -1)


def interval_row(text, c, start, end):
    w = window_index(contig_bases(text, c, start, end))
    return np.bincount(w[w >= 0], minlength=64).astype(np.int64)


def closed_form_rows(text, index, intervals):
    """(len(intervals), 64) rows for (contig index, start, end) intervals over the genome text with index [(name, FastaContig)]."""
    text = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else text
    out = np.zeros((len(intervals), 64), dtype=np.int64)
    for i, (ci, a, b) in enumerate(intervals):
        out[i] = interval_row(text, index[ci][1], a, b)
    return out


def tiled_rows(bases, tile):
    """Rows of the tiling [0, t), [t, 2t), ... of one contig (the last tile may be shorter), from the contig's bases."""
    n_tiles = -(-len(bases) // tile)
    w = window_index(bases)
    p = np.arange(len(w))
    keep = (w >= 0) & (p % tile < tile - 2)              # the window's three bases lie in one tile
    return np.bincount((p[keep] // tile) * 64 + w[keep], minlength=n_tiles * 64).reshape(n_tiles, 64).astype(np.int64)


def wrap(seq, width, eol=b"\n"):
    """Contig bases (uint8 array) as FASTA lines of `width` bases, the last one shorter, each ended by `eol`."""
    seq = np.asarray(seq, dtype=np.uint8)
    rows = -(-len(seq) // width)
    arr = np.zeros((rows, width + len(eol)), dtype=np.uint8)
    flat = np.zeros(rows * width, dtype=np.uint8)
    flat[:len(seq)] = seq
    arr[:, :width] = flat.reshape(rows, width)
    arr[:, width:] = np.frombuffer(eol, dtype=np.uint8)
    last = len(seq) - (rows - 1) * width
    out = arr.reshape(-1)[:(rows - 1) * (width + len(eol)) + last]
    return out.tobytes() + eol
