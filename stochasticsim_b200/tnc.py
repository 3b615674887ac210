"""Trinucleotide-context scan: Python face of ssb_tnc_* (replaces tncCountsProfile.c:391-483)."""
import ctypes as C
import numpy as np
from ._lib import lib, check, TncCarry

OUT_ORDER = ["ACA", "ACC", "ACG", "ACT", "ATA", "ATC", "ATG", "ATT", "CCA", "CCC", "CCG", "CCT", "CTA", "CTC", "CTG", "CTT",
             "GCA", "GCC", "GCG", "GCT", "GTA", "GTC", "GTG", "GTT", "TCA", "TCC", "TCG", "TCT", "TTA", "TTC", "TTG", "TTT"]


def _buf(data):
    """bytes / bytearray / numpy uint8 -> (address, length, keepalive)."""
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data, dtype=np.uint8)
        return a.ctypes.data, a.size, a
    b = bytes(data)
    keep = C.create_string_buffer(b, len(b)) if len(b) else C.create_string_buffer(1)
    return C.addressof(keep), len(b), keep


def count_host(ctx, data, carry_in=None, want_carry=False):
    """64 context counts (index 16a+4b+c, A<C<G<T) of a host-resident FASTA piece."""
    L = lib()
    addr, n, keep = _buf(data)
    out = np.zeros(64, dtype=np.int64)
    cout = TncCarry()
    check(L.ssb_tnc_count_host(ctx.handle, addr, n, C.byref(carry_in) if carry_in is not None else None,
                               C.byref(cout), out.ctypes.data_as(C.POINTER(C.c_int64))), ctx.handle)
    return (out, cout) if want_carry else out


def count_device(ctx, d_ptr, n, d_counts, carry_in=None, want_carry=False):
    """Adds the windows of the device-resident piece [d_ptr, d_ptr+n) to the 64 int64 device counters."""
    L = lib()
    cout = TncCarry()
    check(L.ssb_tnc_count_device(ctx.handle, d_ptr, n, C.byref(carry_in) if carry_in is not None else None,
                                 C.byref(cout) if want_carry else None, d_counts), ctx.handle)
    return cout if want_carry else None


def carry_after(data, carry_in=None):
    """Scanner state after consuming `data` (host only, counts nothing): used to cut shards."""
    L = lib()
    addr, n, keep = _buf(data)
    out = TncCarry()
    check(L.ssb_tnc_carry_after(addr, n, C.byref(carry_in) if carry_in is not None else None, C.byref(out)))
    return out


class FastaContig(C.Structure):
    _fields_ = [("seq_off", C.c_uint64), ("len", C.c_int64), ("line_bases", C.c_uint32), ("line_bytes", C.c_uint32)]


class BedInterval(C.Structure):
    _fields_ = [("contig", C.c_int32), ("reserved", C.c_int32), ("start", C.c_int64), ("end", C.c_int64)]


def fasta_index(data):
    """[(name, FastaContig)] -- ssb_fasta_index (host): a .fai-style index of a FASTA text."""
    L = lib()
    L.ssb_fasta_index.restype = C.c_int
    L.ssb_fasta_index.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(FastaContig), C.POINTER(C.c_char_p), C.POINTER(C.c_uint32), C.c_size_t, C.POINTER(C.c_size_t)]
    addr, n, keep = _buf(data)
    cnt = C.c_size_t()
    check(L.ssb_fasta_index(addr, n, None, None, None, 0, C.byref(cnt)))
    k = cnt.value
    arr = (FastaContig * max(1, k))()
    nl = (C.c_uint32 * max(1, k))()
    names = (C.c_void_p * max(1, k))()
    check(L.ssb_fasta_index(addr, n, arr, C.cast(names, C.POINTER(C.c_char_p)), nl, k, C.byref(cnt)))
    out = []
    for i in range(k):
        name = C.string_at(names[i], nl[i]).decode()
        c = FastaContig(arr[i].seq_off, arr[i].len, arr[i].line_bases, arr[i].line_bytes)
        out.append((name, c))
    return out


def _index_and_intervals(index, intervals):
    """ctypes arrays of an index ([(name, FastaContig)]) and of intervals ((contig index, start, end) rows, or an int64 array of them)."""
    carr = (FastaContig * max(1, len(index)))(*[c for _, c in index])
    if isinstance(intervals, np.ndarray):                      # structured rows (contig, start, end) as int64 columns
        iv = (BedInterval * max(1, len(intervals)))()
        flat = np.zeros((len(intervals), 3), dtype=np.int64)
        flat[:, 0] = intervals[:, 0]; flat[:, 1] = intervals[:, 1]; flat[:, 2] = intervals[:, 2]
        raw = np.zeros(len(intervals), dtype=[("contig", "<i4"), ("reserved", "<i4"), ("start", "<i8"), ("end", "<i8")])
        raw["contig"], raw["start"], raw["end"] = flat[:, 0], flat[:, 1], flat[:, 2]
        C.memmove(iv, raw.ctypes.data, raw.nbytes)
    else:
        iv = (BedInterval * max(1, len(intervals)))(*[BedInterval(c, 0, a, b) for c, a, b in intervals])
    return carr, iv


_IV_ARGS = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(FastaContig), C.c_size_t, C.POINTER(BedInterval), C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p]


def count_bed_device(ctx, d_ptr, n, index, intervals, d_counts, first=0, last=None):
    """Adds the windows of BED intervals [first, last) (in the order given; (contig index, start, end)) to the 64 device counters."""
    L = lib()
    L.ssb_tnc_count_bed_device.restype = C.c_int
    L.ssb_tnc_count_bed_device.argtypes = _IV_ARGS
    carr, iv = _index_and_intervals(index, intervals)
    last = len(intervals) if last is None else last
    check(L.ssb_tnc_count_bed_device(ctx.handle, d_ptr, n, carr, len(index), iv, len(intervals), first, last, d_counts), ctx.handle)


def count_intervals_device(ctx, d_ptr, n, index, intervals, d_rows, first=0, last=None):
    """Adds the windows of each BED interval i in [first, last), on its own, to row i - first of the device int64 rows
    d_rows[(last - first) * 64] (ssb_tnc_count_intervals_device: no straddling windows, so rows are independent of BED order)."""
    L = lib()
    L.ssb_tnc_count_intervals_device.restype = C.c_int
    L.ssb_tnc_count_intervals_device.argtypes = _IV_ARGS
    carr, iv = _index_and_intervals(index, intervals)
    last = len(intervals) if last is None else last
    check(L.ssb_tnc_count_intervals_device(ctx.handle, d_ptr, n, carr, len(index), iv, len(intervals), first, last, d_rows), ctx.handle)


_fold_src = None


def fold32(counts):
    """(..., 64) context counts -> (..., 32): the reference's output lines (ssb_tnc_fold32: context + reverse complement, OUT_ORDER)."""
    global _fold_src
    if _fold_src is None:
        # each output line is the sum of two contexts; read which from ssb_tnc_fold32 itself, one context at a time
        L = lib()
        L.ssb_tnc_fold32.restype = None
        L.ssb_tnc_fold32.argtypes = [C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        src = [[] for _ in range(32)]
        e, o = np.zeros(64, dtype=np.int64), np.zeros(32, dtype=np.int64)
        for k in range(64):
            e[:] = 0
            e[k] = 1
            L.ssb_tnc_fold32(e.ctypes.data_as(C.POINTER(C.c_int64)), o.ctypes.data_as(C.POINTER(C.c_int64)))
            for j in np.flatnonzero(o):
                src[j].append(k)
        _fold_src = np.array(src, dtype=np.int64).T               # (2, 32)
    c = np.asarray(counts, dtype=np.int64)
    return c[..., _fold_src[0]] + c[..., _fold_src[1]]


def format_counts(counts64):
    """The reference's 32-line stdout (tncCountsProfile.c:452-483)."""
    L = lib()
    c = np.ascontiguousarray(counts64, dtype=np.int64)
    buf = C.create_string_buffer(4096)
    w = L.ssb_tnc_format(c.ctypes.data_as(C.POINTER(C.c_int64)), buf, 4096)
    if w < 0:
        check(w)
    return buf.raw[:w].decode()
