"""The TNC path on the FASTA shapes real genomes have (tests/fasta_shapes.py): unwrapped contigs and lines wider than a 4 KiB
segment, base-free stretches on and next to segment boundaries, long lines with a single upper-case base, headers up to 70 kB,
CRLF, IUPAC codes and high bytes, runs of 10 000 blank lines, every byte value at every position of a chunk, and a 64 MB
genome in GRCh38's layout.

CPU: every family places its shapes; the host state transition composes at every boundary offset +-0..3; shards cut there add
up to the whole-file count; the .fai-style index matches the text on CRLF, unwrapped, mixed-width, no-final-newline files and
files with blank lines between records, and refuses a record whose lines are not all as wide as its first.

GPU (marked `gpu`): counts equal to the oracle (and to oracle/_ref/tncCountsProfile when it is built) through one device call,
device pieces of 32 bytes to 64 KiB, host chunks, carry-chained calls cut at every boundary offset +-0..3 (the state after
every piece must equal ssb_tnc_carry_after of the prefix), the CLI, the BED mode and, when two devices are present, two GPUs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import fasta_cases as fc
import fasta_shapes as fs
import oracle_bind as ob
import stochasticsim_b200 as ssb
from stochasticsim_b200 import tnc

EXE = os.path.join(ob.ROOT, "stochasticsim_b200", "lib", "tncCountsProfile")
SSB_E_FORMAT = -5


def _view(data):
    return np.frombuffer(data, dtype=np.uint8)


@pytest.fixture(scope="module")
def grch38():
    return fs.grch38_like()


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", fs.FAMILIES)
def test_every_family_places_its_shapes(name):
    data, bounds, placed = fs.family(name)
    assert not [s for s in fs.FAMILY_SHAPES[name] if placed[s] == 0], placed
    assert bounds == sorted(set(bounds)) and 0 in bounds and bounds[-1] == len(data)
    assert b"\0" not in data
    if name == "stretches":                              # the stretches start on and next to 4 KiB boundaries, as named
        assert placed["align_on"] and placed["align_before"] and placed["align_after"]


def test_byte_sweep_places_every_byte_at_every_chunk_position():
    for v in range(1, 256):
        data, where = fs.byte_sweep(v)
        assert sorted(w % 16 for w in where[:16]) == list(range(16))
        assert where[16] % fs.SWEEP_PIECE == fs.SWEEP_PIECE - 2 and where[17] % fs.SWEEP_PIECE == fs.SWEEP_PIECE - 1
        rest = bytearray(data)
        for w in where:
            assert rest[w] == v
            rest[w] = ord("A")
        assert set(rest) <= set(b"ACGT\n")
        for w in where:                                  # v never sits next to a newline: a misread byte changes a window
            assert data[w - 1] != 10 and data[w + 1] != 10


@pytest.mark.parametrize("name", fs.FAMILIES)
def test_carry_after_composes_at_every_boundary(name):
    """carry_after(a + b) == carry_after(b, carry_after(a)) at every boundary offset +-0..3."""
    data, bounds, _ = fs.family(name)
    v = _view(data)
    st, prev = None, 0
    for c in fs.cuts(bounds, len(data)):
        st = tnc.carry_after(v[prev:c], st)
        assert st.as_tuple() == tnc.carry_after(v[:c]).as_tuple(), c
        prev = c
    assert tnc.carry_after(v[prev:], st).as_tuple() == tnc.carry_after(v).as_tuple()


@pytest.mark.parametrize("name", fs.FAMILIES)
def test_shards_cut_at_every_boundary_add_up(name):
    data, bounds, _ = fs.family(name)
    cuts = [0] + [c for c in fs.cuts(bounds, len(data)) if 0 < c < len(data)] + [len(data)]
    total = sum(fc.shard_counts_with_carry(data, a, b) for a, b in zip(cuts, cuts[1:]))
    assert np.array_equal(total, ob.tnc_counts(data))


def test_grch38_shaped_shards_add_up(grch38):
    data, cut_at = grch38
    want = ob.tnc_counts(data)
    assert int(want.sum()) > 0
    for c in cut_at:
        assert np.array_equal(fc.shard_counts_with_carry(data, 0, c) + fc.shard_counts_with_carry(data, c, len(data)), want), c
    v = _view(data)
    st, prev = None, 0
    for c in cut_at:
        st = tnc.carry_after(v[prev:c], st)
        prev = c
    assert tnc.carry_after(v[prev:], st).as_tuple() == tnc.carry_after(v).as_tuple()


@pytest.mark.parametrize("name,data", fs.index_files(), ids=[n for n, _ in fs.index_files()])
def test_fasta_index_matches_the_text(name, data):
    """Every base of every contig is where the index says, and the lengths are the contigs' (blank lines and line terminators
    after the last base are not part of a contig)."""
    from test_tnc_bed import _contig_seqs
    seqs = _contig_seqs(data)
    idx = tnc.fasta_index(data)
    assert [(n, c.len) for n, c in idx] == [(n, len(s)) for n, s in seqs]
    v = _view(data)
    for (n, c), (_, s) in zip(idx, seqs):
        assert c.line_bytes - c.line_bases == (2 if b"\r\n" in data else 1) or c.line_bytes == c.line_bases == c.len
        p = np.arange(c.len, dtype=np.int64)
        at = c.seq_off + p + (p // c.line_bases) * (c.line_bytes - c.line_bases)
        assert np.array_equal(v[at], _view(s)), n


@pytest.mark.parametrize("name,data", fs.UNEVEN_RECORDS, ids=[n for n, _ in fs.UNEVEN_RECORDS])
def test_fasta_index_refuses_records_of_uneven_lines(name, data):
    with pytest.raises(ssb.SSBError) as err:
        tnc.fasta_index(data)
    assert err.value.code == SSB_E_FORMAT


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctx():
    c = ssb.Context(0)
    yield c
    c.close()


class _Dev:
    """One device buffer and one set of 64 counters: count_device over host pieces copied to the buffer start."""

    def __init__(self, ctx, cap):
        self.ctx, self.cap = ctx, max(cap, 1) + 64
        self.d = ctx.dev_alloc(self.cap)
        self.dc = ctx.dev_alloc(64 * 8)

    def close(self):
        self.ctx.dev_free(self.d)
        self.ctx.dev_free(self.dc)

    def counts(self, data, carry=None, want_carry=False, zero=True):
        if zero:
            self.ctx.memset(self.dc, 0, 64 * 8)
        if len(data):
            buf = C.create_string_buffer(bytes(data), len(data))
            self.ctx.h2d(self.d, C.addressof(buf), len(data))
        cout = tnc.count_device(self.ctx, self.d, len(data), self.dc, carry_in=carry, want_carry=want_carry)
        return cout

    def read(self):
        out = np.zeros(64, dtype=np.int64)
        self.ctx.d2h(out.ctypes.data, self.dc, 64 * 8)
        self.ctx.sync()
        return out


def _count(ctx, data):
    d = _Dev(ctx, len(data))
    try:
        d.counts(data)
        return d.read()
    finally:
        d.close()


def _pieces_for(n):
    return [p for p in (32, 48, 1008, 4096, 12_304, 65_536) if p < n and n // p < 40_000]


@pytest.mark.gpu
@pytest.mark.parametrize("name", fs.FAMILIES)
def test_one_call_and_device_pieces(ctx, monkeypatch, name):
    """One count_device call; then the same buffer in device pieces of 32 bytes to 64 KiB (the scans run ahead of the fix-ups,
    two exception lists alternate); then, for boundaries spread over the file, a piece size and a prefix of blank lines (which
    changes no count) chosen so that a piece starts right at that boundary."""
    data, bounds, _ = fs.family(name)
    want = ob.tnc_counts(data)
    assert np.array_equal(_count(ctx, data), want)
    for piece in _pieces_for(len(data)):
        monkeypatch.setenv("SSB_TNC_PIECE", str(piece))
        assert np.array_equal(_count(ctx, data), want), piece
    sizes = (4096, 12_304, 65_536)
    step = max(1, len(bounds) // 48)
    for k, x in enumerate(bounds[1:-1:step]):
        piece = sizes[k % 3]
        monkeypatch.setenv("SSB_TNC_PIECE", str(piece))
        padded = b"\n" * ((-x) % piece) + data
        assert np.array_equal(_count(ctx, padded), want), (piece, x)


@pytest.mark.gpu
@pytest.mark.parametrize("name", fs.FAMILIES)
def test_host_chunks(ctx, monkeypatch, name):
    data, _, _ = fs.family(name)
    want = ob.tnc_counts(data)
    for chunk in (64, 4096, 65_536 + 32, 1 << 20):
        monkeypatch.setenv("SSB_TNC_CHUNK", str(chunk))
        got, carry = tnc.count_host(ctx, data, want_carry=True)
        assert np.array_equal(got, want), chunk
        assert carry.as_tuple() == tnc.carry_after(data).as_tuple(), chunk


@pytest.mark.gpu
@pytest.mark.parametrize("name", fs.FAMILIES)
def test_carry_chain_cut_at_every_boundary(ctx, name):
    """count_device calls chained through ssb_tnc_carry, cut at every boundary offset +-0..3: the device state after every piece
    equals ssb_tnc_carry_after of the prefix, and the pieces add up to the whole-file count."""
    data, bounds, _ = fs.family(name)
    v = _view(data)
    d = _Dev(ctx, len(data))
    try:
        ctx.memset(d.dc, 0, 64 * 8)
        carry, prev = None, 0
        for c in fs.cuts(bounds, len(data)) + [len(data)]:
            if c == prev and c:
                continue
            carry = d.counts(data[prev:c], carry=carry, want_carry=True, zero=False)
            assert carry.as_tuple() == tnc.carry_after(v[:c]).as_tuple(), (c, carry.as_tuple(), tnc.carry_after(v[:c]).as_tuple())
            prev = c
        assert np.array_equal(d.read(), ob.tnc_counts(data))
    finally:
        d.close()


@pytest.mark.gpu
def test_byte_sweep(ctx, monkeypatch):
    """Every byte value 1..255 at every position of a chunk and as the two bytes in front of a device piece, one call per value:
    the exactness test of the fast path (one table lookup keyed by (b >> 1) & 7, shared by many byte values) and its 2-byte halo."""
    monkeypatch.setenv("SSB_TNC_PIECE", str(fs.SWEEP_PIECE))
    d = _Dev(ctx, 3 * fs.SWEEP_PIECE)
    try:
        bad = []
        for v in range(1, 256):
            data, _ = fs.byte_sweep(v)
            d.counts(data)
            if not np.array_equal(d.read(), ob.tnc_counts(data)):
                bad.append(v)
        assert not bad, "byte values counted wrong: %s" % [hex(v) for v in bad]
    finally:
        d.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", fs.FAMILIES)
def test_cli(tmp_path, ref_dir, name):
    data, _, _ = fs.family(name)
    p = tmp_path / "f.fa"
    p.write_bytes(data)
    got = subprocess.run([EXE, str(p)], capture_output=True)
    assert got.returncode == 0, got.stderr
    assert got.stdout.decode() == ob.tnc_text(ob.tnc_counts(data))
    if ref_dir:
        assert got.stdout == subprocess.run([os.path.join(ref_dir, "tncCountsProfile"), str(p)], capture_output=True).stdout


@pytest.mark.gpu
def test_cli_two_devices_when_present(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one device")
    for name in fs.FAMILIES:
        data, _, _ = fs.family(name)
        p = tmp_path / "f.fa"
        p.write_bytes(data)
        got = subprocess.run([EXE, str(p)], capture_output=True, env=dict(os.environ, SSB_GPUS="2"))
        assert got.returncode == 0, got.stderr
        assert got.stdout.decode() == ob.tnc_text(ob.tnc_counts(data)), name


@pytest.mark.gpu
def test_grch38_shaped(ctx, monkeypatch, grch38, ref_dir, tmp_path):
    """One call over the whole 64 MB, the same in 1 MiB device pieces and through the host chunks, and calls chained at cuts
    inside the N blocks, the unwrapped contig and a soft-masked run."""
    data, cut_at = grch38
    want = ob.tnc_counts(data)
    assert np.array_equal(_count(ctx, data), want)
    monkeypatch.setenv("SSB_TNC_PIECE", str(1 << 20))
    assert np.array_equal(_count(ctx, data), want)
    monkeypatch.delenv("SSB_TNC_PIECE")
    assert np.array_equal(tnc.count_host(ctx, data), want)
    v = _view(data)
    d = _Dev(ctx, len(data))
    try:
        ctx.memset(d.dc, 0, 64 * 8)
        carry, prev = None, 0
        for c in cut_at + [len(data)]:
            carry = d.counts(data[prev:c], carry=carry, want_carry=True, zero=False)
            assert carry.as_tuple() == tnc.carry_after(v[:c]).as_tuple(), c
            prev = c
        assert np.array_equal(d.read(), want)
    finally:
        d.close()
    if ref_dir:
        p = tmp_path / "g.fa"
        p.write_bytes(data)
        out = subprocess.run([os.path.join(ref_dir, "tncCountsProfile"), str(p)], capture_output=True, check=True).stdout.decode()
        assert out == ob.tnc_text(want)


# ------------------------------------------------------------------------------------------------ GPU, BED mode
def _bed_counts(ctx, data, idx, intervals, ranges):
    import torch
    dev = torch.from_numpy(_view(data).copy()).cuda()
    total = np.zeros(64, dtype=np.int64)
    for a, b in ranges:
        cnt = torch.zeros(64, dtype=torch.int64, device="cuda")
        tnc.count_bed_device(ctx, dev.data_ptr(), dev.numel(), idx, intervals, cnt.data_ptr(), a, b)
        ctx.sync()
        total += cnt.cpu().numpy()
    return total


def _line_crossing_intervals(rng, seqs, widths, n):
    """Intervals that start a few bases before a line break and end a few after (or several lines further on)."""
    out = []
    for _ in range(n):
        c = rng.randrange(len(seqs))
        L, w = len(seqs[c][1]), widths[c]
        if L < 8:
            continue
        brk = w * rng.randint(1, max(1, (L - 1) // w)) if w < L else L // 2
        a = max(0, brk - rng.randint(1, 4))
        e = min(L, brk + rng.choice([1, 2, 3, w + 5, 3 * w]))
        out.append((c, a, max(e, a + 1)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,data", fs.index_files(), ids=[n for n, _ in fs.index_files()])
def test_bed_on_index_files(ctx, ref_dir, tmp_path, name, data):
    """Intervals across line breaks in CRLF, unwrapped, mixed-width and no-final-newline files; the whole range and a partition of
    it (each part's context search skips back over the intervals before it)."""
    import random
    from test_tnc_bed import _contig_seqs, virtual_fasta
    rng = random.Random(len(data))
    seqs = _contig_seqs(data)
    idx = tnc.fasta_index(data)
    iv = _line_crossing_intervals(rng, seqs, [c.line_bases or 1 for _, c in idx], 400)
    iv += [(c, 0, len(s)) for c, (_, s) in enumerate(seqs)]             # whole contigs (one line each in `unwrapped`)
    want = ob.tnc_counts(virtual_fasta(data, iv))
    assert np.array_equal(_bed_counts(ctx, data, idx, iv, [(0, len(iv))]), want)
    cuts = sorted({0, len(iv)} | {rng.randrange(len(iv)) for _ in range(5)})
    assert np.array_equal(_bed_counts(ctx, data, idx, iv, list(zip(cuts, cuts[1:]))), want)


@pytest.mark.gpu
def test_bed_context_skips_base_free_intervals(ctx):
    """A range whose nearest earlier interval with an upper-case base lies behind several base-free ones (lower case, N, empty)."""
    import random
    from test_tnc_bed import _contig_seqs, virtual_fasta
    rng = random.Random(77)
    seq = bytearray(rng.choices(b"ACGT", k=30_000))
    seq[10_000:20_000] = bytes(rng.choices(b"acgtnN", k=10_000))
    data = b">m\n" + b"".join(bytes(seq[i:i + 60]) + b"\n" for i in range(0, len(seq), 60))
    idx = tnc.fasta_index(data)
    assert _contig_seqs(data)[0][1] == bytes(seq)
    for k in (1, 5, 40):
        iv = [(0, 9_000, 9_100), (0, 9_995, 10_000)]                    # the second ends in a base: the context record
        iv += [(0, a, a + rng.randint(0, 200)) for a in sorted(rng.randrange(10_000, 19_800) for _ in range(k))]
        iv += [(0, 20_000, 20_100), (0, 25_000, 25_050)]
        want = ob.tnc_counts(virtual_fasta(data, iv))
        first = len(iv) - 2
        parts = _bed_counts(ctx, data, idx, iv, [(0, first), (first, len(iv))])
        assert np.array_equal(parts, want), k


@pytest.mark.gpu
def test_bed_blank_lines_between_records(ctx):
    """Blank lines after a record's last line: every interval, up to the contig's end, gives the bases the text holds."""
    from test_tnc_bed import _contig_seqs, virtual_fasta
    for name, data in fs.index_files():
        if not name.startswith("blank_lines"):
            continue
        seqs = _contig_seqs(data)
        idx = tnc.fasta_index(data)
        for c, (_, s) in enumerate(seqs):
            L = len(s)
            for a, e in [(0, L), (L - 1, L), (L - 3, L)] + [(a, a + 2) for a in range(L - 70, L - 2, 7)]:
                iv = [(c, a, e), ((c + 1) % len(seqs), 0, 3)]
                assert np.array_equal(_bed_counts(ctx, data, idx, iv, [(0, 2)]), ob.tnc_counts(virtual_fasta(data, iv))), (name, iv)


@pytest.mark.gpu
@pytest.mark.parametrize("name,data", fs.UNEVEN_RECORDS, ids=[n for n, _ in fs.UNEVEN_RECORDS])
def test_bed_cli_refuses_records_of_uneven_lines(tmp_path, name, data):
    (tmp_path / "g.fa").write_bytes(data)
    (tmp_path / "t.bed").write_text("s\t0\t3\n" if b">s" in data else "r\t0\t3\n")
    got = subprocess.run([EXE, str(tmp_path / "g.fa"), str(tmp_path / "t.bed")], capture_output=True)
    assert got.returncode == 3 and b"not all as wide" in got.stderr, got
