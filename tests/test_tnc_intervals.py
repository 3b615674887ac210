"""Per-interval trinucleotide counts (ssb_tnc_count_intervals_device, tnc.count_intervals_device, tncCountsProfile --per-interval).

Row i is by definition what the reference counts on the FASTA `bedtools getfasta` writes for interval i alone.  CPU: the numpy
closed form of interval_cases.py against the oracle on that FASTA, and the 32-line fold.  GPU: rows against the oracle, partitions,
accumulation, the relation to the BED-mode total, genome-scale shapes and 64-bit offsets against the closed form, refusals, the CLI."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import fasta_cases as fc
import interval_cases as ic
import oracle_bind as ob
import stochasticsim_b200 as ssb
from stochasticsim_b200 import tnc
from test_tnc_bed import _contig_seqs, virtual_fasta

ROOT = ob.ROOT
EXE = os.path.join(ROOT, "stochasticsim_b200", "lib", "tncCountsProfile")
IUPAC = b"RYKMSWBDHVN"


def _genome(rng, n_bases, width, contigs, crlf=False, iupac=0):
    data = fc.genome_like(rng, n_bases, width=width, n_block=(n_bases // contigs // 5, n_bases // contigs // 4), lower_runs=3, contigs=contigs)
    if iupac:                                            # scattered IUPAC codes inside sequence lines
        b, seq_pos, o = bytearray(data), [], 0
        for line in data.split(b"\n"):
            if not line.startswith(b">"):
                seq_pos += [o + j for j, ch in enumerate(line) if ch in b"ACGT"]
            o += len(line) + 1
        for i in rng.sample(seq_pos, min(iupac, len(seq_pos))):
            b[i] = rng.choice(IUPAC)
        data = bytes(b)
    return data.replace(b"\n", b"\r\n") if crlf else data


def _intervals(rng, seqs, n):
    """Lengths 0..4, intervals at contig starts and ends, whole contigs and random ones."""
    out = []
    for ci, (_, s) in enumerate(seqs):
        L = len(s)
        for ln in range(0, 5):
            if ln <= L:
                out += [(ci, 0, ln), (ci, L - ln, L)]
        out.append((ci, 0, L))
    while len(out) < n:
        ci = rng.randrange(len(seqs))
        L = len(seqs[ci][1])
        ln = min(L, rng.choice([0, 1, 2, 3, 4, 5, rng.randint(1, 400), rng.randint(1, 5000)]))
        a = rng.randrange(0, L - ln + 1)
        out.append((ci, a, a + ln))
    return out


# ------------------------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("width", [1, 9, 60, 61, 70])
@pytest.mark.parametrize("crlf", [False, True])
def test_closed_form_matches_oracle(width, crlf, ref_dir, tmp_path):
    rng = random.Random(1000 * width + crlf)
    for rep in range(3):
        data = _genome(rng, rng.choice([400, 3000]) if width == 1 else rng.choice([3000, 12000]), width, rng.choice([1, 3, 6]), crlf=crlf, iupac=rep * 20)
        seqs = _contig_seqs(data)
        idx = tnc.fasta_index(data)
        assert [c.line_bytes - c.line_bases for _, c in idx if c.len] == [2 if crlf else 1] * sum(1 for _, c in idx if c.len)
        iv = _intervals(rng, seqs, 120)
        got = ic.closed_form_rows(data, idx, iv)
        for row, one in zip(got, iv):
            vf = virtual_fasta(data, [one])
            assert np.array_equal(row, ob.tnc_counts(vf)), (one, width, crlf)
        if ref_dir and rep == 0:                         # the unmodified reference on the extracted FASTA of a few intervals
            for row, one in list(zip(got, iv))[:20]:
                p = tmp_path / "one.fa"
                p.write_bytes(virtual_fasta(data, [one]))
                out = subprocess.run([os.path.join(ref_dir, "tncCountsProfile"), str(p)], capture_output=True, check=True).stdout.decode()
                assert out == ob.tnc_text(row)


def test_fold32_matches_the_oracle_fold():
    L = ob.oracle()
    L.tnc_oracle_fold.restype = None
    L.tnc_oracle_fold.argtypes = [C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    rng = np.random.default_rng(7)
    rows = rng.integers(0, 1 << 40, size=(50, 64)).astype(np.int64)
    want = np.zeros((50, 32), dtype=np.int64)
    for r, w in zip(rows, want):
        L.tnc_oracle_fold(r.ctypes.data_as(C.POINTER(C.c_int64)), w.ctypes.data_as(C.POINTER(C.c_int64)))
    assert np.array_equal(tnc.fold32(rows), want)
    assert np.array_equal(tnc.fold32(rows.reshape(5, 10, 64)), want.reshape(5, 10, 32))
    one = np.zeros(32, dtype=np.int64)
    ssb.lib().ssb_tnc_fold32.restype = None
    ssb.lib().ssb_tnc_fold32(rows[0].ctypes.data_as(C.POINTER(C.c_int64)), one.ctypes.data_as(C.POINTER(C.c_int64)))
    assert np.array_equal(one, want[0])
    # the 32 lines of format_counts are the fold's values
    assert [int(l.split("\t")[1]) for l in tnc.format_counts(rows[1]).splitlines()] == list(want[1])


# ------------------------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    c = ssb.Context(0)
    yield c
    c.close()


def _device(data):
    import torch
    return torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()


def _rows(ctx, d, idx, iv, first=0, last=None, rows=None):
    import torch
    last = len(iv) if last is None else last
    if rows is None:
        rows = torch.zeros((last - first, 64), dtype=torch.int64, device="cuda")
    tnc.count_intervals_device(ctx, d.data_ptr(), d.numel(), idx, iv, rows.data_ptr(), first, last)
    ctx.sync()
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(6))
def test_rows_match_the_oracle(seed, ctx):
    rng = random.Random(300 + seed)
    data = _genome(rng, rng.choice([5000, 40000, 200000]), rng.choice([60, 61, 70, 9]), contigs=1 + seed, crlf=seed == 4, iupac=30 * (seed % 2))
    seqs = _contig_seqs(data)
    idx = tnc.fasta_index(data)
    iv = _intervals(rng, seqs, 400)
    iv += [iv[rng.randrange(len(iv))] for _ in range(30)]                                  # duplicates
    iv += [(c, a, min(len(seqs[c][1]), b + 7)) for c, a, b in iv[:30]]                   # overlaps
    iv += [(c, 0, len(seqs[c][1])) for c in range(len(seqs))] + [(0, 5, 6), (0, 9, 10)]   # whole contigs next to 1-base intervals
    rng.shuffle(iv)
    got = _rows(ctx, _device(data), idx, iv).cpu().numpy()
    want = np.array([ob.tnc_counts(virtual_fasta(data, [one])) for one in iv])
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_partitions_concatenate_and_calls_accumulate(ctx):
    import torch
    rng = random.Random(21)
    data = _genome(rng, 300000, 60, contigs=4)
    seqs = _contig_seqs(data)
    idx = tnc.fasta_index(data)
    iv = _intervals(rng, seqs, 3000)
    rng.shuffle(iv)
    d = _device(data)
    whole = _rows(ctx, d, idx, iv)
    cuts = sorted({0, len(iv)} | {rng.randrange(0, len(iv) + 1) for _ in range(5)})
    parts = torch.cat([_rows(ctx, d, idx, iv, a, b) for a, b in zip(cuts, cuts[1:])])
    assert torch.equal(parts, whole)
    _rows(ctx, d, idx, iv, rows=whole)                   # adds to what is there
    assert torch.equal(whole, 2 * parts)
    assert np.array_equal(whole.cpu().numpy(), 2 * ic.closed_form_rows(data, idx, iv))


@pytest.mark.gpu
def test_bed_total_minus_rows_is_the_straddling_windows(ctx):
    import torch
    rng = random.Random(8)
    data = _genome(rng, 60000, 60, contigs=3)
    seqs = _contig_seqs(data)
    idx = tnc.fasta_index(data)
    iv = _intervals(rng, seqs, 300)
    d = _device(data)
    rows = _rows(ctx, d, idx, iv).cpu().numpy()
    total = torch.zeros(64, dtype=torch.int64, device="cuda")
    tnc.count_bed_device(ctx, d.data_ptr(), d.numel(), idx, iv, total.data_ptr())
    ctx.sync()
    straddle = ob.tnc_counts(virtual_fasta(data, iv)) - sum(ob.tnc_counts(virtual_fasta(data, [one])) for one in iv)
    assert straddle.sum() > 0
    assert np.array_equal(total.cpu().numpy() - rows.sum(axis=0), straddle)


def _big_genome(seed, lengths, width=60):
    """Genome text of random contigs with N blocks and soft-masked runs (numpy, fast), and each contig's bases."""
    g = np.random.default_rng(seed)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    parts, seqs = [], []
    for k, ln in enumerate(lengths):
        s = lut[g.integers(0, 4, ln)]
        for a in g.integers(0, ln - 5000, 20):
            s[a:a + g.integers(1, 5000)] = ord("N")
        for a in g.integers(0, ln - 3000, 200):
            s[a:a + g.integers(1, 3000)] |= 0x20
        seqs.append(s)
        parts += [b">c%d\n" % k, ic.wrap(s, width)]
    return b"".join(parts), seqs


@pytest.mark.gpu
def test_a_million_tiles_and_one_50mb_interval(ctx):
    data, seqs = _big_genome(5, [17_000_003, 52_000_000, 16_999_989])
    idx = tnc.fasta_index(data)
    d = _device(data)
    # 31- and 29-base tiles over contigs 0 and 2 (about 1.1 M rows), plus one 50 Mb interval of contig 1 split over many warps
    tiles = {0: 31, 2: 29}
    iv = [(c, a, min(a + t, len(seqs[c]))) for c, t in tiles.items() for a in range(0, len(seqs[c]), t)]
    iv.append((1, 1_000_001, 51_000_001))
    assert len(iv) > 1_000_000
    got = _rows(ctx, d, idx, np.array(iv, dtype=np.int64)).cpu().numpy()
    w = ic.window_index(seqs[1][1_000_001:51_000_001])
    want = np.concatenate([ic.tiled_rows(seqs[c], t) for c, t in tiles.items()] + [np.bincount(w[w >= 0], minlength=64)[None]])
    assert np.array_equal(got, want)
    assert got[-1].sum() > 40_000_000


@pytest.mark.gpu
def test_offsets_past_4gib(ctx):
    import torch
    n = (1 << 32) + (1 << 22)
    buf = torch.full((n,), ord("N"), dtype=torch.uint8, device="cuda")
    rng = random.Random(4)
    seq = np.frombuffer(fc.genome_like(rng, 40000, width=40000, lower_runs=4).split(b"\n")[1], dtype=np.uint8)
    text = ic.wrap(seq, 61)
    off = (1 << 32) - 12345                              # the contig straddles 2^32
    buf[off:off + len(text)] = torch.from_numpy(np.frombuffer(text, dtype=np.uint8).copy()).cuda()
    idx = [("x", tnc.FastaContig(off, len(seq), 61, 62))]
    host_idx = [("x", tnc.FastaContig(0, len(seq), 61, 62))]
    iv = [(0, 0, len(seq))] + [(0, a, a + rng.randint(0, 3000)) for a in (rng.randrange(0, len(seq) - 3000) for _ in range(200))]
    rows = torch.zeros((len(iv), 64), dtype=torch.int64, device="cuda")
    tnc.count_intervals_device(ctx, buf.data_ptr(), n, idx, iv, rows.data_ptr())
    ctx.sync()
    assert np.array_equal(rows.cpu().numpy(), ic.closed_form_rows(text, host_idx, iv))
    assert rows[0].sum().item() > 30000


@pytest.mark.gpu
def test_refusals(ctx):
    import torch
    data = b">a\nACGTACGTAC\nGTACGTAC\n>b\nACGTAC\n"
    idx = tnc.fasta_index(data)
    d = _device(data)
    rows = torch.zeros((2, 64), dtype=torch.int64, device="cuda")

    def call(index, iv):
        tnc.count_intervals_device(ctx, d.data_ptr(), d.numel(), index, iv, rows.data_ptr())

    with pytest.raises(ssb.SSBError) as e:
        call(idx, [(0, 0, 5), (0, 6, 4)])
    assert e.value.code == -3
    with pytest.raises(ssb.SSBError) as e:
        call(idx, [(0, 0, 5), (1, 0, 7)])
    assert e.value.code == -5
    wrong = [(n, tnc.FastaContig(c.seq_off, c.len, c.line_bases + 1, c.line_bytes + 1)) for n, c in idx]
    with pytest.raises(ssb.SSBError) as e:
        call(wrong, [(0, 0, 18)])
    assert e.value.code == -5
    rows.zero_()
    call(idx, [(0, 0, 18), (1, 0, 6)])                 # and the right index is accepted
    ctx.sync()
    assert rows[0].sum().item() == 16 and rows[1].sum().item() == 4


def _cli_text(data, seqs, iv):
    names = [l.split("\t")[0] for l in ob.tnc_text(np.zeros(64, dtype=np.int64)).splitlines()]
    out = ["\t".join(["#chrom", "start", "end"] + names)]
    for c, a, b in iv:
        vals = [l.split("\t")[1] for l in ob.tnc_text(ob.tnc_counts(virtual_fasta(data, [(c, a, b)]))).splitlines()]
        out.append("\t".join([seqs[c][0], str(a), str(b)] + vals))
    return "\n".join(out) + "\n"


@pytest.mark.gpu
def test_cli_per_interval(tmp_path):
    rng = random.Random(6)
    data = _genome(rng, 60000, 60, contigs=3)
    seqs = _contig_seqs(data)
    iv = _intervals(rng, seqs, 400)
    (tmp_path / "g.fa").write_bytes(data)
    (tmp_path / "t.bed").write_text("track name=x\n" + "".join("%s\t%d\t%d\tname%d\n" % (seqs[c][0], a, b, i) for i, (c, a, b) in enumerate(iv)))
    args = [EXE, str(tmp_path / "g.fa"), str(tmp_path / "t.bed")]
    got = subprocess.run(args + ["--per-interval"], capture_output=True)
    assert got.returncode == 0, got.stderr
    assert got.stdout.decode() == _cli_text(data, seqs, iv)
    # another third argument leaves BED mode as it is
    other = subprocess.run(args + ["--other"], capture_output=True)
    assert other.returncode == 0 and other.stdout.decode() == ob.tnc_text(ob.tnc_counts(virtual_fasta(data, iv)))
    (tmp_path / "bad.bed").write_text("%s\t0\t%d\n" % (seqs[0][0], len(seqs[0][1]) + 1))
    bad = subprocess.run([EXE, str(tmp_path / "g.fa"), str(tmp_path / "bad.bed"), "--per-interval"], capture_output=True)
    assert bad.returncode == 3 and b"outside its contig" in bad.stderr


@pytest.mark.gpu
def test_cli_per_interval_on_two_gpus(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = random.Random(16)
    data = _genome(rng, 200000, 70, contigs=2)
    seqs = _contig_seqs(data)
    iv = _intervals(rng, seqs, 2000)
    (tmp_path / "g.fa").write_bytes(data)
    (tmp_path / "t.bed").write_text("".join("%s\t%d\t%d\n" % (seqs[c][0], a, b) for c, a, b in iv))
    args = [EXE, str(tmp_path / "g.fa"), str(tmp_path / "t.bed"), "--per-interval"]
    one = subprocess.run(args, capture_output=True)
    two = subprocess.run(args, capture_output=True, env=dict(os.environ, SSB_GPUS="2"))
    assert one.returncode == 0 and two.returncode == 0, (one.stderr, two.stderr)
    assert two.stdout == one.stdout
    assert one.stdout.decode() == _cli_text(data, seqs, iv)
