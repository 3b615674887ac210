"""Emit copies runs of output lines that are contiguous in the input as one segment.  With a `.spike` table whose targets all lie
outside the covered range a pass spikes nothing, so its output is exactly the kept lines, stably sorted by (tid, end): restated here
in Python (the read filter of read_bam, the end from POS + CIGAR) and compared byte for byte on inputs whose segments are long,
short, longer than a warp's task, cut by shards and by streamed pieces, and at the end of a body without a final newline.  The
restatement is pinned to the CPU checker first."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

import bench_spike as bs
import spike_cases as sc
from stochasticsim_b200 import spike as sp

EMPTY = "chrE"                                    # a contig without reads: the targets sit there, so nothing is spiked
CIGAR_REF = re.compile(rb"(\d+)([MDN=X])")


def restated_output(body: bytes, names):
    """The kept lines of `body` in (tid, end) order, ties in input order; a last line without a newline gets one."""
    parts = body.split(b"\n")
    lines = [p + b"\n" for p in parts[:-1]] + ([parts[-1] + b"\n"] if parts[-1] else [])
    kept = []
    for i, line in enumerate(lines):
        f = line.split(b"\t", 6)
        flag, rname, pos, mapq = int(f[1]), f[2], int(f[3]), int(f[4])
        rlen = sum(int(n) for n, _ in CIGAR_REF.findall(f[5]))
        if rname == b"*" or flag & (4 | 256 | 512 | 1024) or mapq < 30 or ((flag & 1) and not (flag & 2)) or not rlen:
            continue
        kept.append((names.index(rname.decode()), pos - 1 + rlen, i))
    kept.sort()
    return b"".join(lines[i] for _, _, i in kept)


def synth(contig_len, coverage, read_len=150, seed=2, **rates):
    """(reference, SAM body) of one contig from the C2 generator, with `rates` (softclip_rate, ...) changed."""
    L = bs.synth_lib()
    p = bs.c2_params(L, seed, coverage)
    p.read_len = read_len
    for k, v in rates.items():
        setattr(p, k, v)
    ref = np.empty(contig_len + 1, dtype=np.uint8)
    L.synth_ref_contig(C.byref(p), 0, contig_len, 0, contig_len, 0, ref.ctypes.data)
    need = L.synth_sam_range(C.byref(p), 0, b"chr1", ref.ctypes.data, contig_len, 0, contig_len, 0, contig_len, None, 0, None)
    buf = np.empty(need, dtype=np.uint8)
    L.synth_sam_range(C.byref(p), 0, b"chr1", ref.ctypes.data, contig_len, 0, contig_len, 0, contig_len, buf.ctypes.data, need, None)
    return ref[:contig_len].tobytes(), buf.tobytes()


def long_reads(contig_len, n_reads, seed):
    """(reference, SAM body): single-end reads of 5-100 kb, some soft clipped at the end (so that they leave the input order)."""
    rng = random.Random(seed)
    ref = bytes(rng.choice(b"ACGT") for _ in range(contig_len))
    recs = []
    for k in range(n_reads):
        span = rng.randrange(5_000, 100_000)
        pos = rng.randrange(0, contig_len - span)
        clip = rng.randrange(1, 3_000) if rng.random() < 0.4 else 0
        cig = b"%dM" % (span - clip) + (b"%dS" % clip if clip else b"")
        seq = ref[pos:pos + span]
        recs.append((pos, b"L%d\t0\tchr1\t%d\t60\t%s\t*\t0\t0\t%s\t%s\n" % (k, pos + 1, cig, seq, b"I" * span)))
    recs.sort(key=lambda r: r[0])
    return ref, b"".join(r[1] for r in recs)


def case(kind):
    """(names, {name: sequence}, body, targets) of one input family."""
    if kind == "c2":
        ref, body = synth(2_000_000, 100.0)
    elif kind in ("short36", "short76"):
        ref, body = synth(300_000, 100.0, read_len=int(kind[5:]), seed=5, softclip_rate=0.1, indel_rate=0.02, refskip_rate=0.03, filt_rate=0.05)
    elif kind == "long":
        ref, body = long_reads(1_500_000, 120, seed=9)
    elif kind == "no_final_newline":
        ref, body = synth(60_000, 40.0, read_len=76, seed=3, softclip_rate=0.1)
        body = body[:-1]
    names = ["chr1", EMPTY]
    seqs = {"chr1": ref, EMPTY: b"ACGT" * 500}
    targets = sp.parse_spike(b"".join(b"%s\t%d\t.\t0.5\n" % (EMPTY.encode(), x) for x in range(100, 1100, 100)), names)
    return names, seqs, body, targets


def test_restatement_matches_checker(tmp_path):
    """The restatement against the CPU checker on one small input with soft clips, indels, ref-skips and filtered pairs."""
    names, seqs, body, targets = case("short76")
    body = body[:body.index(b"\n", 2_000_000) + 1]
    hdr = b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n.encode(), len(seqs[n])) for n in names)
    with open(tmp_path / "in.fa", "wb") as f:
        for n in names:
            f.write(b">%s\n" % n.encode() + b"".join(seqs[n][i:i + 60] + b"\n" for i in range(0, len(seqs[n]), 60)))
    (tmp_path / "in.sam").write_bytes(hdr + body)
    (tmp_path / "in.spike").write_bytes(b"%s\t100\t.\t0.5\n%s\t700\tG\t0.5\n" % (EMPTY.encode(), EMPTY.encode()))
    rc, _, out, _, err = sc.run_cli(sc.CHECKER, str(tmp_path / "in"), str(tmp_path / "ref"), cmdname="stochasticSpike")
    assert rc == 0, err
    assert out.startswith(hdr)
    want = restated_output(body, names)
    assert len(want) < len(body), "expected the filter to drop lines"
    assert out[len(hdr):] == want


@pytest.fixture(scope="module")
def ctx():
    import stochasticsim_b200 as ssb
    c = ssb.Context(0)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["c2", "short36", "short76", "long", "no_final_newline"])
def test_single_run(kind, ctx):
    names, seqs, body, targets = case(kind)
    with sp.Spike(ctx, names, seqs) as s:
        out, res, st = s.run_host(body, targets, 434)
    assert all(r.status != sp.T_HIT for r in res)
    assert out == restated_output(body, names)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["short76", "no_final_newline"])
def test_two_shards(kind, ctx):
    names, seqs, body, targets = case(kind)
    out, res, sts, _, n = sp.run_sharded([ctx], names, seqs, body, targets, 434, 2, 600)
    assert n == 2
    assert out == restated_output(body, names)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,piece", [("short76", 200_000), ("no_final_newline", 40_000)])
def test_streamed_in_many_pieces(kind, piece, ctx, monkeypatch):
    names, seqs, body, targets = case(kind)
    monkeypatch.setenv("SSB_STREAM_BYTES", str(piece))
    with sp.Spike(ctx, names, seqs) as s:
        out, res, st = s.run_host(body, targets, 434)
    assert st.n_forwarded >= 3, "expected the body to be streamed in several pieces"
    assert out == restated_output(body, names)
