"""GPU parity: the spike path of libssb200 (through the C ABI and through the drop-in C main) against the reference binary
(oracle/_ref/stochasticSpike = the unmodified reference over the htslib shim; the restated oracle when that binary is absent)
-- SAM bytes, truth.vcf and the stats block must be identical."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import oracle_bind as ob
import spike_cases as sc
import stochasticsim_b200 as ssb
from stochasticsim_b200 import spike as sp

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "spike_toy")
FULL_VCF = os.environ.get("SSB_TEST_FULL_VCF", "1") == "1"


@pytest.fixture(scope="module")
def ctx():
    c = ssb.Context(0)
    yield c
    c.close()


def vcf_cmp(a, b):
    if FULL_VCF:
        return a == b
    return sc.vcf_without_seq_errors(a) == sc.vcf_without_seq_errors(b)


def first_diff(a, b):
    n = min(len(a), len(b))
    for i in range(n):
        if a[i] != b[i]:
            lo = a.rfind(b"\n", 0, i) + 1
            return "offset %d: want %r got %r" % (i, a[lo:lo + 300], b[lo:lo + 300])
    return "lengths %d vs %d" % (len(a), len(b))


def test_rand_stream_matches_glibc(ctx):
    with sp.Spike(ctx, ["c"], {"c": b"ACGT"}) as s:
        for seed in (434, 42, 0, 1, 4294967295):
            got = s.rand(seed, 0, 70000)
            assert np.array_equal(got, ob.glibc_rand(seed, 0, 70000)), seed
        assert list(s.rand(434, 0, 5)) == [43521843, 555289354, 711778510, 1948175914, 749459303]     # SURVEY App. C
        assert int(s.rand(434, 10**6, 1)[0]) == 1066614699
        assert int(s.rand(434, 10**9, 1)[0]) == 586798013
        assert int(s.rand(434, 2**32, 1)[0]) == 2013220912
        assert int(s.rand(434, 5 * 10**9, 1)[0]) == 1050868447
        got = s.rand(434, 999_000, 600_000)
        assert np.array_equal(got, ob.glibc_rand(434, 999_000, 600_000))


@pytest.mark.parametrize("name", sorted(sc.CASES))
def test_cli_parity(name, tmp_path, ctx):
    prefix = sc.generate(name, str(tmp_path))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0
    assert got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1], "stats differ: %r vs %r" % (want[1], got[1])
    assert vcf_cmp(want[3], got[3]), "truth.vcf differs: " + first_diff(want[3], got[3])


@pytest.mark.parametrize("seed", [1, 434, 99991])
def test_seeds(seed, tmp_path, ctx):
    prefix = sc.generate("overlap_heavy", str(tmp_path), coverage=25, contigs="chr19:8000", spikes=60)
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), seed=seed, cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"), seed=seed)
    assert got[0] == 0, got[4]
    assert got[2] == want[2], first_diff(want[2], got[2])
    assert vcf_cmp(want[3], got[3]), first_diff(want[3], got[3])


@pytest.mark.parametrize("name,chunk,group,slice_", [("plain", 512, 4, 4096), ("deep_lowvaf", 256, 1, 16), ("mask_n_ref", 1024, 3, 5), ("overlap_heavy", 512, 4, 4096),
                                                     ("two_contigs_window", 640, 2, 9), ("plain", 96, 8, 3), ("deep_lowvaf", 64, 5, 1)])
def test_parallel_chain_matches_serial(name, chunk, group, slice_, tmp_path, ctx, monkeypatch):
    """The chunked chain (windows of candidate offsets cut into slices, merging walkers, recorded chunk boundaries, composed
    group maps) against the oracle, and against the one-warp serial chain: same SAM, same per-target results, same draw count."""
    prefix = sc.generate(name, str(tmp_path))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    with sp.Spike(ctx, names, seqs) as s:
        monkeypatch.setenv("SSB_CHAIN_SERIAL", "1")
        out_s, res_s, st_s = s.run_host(body, targets, 434)
        monkeypatch.delenv("SSB_CHAIN_SERIAL")
        monkeypatch.setenv("SSB_CHAIN_CHUNK", str(chunk))
        monkeypatch.setenv("SSB_CHAIN_GROUP", str(group))
        monkeypatch.setenv("SSB_CHAIN_SLICE", str(slice_))
        out_p, res_p, st_p = s.run_host(body, targets, 434)
    assert st_s.chain_mode == 1
    assert hdr + out_s == want[2] and hdr + out_p == want[2]
    assert st_p.rng_draws == st_s.rng_draws
    key = lambda r: (r.status, r.at_pos, r.filter, r.ref_cnt, r.mut_cnt, tuple(r.err_cnt), r.rng_offset, r.mutant_allele)
    assert [key(r) for r in res_p] == [key(r) for r in res_s]
    if name in ("plain", "deep_lowvaf", "mask_n_ref"):
        assert st_p.chain_mode > 1, "expected the chunked chain to be used"


@pytest.mark.parametrize("name,chunk,resident", [("plain", 96, 3), ("deep_lowvaf", 64, 2), ("mask_n_ref", 128, 5), ("two_contigs_window", 96, 1)])
def test_chain_geometry_is_chosen_to_fit_the_device(name, chunk, resident, tmp_path, ctx, monkeypatch):
    """Phase 1 picks the group length and the slice width from the number of blocks the device holds at once (longer groups when the
    slices of the windows would not all be resident, then the narrowest slices that still fit).  With a "device" of a few blocks the
    small inputs exercise what a shard far down the stream does at full size.
    Same SAM, same per-target results and the same draw count as the one-warp serial chain and the reference."""
    prefix = sc.generate(name, str(tmp_path))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    with sp.Spike(ctx, names, seqs) as s:
        monkeypatch.setenv("SSB_CHAIN_SERIAL", "1")
        out_s, res_s, st_s = s.run_host(body, targets, 434)
        monkeypatch.delenv("SSB_CHAIN_SERIAL")
        monkeypatch.setenv("SSB_CHAIN_CHUNK", str(chunk))
        monkeypatch.setenv("SSB_P1_RESIDENT", str(resident))
        monkeypatch.setenv("SSB_SORT64", "1")              # and the 8-byte end-order keys (genomes whose keys do not fit 32 bits)
        out_p, res_p, st_p = s.run_host(body, targets, 434)
    assert hdr + out_s == want[2] and hdr + out_p == want[2]
    assert st_p.rng_draws == st_s.rng_draws
    key = lambda r: (r.status, r.at_pos, r.filter, r.ref_cnt, r.mut_cnt, tuple(r.err_cnt), r.rng_offset, r.mutant_allele)
    assert [key(r) for r in res_p] == [key(r) for r in res_s]
    if name in ("plain", "deep_lowvaf", "mask_n_ref"):
        assert st_p.chain_mode > 1, "expected the chunked chain to be used"


@pytest.mark.parametrize("name", ["plain", "overlap_heavy", "two_contigs_window"])
def test_bam_input(name, tmp_path, ctx):
    """argv[1] as a real BGZF BAM (what bin/spikeIn.bash passes): same SAM, truth.vcf body and stats as from the SAM text."""
    import bam_writer
    prefix = sc.generate(name, str(tmp_path))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    bam = tmp_path / "in.bam"
    bam.write_bytes(bam_writer.sam_to_bam(open(prefix + ".sam", "rb").read()))
    # the reference insists on an index next to the BAM (stochasticSpike.c:1035-1039)
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "noidx"), sam=str(bam))
    assert got[0] == 1 and b"Can't load index" in got[4]
    (tmp_path / "in.bam.bai").write_bytes(b"BAI\1")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"), sam=str(bam))
    assert got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1]
    strip = lambda v: b"\n".join(l for l in v.split(b"\n") if not l.startswith(b"##stochasticSpikeCommand="))
    assert strip(got[3]) == strip(want[3]), first_diff(strip(want[3]), strip(got[3]))


@pytest.mark.parametrize("k", range(8))
def test_fuzz_configs(k, tmp_path, ctx, monkeypatch):
    """Seeded random generator settings (depth, read/fragment geometry, error mix, contigs, spike density), alternating
    the chain mode: SAM, truth.vcf and stats must match the oracle byte for byte."""
    import random
    rng = random.Random(1000 + k)
    rl = rng.choice([36, 50, 76, 100, 151])
    args = dict(seed=2000 + k, contigs=rng.choice(["c1:9000", "chrA:6000,chrB:5000", "chr1:4000,chr2:4000,chr3:3000"]),
                coverage=rng.choice([3, 12, 40, 150]), read_len=rl, frag_mean=int(rl * rng.choice([1.05, 1.4, 2.2, 3.0])), frag_sd=rng.choice([3, 15, 40]),
                sub=rng.choice([0.0, 0.002, 0.03]), indel=rng.choice([0.0, 0.01, 0.08]), nrate=rng.choice([0.0, 0.005]), q0=rng.choice([0.0, 0.02]),
                softclip=rng.choice([0.0, 0.1]), refskip=rng.choice([0.0, 0.04]), filt=rng.choice([0.0, 0.1]), lower=rng.choice([0.0, 0.2]),
                spikes=rng.choice([5, 60, 400]), alt_mode=rng.choice([0, 1]), aux=rng.choice([0, 1]), af=rng.choice(["0.01:0.5", "0.3:1.0", "0.001:0.02"]))
    prefix = sc.generate("plain", str(tmp_path), **args)
    if k % 2:
        monkeypatch.setenv("SSB_CHAIN_CHUNK", str(rng.choice([96, 320, 1024])))
        monkeypatch.setenv("SSB_CHAIN_GROUP", str(rng.choice([1, 2, 4, 7])))
        monkeypatch.setenv("SSB_CHAIN_SLICE", str(rng.choice([2, 33, 4096])))
    if k % 3 == 0:
        monkeypatch.setenv("SSB_NO_EXC_LIST", "1")
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), seed=434 + k, cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"), seed=434 + k)
    assert want[0] == 0 and got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1]
    assert vcf_cmp(want[3], got[3]), "truth.vcf differs: " + first_diff(want[3], got[3])


def test_golden_fixture(tmp_path, ctx):
    """tests/golden/spike_toy was produced by the unmodified reference over the htslib shim."""
    for f in ("in.sam", "in.fa", "in.spike"):
        shutil.copy(os.path.join(GOLD, f), tmp_path / f)
    r = subprocess.run([sc.PRODUCT, "in.sam", "in.fa", "in.spike", "434", "out.sam"], cwd=tmp_path, capture_output=True)
    assert r.returncode == 0, r.stderr
    rd = lambda n: open(os.path.join(GOLD, n), "rb").read()
    assert (tmp_path / "out.sam").read_bytes() == rd("out.sam")
    assert r.stdout == rd("stdout.txt")
    assert vcf_cmp(rd("truth.vcf"), (tmp_path / "truth.vcf").read_bytes())


def test_abi_run_host(tmp_path, ctx):
    """The same through the ctypes binding: body in, body out, per-target results."""
    prefix = sc.generate("plain", str(tmp_path))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    with sp.Spike(ctx, names, seqs) as s:
        out, res, st = s.run_host(body, targets, 434)
    assert hdr + out == want[2]
    assert st.alignmentCount == out.count(b"\n")
    hits = [r for r in res if r.status == sp.T_HIT]
    assert len(hits) == st.n_hits > 0
    assert all(r.rng_offset >= 0 for r in hits)


def test_edge_inputs(tmp_path, ctx):
    prefix = sc.generate("plain", str(tmp_path), contigs="chr19:3000", spikes=10)
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    lines = body.split(b"\n")[:-1]
    with sp.Spike(ctx, names, seqs) as s:
        # no alignments at all: every target is left over
        out, res, st = s.run_host(b"", targets, 434)
        assert out == b"" and all(r.status == sp.T_TAIL for r in res) and st.numberOfLociCovered == 0
        # no targets: reads pass through in end order
        out, res, st = s.run_host(body, [], 434)
        assert sorted(out.split(b"\n")) == sorted(body.split(b"\n"))
        # a body without the final newline gets one
        out2, _, _ = s.run_host(body[:-1], [], 434)
        assert out2 == out
        # unsorted input is refused (htslib's pileup errors out, stochasticSpike.c:1129)
        with pytest.raises(ssb.SSBError) as e:
            s.run_host(b"\n".join(lines[::-1]) + b"\n", targets, 434)
        assert e.value.code == -6
        # a malformed line is refused
        with pytest.raises(ssb.SSBError) as e:
            s.run_host(body + b"garbage\n", targets, 434)
        assert e.value.code == -5


def test_cli_usage_and_errors(tmp_path, ctx):
    r = subprocess.run([sc.PRODUCT], capture_output=True)
    assert r.returncode == 0 and b"Usage" in r.stderr                                     # stochasticSpike.c:938-941
    prefix = sc.generate("plain", str(tmp_path), contigs="chr19:3000", spikes=5)
    r = subprocess.run([sc.PRODUCT, "/nonexistent.sam", prefix + ".fa", prefix + ".spike", "1", "o.sam"], cwd=tmp_path, capture_output=True)
    assert r.returncode == 1 and b"Couldn't open bam" in r.stderr
    r = subprocess.run([sc.PRODUCT, prefix + ".sam", prefix + ".fa", "/nonexistent.spike", "1", "o.sam"], cwd=tmp_path, capture_output=True)
    assert r.returncode == 255


def test_large_properties(ctx, monkeypatch):
    """Size-independent properties on a chr19-length input (C2's generator at 5x: ~1.95 M reads, ~0.7 GB, 58.6 M covered loci),
    too large for the CPU oracle: (a) without targets the output is the input's lines in another order (same bytes, same
    line lengths); (b) with the 10,000 targets the lines stay where they are and only A/C/G/T bytes change, no more than
    two per pileup entry; (c) the chunked chain (grouped, sliced phase 1 at its production geometry) gives byte for byte
    what the one-warp serial chain gives, with the same draw count and per-target results; (d) a second run repeats it."""
    import numpy as np
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    import bench_spike as bs
    L = bs.synth_lib()
    ref, parts, n_reads, spike_text = bs.make_workload(L, 2, bs.CHR19, 5.0, 10_000)
    body = np.concatenate(parts).tobytes()
    del parts
    names = ["chr19"]
    targets = sp.parse_spike(spike_text, names)
    key = lambda r: (r.status, r.at_pos, r.filter, r.ref_cnt, r.mut_cnt, tuple(r.err_cnt), r.rng_offset, r.mutant_allele)
    with sp.Spike(ctx, names, {"chr19": ref.tobytes()}) as s:
        out0, _, st0 = s.run_host(body, [], 434)
        out_p, res_p, st_p = s.run_host(body, targets, 434)
        out_p2, res_p2, st_p2 = s.run_host(body, targets, 434)
        monkeypatch.setenv("SSB_CHAIN_SERIAL", "1")
        out_s, res_s, st_s = s.run_host(body, targets, 434)
    a, b0 = np.frombuffer(body, dtype=np.uint8), np.frombuffer(out0, dtype=np.uint8)
    # (a)
    assert st0.as_dict()["n_kept"] == n_reads and len(out0) == len(body)
    assert np.array_equal(np.bincount(a, minlength=256), np.bincount(b0, minlength=256))
    la = np.sort(np.diff(np.flatnonzero(a == 10), prepend=-1)); lb = np.sort(np.diff(np.flatnonzero(b0 == 10), prepend=-1))
    assert np.array_equal(la, lb)
    # (b)
    bp = np.frombuffer(out_p, dtype=np.uint8)
    assert len(out_p) == len(out0)
    d = np.flatnonzero(bp != b0)
    n_entries = sum(r.ref_cnt + r.mut_cnt + sum(r.err_cnt) for r in res_p)
    assert 0 < d.size <= 2 * max(1, n_entries)
    assert set(np.unique(bp[d]).tolist()) <= set(b"ACGT")
    assert np.array_equal(np.flatnonzero(bp == 10), np.flatnonzero(b0 == 10))
    # (c), (d)
    assert st_p.chain_mode > 1 and st_s.chain_mode == 1
    assert out_p == out_s and out_p == out_p2
    assert st_p.rng_draws == st_s.rng_draws == st_p2.rng_draws
    assert [key(r) for r in res_p] == [key(r) for r in res_s] == [key(r) for r in res_p2]


def _long_read_case(dirname, read_lens, seed=7):
    """Single-end reads far longer than the tokeniser's overhang (3 KiB) and tile (32 KiB): written here, the generator's reads stop at 1 kb."""
    import random
    rng = random.Random(seed)
    n = 260_000
    ref = "".join(rng.choice("ACGT") for _ in range(n))
    reads = []
    for i, L in enumerate(read_lens):
        pos = rng.randrange(0, n - L)
        seq = list(ref[pos:pos + L])
        for _ in range(max(1, L // 400)):
            k = rng.randrange(L); seq[k] = rng.choice("ACGTN")
        qual = "".join(rng.choice("#5AFI") for _ in range(L))
        reads.append((pos, "r%d" % i, "".join(seq), qual, L))
    reads.sort()
    prefix = os.path.join(dirname, "in")
    with open(prefix + ".fa", "w") as f:
        f.write(">chrL\n" + "\n".join(ref[i:i + 60] for i in range(0, n, 60)) + "\n")
    with open(prefix + ".sam", "w") as f:
        f.write("@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:chrL\tLN:%d\n" % n)
        for pos, name, seq, qual, L in reads:
            f.write("%s\t0\tchrL\t%d\t60\t%dM\t*\t0\t0\t%s\t%s\tNM:i:0\n" % (name, pos + 1, L, seq, qual))
    with open(prefix + ".spike", "w") as f:
        f.write("#CHROM\tPOS\tALT\tAF\n")
        for p in sorted(rng.sample(range(1000, n - 1000), 60)):
            f.write("chrL\t%d\t%s\t%.4g\n" % (p, rng.choice(".ACGT"), rng.uniform(0.05, 0.6)))
    return prefix


@pytest.mark.parametrize("read_lens", [[5000] * 150, [40000] * 12 + [5000] * 40 + [150] * 300, [100000, 90000, 70000]])
def test_long_reads(read_lens, tmp_path, ctx):
    """Lines longer than the staged overhang, than a whole tile, and tiles that hold no line start at all."""
    prefix = _long_read_case(str(tmp_path), read_lens)
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0 and got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1]
    assert vcf_cmp(want[3], got[3]), "truth.vcf differs: " + first_diff(want[3], got[3])


def test_short_reads_many_lines_per_tile(tmp_path, ctx):
    """36 bp reads: ~300 lines per 32 KiB tile, more than the tokeniser has parsing threads, so every tile also takes its
    second-round path (careful parser, no exception list for those reads)."""
    prefix = sc.generate("plain", str(tmp_path), contigs="chr19:20000", read_len=36, frag_mean=60, frag_sd=6, coverage=60, spikes=80)
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0 and got[0] == 0, got[4]
    assert len(want[2]) > 3_000_000
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1]
    assert vcf_cmp(want[3], got[3]), "truth.vcf differs: " + first_diff(want[3], got[3])


def test_error_rich_reads_overflow_the_tile_exception_buffer(tmp_path, ctx):
    """15 % substitutions, 10 % BQ-0 bases, 2 % N: far more than 1024 exceptional bases per tile, so the tokeniser's per-tile
    buffer fills up and the reads that no longer fit are left to the generic tally."""
    prefix = sc.generate("plain", str(tmp_path), contigs="chr19:12000", coverage=40, sub=0.15, q0=0.1, nrate=0.02, spikes=60)
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0 and got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1]
    assert vcf_cmp(want[3], got[3]), "truth.vcf differs: " + first_diff(want[3], got[3])


def _with_float_tags(sam: bytes, bad_line=None) -> bytes:
    """Every alignment line gets de:f / B:f fields in the form "%g" prints (what htslib would print back unchanged)."""
    import random
    rng = random.Random(3)
    out = []
    k = 0
    for line in sam.split(b"\n"):
        if line and not line.startswith(b"@"):
            vals = [rng.choice([0.0, 0.0123, 1.5, -2e-07, 123456.0, 1e+06, 3.33333e-05, 0.5])] + [rng.uniform(-5, 5) for _ in range(2)]
            txt = [("%g" % float(np.float32(v))).encode() for v in vals]
            line += b"\tde:f:" + txt[0] + b"\tXF:B:f," + txt[1] + b"," + txt[2]
            if bad_line is not None and k == bad_line:
                line += b"\tzz:f:1.50"                      # htslib would print 1.5: not a pass-through
            k += 1
        out.append(line)
    return b"\n".join(out)


def test_float_typed_optional_fields(tmp_path, ctx):
    """TAG:f and TAG:B:f fields (minimap2's de:f ...) in canonical "%g" form pass through, SAM and BAM; a float that htslib would print
    differently is refused (ADVICE r1: BAM float tags used to abort the run)."""
    import bam_writer
    prefix = sc.generate("plain", str(tmp_path), contigs="chr19:6000", spikes=20)
    sam = open(prefix + ".sam", "rb").read()
    tagged = _with_float_tags(sam)
    open(prefix + ".sam", "wb").write(tagged)
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0 and got[0] == 0, got[4]
    assert got[2] == want[2] and got[1] == want[1] and vcf_cmp(want[3], got[3])
    assert b"\tde:f:" in got[2]
    bam = tmp_path / "in.bam"
    bam.write_bytes(bam_writer.sam_to_bam(tagged))
    (tmp_path / "in.bam.bai").write_bytes(b"BAI\1")
    got_b = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpub"), sam=str(bam))
    assert got_b[0] == 0, got_b[4]
    assert got_b[2] == want[2]
    open(prefix + ".sam", "wb").write(_with_float_tags(sam, bad_line=17))
    bad = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "bad"))
    assert bad[0] == 3 and b"precondition" in bad[4]


def test_reference_length_zero_reads(tmp_path, ctx):
    """Reads whose CIGAR consumes no reference (all soft clip / insertion): htslib's pileup takes pos + bam_cigar2rlen as their end (not
    bam_endpos), so they never enter a pileup, never count in depth and are never written -- but they take part in the sortedness check."""
    prefix = sc.generate("plain", str(tmp_path), contigs="chr19:5000", spikes=20, coverage=15)
    sam = open(prefix + ".sam", "rb").read()
    lines = sam.split(b"\n")
    out = []
    k = 0
    for line in lines:
        out.append(line)
        if line and not line.startswith(b"@"):
            k += 1
            if k % 40 == 0:
                f = line.split(b"\t")
                n = len(f[9])
                f[0] = b"zero%d" % k
                f[5] = (b"%dS" % n) if k % 80 else (b"%dI" % n)
                f[1] = b"0"
                f[6], f[7], f[8] = b"*", b"0", b"0"
                out.append(b"\t".join(f[:11]))
    open(prefix + ".sam", "wb").write(b"\n".join(out))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0 and got[0] == 0, got[4]
    assert b"zero40\t" not in want[2]
    assert got[2] == want[2] and got[1] == want[1] and vcf_cmp(want[3], got[3])


@pytest.mark.parametrize("name,chunk,group,sigma", [("plain", 512, 2, 1.0), ("mask_n_ref", 256, 1, 0.7), ("deep_lowvaf", 96, 2, 1.5), ("plain", 256, 1, 0.5)])
def test_window_miss_is_walked_again(name, chunk, group, sigma, tmp_path, ctx, monkeypatch):
    """Windows far narrower than production (4 sigma): the exact walker leaves some group's window, that group is walked again from the
    exact offset (one block) and the maps are composed again -- same bytes as the serial chain; too many misses end in the serial chain."""
    prefix = sc.generate(name, str(tmp_path))
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    monkeypatch.setenv("SSB_CHAIN_CHUNK", str(chunk))
    monkeypatch.setenv("SSB_CHAIN_GROUP", str(group))
    monkeypatch.setenv("SSB_CHAIN_SIGMA", str(sigma))
    with sp.Spike(ctx, names, seqs) as s:
        out, res, st = s.run_host(body, targets, 434)
    assert hdr + out == want[2]
    if sigma <= 0.5:
        assert st.n_window_retries > 0 or st.chain_mode == 1, "expected misses with windows this narrow"


def test_deep_pileup_2000x(tmp_path, ctx):
    """BASELINE C5's depth: ~2000 entries per pileup, a target every 20 bases, low VAF, overlapping pairs -- the one-warp chain with the
    pileup staged in shared memory against the reference (whose mate search is quadratic in the depth: a short window)."""
    prefix = sc.generate("deep_lowvaf", str(tmp_path), contigs="chr1:900", coverage=2000, read_len=150, frag_mean=200, frag_sd=20, spikes=30, af="0.005:0.05")
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert want[0] == 0 and got[0] == 0, got[4]
    assert b"maxDepth = 2" in want[1] or b"maxDepth = 1" in want[1]
    assert got[2] == want[2], "SAM differs: " + first_diff(want[2], got[2])
    assert got[1] == want[1]
    assert vcf_cmp(want[3], got[3]), "truth.vcf differs: " + first_diff(want[3], got[3])
