"""The spike path on the reference layouts real genomes have (tests/layout_cases.py): GRCh38 with its alt, decoy and HLA contigs
(3,366 @SQ lines), a draft assembly of 12,000 scaffolds, and 4,097 contigs at the 32-bit boundary of the packed output-order keys.

Which code only acts differently when there are many contigs, and where it is checked here:
- RNAME / RNEXT lookup (sam_parse.cuh name_lookup): names that are prefixes of one another, HLA names with '*' and ':', RNEXT naming
  a decoy or HLA contig: test_builder_places_the_layout, then every parity test.
- the reference window staged per tile for its lowest tid (sam_parse.cuh): tiles that span several contigs (the scaffolds),
  test_builder_places_the_layout; the generic tally against the exception list, test_abi_modes_agree (SSB_NO_EXC_LIST).
- packed 32-bit against 8-byte output-order keys (spike_run.cuh): test_key_boundary_bits, then test_abi_modes_agree (SSB_SORT64
  against the packed default on key_boundary) and test_main_matches_checker.
- (tid, pos) keys over thousands of contigs, covered runs from a contig's first to its last base, targets on contigs without reads,
  on @SQ contigs missing from the FASTA and on unknown names: test_builder_places_the_layout, test_main_matches_checker.
- the target advance (the if-not-while skip) under a .spike table in `sort -k1,1 -k2,2n` order: test_lexicographic_table_goes_back,
  test_main_matches_checker[*-lexicographic].
- the FASTA in another order than @SQ, with extra contigs and without some @SQ contigs; per-shard upload of [lo_tid, hi_tid]:
  test_builder_places_the_layout, test_main_matches_checker, test_shards_through_the_main.
- cuts between contigs, inside runs of empty contigs and inside a contig; streamed pieces of many contigs:
  test_shard_cuts_fall_between_and_inside_contigs, test_shards_through_the_main, test_run_sharded_equals_single_run,
  test_streamed_host_run_equals_single_run.
- a BAM header with thousands of n_ref entries (host/bam_input.h): test_bam_input_of_grch38_like.

GPU (marked `gpu`): byte for byte against spike_cases.CHECKER on the SAM, the stats block and the full truth.vcf."""
import os
import re

import pytest

import layout_cases as lc
import spike_cases as sc
from test_spike_shapes import _envelope_errors, _first_diff, _kept_by_filter

SEED = 1
LAYOUT_ORDERS = [(l, o) for l in lc.LAYOUTS for o in lc.ORDERS]
TILE = 32768


@pytest.fixture(scope="module")
def layout(tmp_path_factory):
    """layout(name, order) -> (prefix, facts); each layout is built once, the second .spike order shares its .fa and .sam."""
    memo = {}

    def get(name, order="sam"):
        if (name, "sam") not in memo:
            d = tmp_path_factory.mktemp(name)
            memo[(name, "sam")] = lc.generate(str(d / "sam"), name, SEED)
        if (name, order) not in memo:
            prefix, facts = memo[(name, "sam")]
            memo[(name, order)] = (lc.respike(prefix, facts, order, os.path.join(os.path.dirname(os.path.dirname(prefix)), order)), facts)
        return memo[(name, order)]
    return get


def _load(prefix):
    from stochasticsim_b200 import spike as sp
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    return hdr, body, names, seqs, targets


def _survey(prefix):
    """What the written files hold, read back without the builder: per line (tid, pos, end, kept, rnext), the FASTA names in order."""
    sam = open(prefix + ".sam", "rb").read().decode()
    names = re.findall(r"^@SQ\tSN:(\S+)\tLN:(\d+)", sam, re.M)
    tid = {}
    for t, (n, _) in enumerate(names):
        tid.setdefault(n, t)
    body_at = sam.index("\n", sam.rindex("\n@") + 1) + 1 if "\n@" in sam else 0
    lines = []
    for line in sam[body_at:].split("\n"):
        if not line:
            continue
        f = line.split("\t")
        flag, mapq = int(f[1]), int(f[4])
        rlen = sum(int(a) for a, op in re.findall(r"(\d+)([MDN=X])", f[5]))
        kept = f[2] != "*" and not (flag & 0x704) and mapq >= 30 and not ((flag & 1) and not (flag & 2)) and rlen > 0
        t = tid.get(f[2], -1)
        lines.append((t, int(f[3]) - 1, int(f[3]) - 1 + rlen, kept, f[6], mapq, len(line) + 1))
    fasta = re.findall(r"^>(\S+)", open(prefix + ".fa").read(), re.M)
    return [n for n, _ in names], [int(l) for _, l in names], lines, fasta, body_at


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_builder_places_the_layout(name, layout):
    prefix, facts = layout(name)
    names, lens, lines, fasta, _ = _survey(prefix)
    assert names == facts["names"] and len(names) == facts["n_sq"] == {"grch38_like": 3366, "scaffolds": 12_000}.get(name, 4097)
    assert len(set(names)) == len(names)
    with_lines = {l[0] for l in lines if l[0] >= 0}
    with_kept = {l[0] for l in lines if l[3]}
    assert with_lines == with_kept == set(facts["covered"]), "contigs with reads are not the ones the builder covered"
    bare_runs = [b - a - 1 for a, b in zip(sorted(with_lines), sorted(with_lines)[1:])]
    # contigs whose whole length is covered by kept reads, first base to last
    for t in facts["full"]:
        cov = bytearray(lens[t])
        for l in lines:
            if l[0] == t and l[3]:
                cov[l[1]:l[2]] = b"\1" * (l[2] - l[1])
        assert all(cov), "%s is not covered base to base" % names[t]
    # every covered contig has a kept read on its first and on its last base
    first = {l[0] for l in lines if l[3] and l[1] == 0}
    last = {l[0] for l in lines if l[3] and l[2] == lens[l[0]]}
    assert first == last == with_kept - ({4096} if name.startswith("key_boundary") else set())
    # kept and dropped lines on both sides of MAPQ 30
    mq = {(l[3], l[5]) for l in lines}
    assert {(True, 30), (True, 60), (False, 29), (False, 0)} <= mq
    on = facts["on"]
    assert all(on[k] > 0 for k in ("covered", "contig_first", "contig_last", "no_reads", "unknown_name")), on
    if name == "grch38_like":
        kinds = {"random": [n for n in names if n.endswith("_random")], "un": [n for n in names if n.startswith("chrUn_") and not n.endswith("_decoy")],
                 "alt": [n for n in names if n.endswith("_alt")], "decoy": [n for n in names if n.endswith("_decoy")],
                 "hla": [n for n in names if n.startswith("HLA-")]}
        assert names[:25] == ["chr%d" % i for i in range(1, 23)] + ["chrX", "chrY", "chrM"] and "chrEBV" in names
        assert {k: len(v) for k, v in kinds.items()} == {"random": 42, "un": 127, "alt": 261, "decoy": 2385, "hla": 525}
        assert all("*" in n and ":" in n for n in kinds["hla"]) and "chr1_KI270706v1_random" in names
        assert {"chr1", "chr10", "chr1_KI270706v1_random"} <= set(names)                 # names that are prefixes of one another
        assert max(bare_runs) >= 24, "expected runs of dozens of @SQ contigs without reads"
        # mates on another contig: RNEXT names a decoy or HLA contig (or the primary one back); not proper, so dropped
        other = [l for l in lines if l[4] not in ("=", "*")]
        assert len(other) == 2 * facts["rnext_other"] and not any(l[3] for l in other)
        far = [l[4] for l in other if l[0] < 25]
        assert any(n.endswith("_decoy") for n in far) and any(n.startswith("HLA-") for n in far)
        assert all(n.endswith("_decoy") or n.startswith("HLA-") for n in far)
        # the FASTA: lexicographic, with contigs the header does not name and without @SQ contigs that carry no reads
        assert fasta != [n for n in names if n in set(fasta)] and fasta[:-3] == sorted(fasta[:-3])
        assert set(fasta) - set(names) == set(facts["extra"]) and len(facts["extra"]) == 3
        gone = set(names) - set(fasta)
        assert gone == {names[t] for t in facts["missing"]} and len(gone) == 6
        assert not {names.index(n) for n in gone} & with_lines
        assert on["missing_fa"] == 6
    else:
        assert fasta == names
    if name == "scaffolds":
        assert max(bare_runs) >= 2 and lc.key_bits(len(names), 0)[0] == 14
    if name.startswith("key_boundary"):
        assert names[-1] == "ctg4097" and lens[-1] > lc.KEY_POS and max(l[2] for l in lines if l[0] == 4096 and l[3]) >= lc.KEY_POS - 1


def test_scaffold_tiles_span_several_contigs(layout):
    """Nearly every 32 KiB tile of the scaffolds body holds lines of several contigs, so the tokeniser's per-tile reference window
    (staged for the tile's lowest tid) leaves the reads of the other contigs to the generic tally."""
    prefix, _ = layout("scaffolds")
    _, _, lines, _, _ = _survey(prefix)
    per_tile, off = {}, 0
    for l in lines:
        per_tile.setdefault(off // TILE, set()).add(l[0])
        off += l[6]
    spans = [len(s) for s in per_tile.values()]
    assert len(spans) > 500
    assert sum(s >= 3 for s in spans) >= 0.95 * len(spans), sorted(spans)[:20]


@pytest.mark.parametrize("name,bits", [("key_boundary", 32), ("key_boundary_plus1", 33)])
def test_key_boundary_bits(name, bits, layout):
    """From the input itself: 4,097 @SQ lines give tid_bits 13; the largest end of a kept read is 2^19 - 1 (pos_bits 19, packed
    32-bit keys with every bit used) or 2^19 (pos_bits 20, the 8-byte keys)."""
    prefix, facts = layout(name)
    names, _, lines, _, _ = _survey(prefix)
    max_end = max(l[2] for l in lines if l[3])
    assert max_end == facts["max_kept_end"] == lc.KEY_POS - 1 + (bits - 32)
    tid_bits, pos_bits = lc.key_bits(len(names), max_end)
    assert (tid_bits, pos_bits) == (13, 19 + bits - 32) and tid_bits + pos_bits == bits
    # a dropped read ends past 2^19 in both: only kept reads count
    assert max(l[2] for l in lines if l[0] >= 0) > lc.KEY_POS


@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_lexicographic_table_goes_back(name, layout):
    """`sort -k1,1 -k2,2n` next to karyotypic @SQ order: the table's contigs step back in @SQ order again and again (chr10..chr19
    before chr2, scaffold_10 before scaffold_2), while the `sam` table never does."""
    from stochasticsim_b200 import spike as sp
    steps = {}
    for order in lc.ORDERS:
        prefix, _ = layout(name, order)
        names = _survey(prefix)[0]
        recs = [(t, p) for _, t, p, _, _ in sp.parse_spike(open(prefix + ".spike", "rb").read(), names) if t >= 0]
        steps[order] = sum(b < a for a, b in zip(recs, recs[1:]))
        text = open(prefix + ".spike").read().splitlines()[1:]
        if order == "lexicographic":
            keys = [(l.split("\t")[0].encode(), int(l.split("\t")[1])) for l in text]
            assert keys == sorted(keys)
    assert steps["sam"] == 0
    assert steps["lexicographic"] >= 20, steps


@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_lines_are_in_the_envelope_and_sorted(name, layout):
    prefix, _ = layout(name)
    errs = _envelope_errors(open(prefix + ".sam", "rb").read())
    assert not errs, "\n".join(errs[:5])


@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_shard_cuts_fall_between_and_inside_contigs(name, layout):
    """ssb_spike_plan_shards on the body: the two-shard cut is the first line of a contig behind contigs without reads (the builder
    sizes the trailing unmapped line for that); of the five-shard cuts one falls inside a contig."""
    from stochasticsim_b200 import spike as sp
    prefix, facts = layout(name)
    hdr, body, names, _, _ = _load(prefix)
    kinds = set()
    for count in (2, 5):
        plan = sp.plan_shards(body, names, count, 600)
        assert len(plan) == count
        for (a, pa), (b, pb) in zip(plan, plan[1:]):
            last = pa[a.halo_bytes:].rstrip(b"\n").rsplit(b"\n", 1)[-1].split(b"\t")
            t_before, t_after = names.index(last[2].decode()), b.lo_tid
            assert (a.hi_tid, a.hi_pos) == (b.lo_tid, b.lo_pos)
            if t_before == t_after:
                kinds.add("inside")
            elif t_after - t_before >= 2:
                kinds.add("between_after_empty")
                if count == 2:
                    assert (t_before, t_after) == tuple(facts["cut"])
    assert kinds == {"inside", "between_after_empty"}, kinds


@pytest.mark.parametrize("name,order", LAYOUT_ORDERS)
def test_restatement_accepts_and_keeps_what_the_filter_keeps(name, order, layout, tmp_path):
    prefix, _ = layout(name, order)
    rc, out, sam, vcf, err = sc.run_cli(sc.ORACLE, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    assert rc == 0 and err == b"", err
    kept = _kept_by_filter(open(prefix + ".sam", "rb").read())
    assert sum(1 for l in sam.split(b"\n") if l and not l.startswith(b"@")) == kept
    assert b"alignmentCount (#reads) = %d," % kept in out
    assert vcf.count(b"\tNO_COVERAGE\t") > 0 and vcf.count(b"\tPASS\t") > 0


@pytest.mark.parametrize("name,order", LAYOUT_ORDERS)
def test_restatement_matches_reference_on_layouts(name, order, layout, tmp_path, ref_dir):
    """Every input the GPU tests below compare with CHECKER: the restatement against the unmodified reference over the shim."""
    if ref_dir is None or not os.path.exists(sc.REF):
        pytest.skip("oracle/_ref/stochasticSpike is not built (STOCHASTICSIM_SRC): the GPU tests compare with the restatement")
    prefix, _ = layout(name, order)
    a = sc.run_cli(sc.REF, prefix, str(tmp_path / "ref"))
    b = sc.run_cli(sc.ORACLE, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    assert a[0] == b[0] == 0
    assert a[2] == b[2], "SAM differs"
    assert a[3] == b[3], "truth.vcf differs"
    assert a[1] == b[1], "stdout differs"


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctx():
    import stochasticsim_b200 as ssb
    c = ssb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def checker(layout, tmp_path_factory):
    """checker(name, order) -> CHECKER's (rc, stdout, SAM, truth.vcf, stderr) on that input, run once."""
    memo = {}

    def get(name, order="sam"):
        if (name, order) not in memo:
            prefix, _ = layout(name, order)
            want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path_factory.mktemp("checker")), cmdname="stochasticSpike")
            assert want[0] == 0 and want[4] == b"", want[4]
            memo[(name, order)] = want
        return memo[(name, order)]
    return get


def _strip_cmd(vcf):
    return b"\n".join(l for l in vcf.split(b"\n") if not l.startswith(b"##stochasticSpikeCommand="))


def _main_parity(want, prefix, outdir, monkeypatch, env=None, sam=None):
    with monkeypatch.context() as m:
        for k, v in (env or {}).items():
            m.setenv(k, v)
        got = sc.run_cli(sc.PRODUCT, prefix, outdir, sam=sam)
    assert got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + _first_diff(want[2], got[2])
    assert got[1] == want[1], "stats differ: %r vs %r" % (want[1], got[1])
    if sam is None:
        assert got[3] == want[3], "truth.vcf differs: " + _first_diff(want[3], got[3])
    else:                                                       # the command line echoes the input's file name
        assert _strip_cmd(got[3]) == _strip_cmd(want[3]), "truth.vcf differs: " + _first_diff(_strip_cmd(want[3]), _strip_cmd(got[3]))


@pytest.mark.gpu
@pytest.mark.parametrize("name,order", LAYOUT_ORDERS)
def test_main_matches_checker(name, order, layout, checker, tmp_path, ctx, monkeypatch):
    prefix, _ = layout(name, order)
    _main_parity(checker(name, order), prefix, str(tmp_path / "gpu"), monkeypatch)


def _res_key(r):
    return (r.status, r.at_tid, r.at_pos, r.locus_index, r.filter, r.ref_cnt, r.mut_cnt, tuple(r.err_cnt), r.rng_offset, r.mutant_allele, r.ref_base)


def _se_key(e):
    return (e.tid, e.pos, e.locus_index, e.ref_cnt, tuple(e.err_cnt), e.ref_base)


@pytest.mark.gpu
@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_abi_modes_agree(name, layout, checker, ctx, monkeypatch):
    """Through the C ABI: the default run, the one-warp serial chain, chunked chains with chunks far smaller than a contig's reads
    (chunk boundaries meet contig boundaries), the generic tally without the exception list and the 8-byte output-order keys give
    the checker's SAM, the same per-target results (rng_offset included), draw count and SEQ_ERROR records.  On key_boundary the
    default packs its keys into 32 bits with every bit used, so SSB_SORT64 against the default checks the packed keys directly."""
    from stochasticsim_b200 import spike as sp
    prefix, _ = layout(name)
    want = checker(name)
    hdr, body, names, seqs, targets = _load(prefix)
    # chunks of 96 and 512 loci: each layout has hundreds of covered contigs per thousand chunks.  The phase-1 slices are left to
    # the run (96) or kept at the default's lower bound of 4096 offsets (512): a slice of a few offsets, as test_spike_shapes
    # forces on its 10^5-locus inputs, would ask here for over a million phase-1 blocks, more descriptors than the run's mapped
    # scratch holds (SSB_E_NOMEM)
    modes = [{}, {"SSB_CHAIN_SERIAL": "1"}, {"SSB_CHAIN_CHUNK": "96", "SSB_CHAIN_GROUP": "8"},
             {"SSB_CHAIN_CHUNK": "512", "SSB_CHAIN_GROUP": "4", "SSB_CHAIN_SLICE": "4096"}, {"SSB_NO_EXC_LIST": "1"}, {"SSB_SORT64": "1"}]
    runs = []
    with sp.Spike(ctx, names, seqs) as s:
        for env in modes:
            with monkeypatch.context() as m:
                for k, v in env.items():
                    m.setenv(k, v)
                try:
                    out, res, st = s.run_host(body, targets, 434)
                except Exception as e:
                    raise AssertionError("%s: %s" % (env, e)) from e
            runs.append((env, out, [_res_key(r) for r in res], st.rng_draws, st.chain_mode, [_se_key(e) for e in s.seq_errors()]))
    base = runs[1]
    assert base[4] == 1 and all(r[4] > 1 for r in runs[2:4]), ("expected the serial and the chunked chain", [r[4] for r in runs])
    assert any(r[0] == sp.T_HIT for r in base[2]) and any(r[0] == sp.T_NOCOV for r in base[2])
    for env, out, res, draws, mode, se in runs:
        assert hdr + out == want[2], "%s: SAM differs: %s" % (env, _first_diff(want[2], hdr + out))
        assert res == base[2], env
        assert draws == base[3], env
        assert se == base[5], env


@pytest.mark.gpu
@pytest.mark.parametrize("name", lc.LAYOUTS)
@pytest.mark.parametrize("shards", [2, 5])
def test_shards_through_the_main(name, shards, layout, checker, tmp_path, ctx, monkeypatch):
    """SSB_SHARDS coordinate shards on one device: each uploads only the contigs in [lo_tid, hi_tid]; the cuts fall between contigs
    behind empty ones and inside contigs (test_shard_cuts_fall_between_and_inside_contigs)."""
    prefix, _ = layout(name)
    _main_parity(checker(name), prefix, str(tmp_path / "gpu"), monkeypatch, env={"SSB_SHARDS": str(shards), "SSB_HALO": "600"})


@pytest.mark.gpu
@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_run_sharded_equals_single_run(name, layout, ctx):
    from stochasticsim_b200 import spike as sp
    prefix, _ = layout(name)
    hdr, body, names, seqs, targets = _load(prefix)
    with sp.Spike(ctx, names, seqs) as s:
        out1, res1, st1 = s.run_host(body, targets, 434)
        se1 = s.seq_errors()
    out, res, sts, se, n = sp.run_sharded([ctx], names, seqs, body, targets, 434, 5, 600)
    assert n == 5
    assert out == out1, "concatenated shard outputs differ from the single run"
    assert [_res_key(r) for r in res] == [_res_key(r) for r in res1]
    assert [_se_key(e) for e in se] == [_se_key(e) for e in se1]
    for f in ("alignmentCount", "numberOfLociCovered", "totalFoldCoverage"):
        assert sum(getattr(s_, f) for s_ in sts) == getattr(st1, f), f
    assert max(s_.maxDepth for s_ in sts) == st1.maxDepth
    for a, b in zip(sts, sts[1:]):
        assert a.rng_k_out == b.rng_k_in


@pytest.mark.gpu
@pytest.mark.parametrize("name", lc.LAYOUTS)
def test_streamed_host_run_equals_single_run(name, layout, ctx, monkeypatch):
    """The body streamed through the device in 40 pieces, each holding the lines of many contigs."""
    from stochasticsim_b200 import spike as sp
    prefix, facts = layout(name)
    hdr, body, names, seqs, targets = _load(prefix)
    piece = len(body) // 40
    assert len(facts["covered"]) >= 40 * 12
    with sp.Spike(ctx, names, seqs) as s:
        monkeypatch.setenv("SSB_NO_STREAM", "1")
        out1, res1, st1 = s.run_host(body, targets, 434)
        se1 = s.seq_errors()
        monkeypatch.delenv("SSB_NO_STREAM")
        monkeypatch.setenv("SSB_STREAM_BYTES", str(piece))
        out2, res2, st2 = s.run_host(body, targets, 434)
        se2 = s.seq_errors()
    assert st2.n_forwarded >= 3, "expected the body to be streamed in several pieces"
    assert out2 == out1
    assert [_res_key(r) for r in res2] == [_res_key(r) for r in res1]
    assert [_se_key(e) for e in se2] == [_se_key(e) for e in se1]
    for f in ("alignmentCount", "numberOfLociCovered", "totalFoldCoverage", "maxDepth", "rng_draws"):
        assert getattr(st2, f) == getattr(st1, f), f


@pytest.mark.gpu
def test_bam_input_of_grch38_like(layout, checker, tmp_path, ctx, monkeypatch):
    """A BAM whose header has 3,366 n_ref entries, HLA names among them, through the BAM reader: same SAM, stats and truth.vcf body."""
    import bam_writer
    prefix, _ = layout("grch38_like")
    bam = tmp_path / "in.bam"
    bam.write_bytes(bam_writer.sam_to_bam(open(prefix + ".sam", "rb").read()))
    (tmp_path / "in.bam.bai").write_bytes(b"BAI\1")
    _main_parity(checker("grch38_like"), prefix, str(tmp_path / "gpu"), monkeypatch, sam=str(bam))
