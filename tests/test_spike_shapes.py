"""The spike path on the alignment shapes real aligners write (tests/shape_cases.py): hard and soft clips, P, several indels per
read, I/D/N next to clips and to each other, long N skips, single-end and supplementary reads, every dropped flag kind, MAPQ at
the filter's boundary, RNEXT naming another @SQ, QUAL '*', and chains of up to eight reads of one QNAME over one locus.

GPU (marked `gpu`): the drop-in main and the C ABI against spike_cases.CHECKER, byte for byte on the SAM, the stats block and the
full truth.vcf.  CHECKER is the unmodified reference over the htslib shim (oracle/_ref/stochasticSpike) when it has been built;
without it the GPU path is compared with the CPU restatement (oracle/_build/spike_oracle), and
test_restatement_matches_reference_on_shape_inputs, which pins the restatement to the reference on these inputs, is skipped.
The pileup rules for the rarer shapes (an alignment that starts with I or D after its clip, D next to N, P) are htslib's as the
restatement and the shim state them (SURVEY App. D): they have not been checked against htslib itself here.

CPU: the builder places every shape and every kind of target, writes lines inside the pass-through envelope in coordinate
order, the restatement accepts every input and keeps exactly the lines read_bam's filter keeps, and the shifted inputs put
kept lines on each of the tokeniser's three routes: its fast parser, and its careful parser over the staged tile and over
global memory."""
import os
import re

import pytest

import shape_cases as sh
import spike_cases as sc

SEEDS = (1, 2, 3)
FAMILY_CASES = [(fam, seed) for fam in sh.FAMILIES + ("mixed",) for seed in SEEDS]
# bytes in front of the body: 0 = the plain mixed case, else one dropped line carrying a ZZ:Z: tag of that length
SHIFTS = (0, 1, 5, 13, 16381)
MIXED_SEED = 7


def _families(name):
    return sh.FAMILIES if name == "mixed" else (name,)


def _case(tmp_path, name, seed, shift=0):
    d = str(tmp_path / ("in_%s_%d_%d" % (name, seed, shift)))
    os.makedirs(d, exist_ok=True)
    return sh.generate(d, seed, _families(name), shift=shift)


def _first_diff(a, b):
    from test_spike_gpu import first_diff
    return first_diff(a, b)


# ------------------------------------------------------------------------------------------------ CPU
CIGAR_RE = re.compile(r"(?:[1-9][0-9]*[MIDNSHP=X])+")
INT_RE = re.compile(r"0|[1-9][0-9]*")


def _envelope_errors(sam: bytes):
    """Lines outside what htslib prints back unchanged, and lines out of coordinate order."""
    text = sam.decode()
    sq = re.findall(r"^@SQ\tSN:(\S+)", text, re.M)
    names = {}
    for tid, name in enumerate(sq):
        names.setdefault(name, tid)                             # the first @SQ of a name is its tid (sam_hdr_name2tid)
    errs, last = [], (-1, -1)
    for k, line in enumerate(l for l in text.split("\n") if l and not l.startswith("@")):
        f = line.split("\t")
        ok = len(f) >= 11 and 0 < len(f[0]) <= 254 and all(INT_RE.fullmatch(f[i]) for i in (1, 3, 4, 7))
        ok = ok and int(f[1]) < 65536 and int(f[4]) < 256 and re.fullmatch(r"-?(0|[1-9][0-9]*)", f[8]) and f[8] != "-0"
        ok = ok and (f[2] == "*" or f[2] in names) and (f[5] == "*" or CIGAR_RE.fullmatch(f[5]))
        ok = ok and (f[6] in ("*", "=") or (f[6] in names and f[6] != f[2])) and not (f[6] == "=" and f[2] == "*")
        ok = ok and (f[9] == "*" or re.fullmatch(r"[=ACMGRSVTWYHKDBN]+", f[9]))
        if ok and f[5] != "*" and f[9] != "*":
            ok = sum(int(n) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", f[5]) if op in "MIS=X") == len(f[9])
        ok = ok and (f[10] == "*" or (len(f[10]) == len(f[9]) and all("!" <= c <= "~" for c in f[10])))
        ok = ok and all(re.fullmatch(r"[A-Za-z][A-Za-z0-9]:(i:-?(0|[1-9][0-9]*)|Z:[ -~]*)", t) for t in f[11:])
        if not ok:
            errs.append("line %d outside the envelope: %s" % (k, line[:200]))
        key = (names.get(f[2], len(sq)), int(f[3]))
        if key < last:
            errs.append("line %d out of order: %s" % (k, line[:200]))
        last = key
    return errs


def _kept_by_filter(sam: bytes):
    """Alignment lines read_bam (stochasticSpike.c:243-268) keeps and the pileup writes: mapped, none of 4/256/512/1024, MAPQ >= 30,
    proper if paired, consuming reference."""
    n = 0
    for line in sam.split(b"\n"):
        if not line or line.startswith(b"@"):
            continue
        f = line.split(b"\t")
        flag, mapq = int(f[1]), int(f[4])
        rlen = sum(int(a) for a, op in re.findall(rb"(\d+)([MDN=X])", f[5]))
        if f[2] != b"*" and not (flag & (4 | 256 | 512 | 1024)) and mapq >= 30 and not ((flag & 1) and not (flag & 2)) and rlen:
            n += 1
    return n


@pytest.mark.parametrize("name", sh.FAMILIES + ("mixed",))
def test_builder_places_every_shape(name, tmp_path):
    for seed in SEEDS:
        prefix, shapes, on = _case(tmp_path, name, seed)
        for fam in _families(name):
            missing = [s for s in sh.FAMILY_SHAPES[fam] if not shapes.get(s)]
            assert not missing, "seed %d: shapes never placed: %s" % (seed, missing)
            bare = [s for s in sh.FAMILY_SPOTS[fam] + sh.COMMON_SPOTS if not on.get(s)]
            assert not bare, "seed %d: no target on: %s" % (seed, bare)


@pytest.mark.parametrize("name,seed", FAMILY_CASES)
def test_builder_lines_are_in_the_envelope_and_sorted(name, seed, tmp_path):
    prefix, _, _ = _case(tmp_path, name, seed)
    sam = open(prefix + ".sam", "rb").read()
    errs = _envelope_errors(sam)
    assert not errs, "\n".join(errs[:5])
    if name == "mixed":
        assert len(sam) > 300_000


@pytest.mark.parametrize("name,seed,shift", [(n, s, 0) for n, s in FAMILY_CASES] + [("mixed", MIXED_SEED, k) for k in SHIFTS])
def test_restatement_accepts_and_keeps_what_the_filter_keeps(name, seed, shift, tmp_path):
    prefix, _, _ = _case(tmp_path, name, seed, shift)
    rc, out, sam, vcf, err = sc.run_cli(sc.ORACLE, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    assert rc == 0 and err == b"", err
    kept = _kept_by_filter(open(prefix + ".sam", "rb").read())
    assert sum(1 for l in sam.split(b"\n") if l and not l.startswith(b"@")) == kept
    assert b"alignmentCount (#reads) = %d," % kept in out


def test_shifts_put_kept_lines_on_every_tokeniser_path(tmp_path):
    """The shifted mixed inputs move every line against the 32 KiB tiles: kept MAPQ-30 lines, kept QUAL '*' lines and kept lines
    with H / P reach the common-shape parser, the careful parser over the staged tile (lines beyond the tile's parsing threads) and
    the careful parser over global memory (lines that end past the staged overhang), so a slip on any route shows."""
    seen = {"mapq30": set(), "qualstar": set(), "hp": set()}
    global_shifts = 0
    for k in SHIFTS:
        prefix, _, _ = _case(tmp_path, "mixed", MIXED_SEED, k)
        body = _load(prefix)[1]
        paths = sh.tokeniser_paths(body)
        global_shifts += any(p == "global" for _, p in paths)
        for s, p in paths:
            f = body[s:body.find(b"\n", s)].split(b"\t")
            flag = int(f[1])
            kept = f[2] != b"*" and not (flag & 0x704) and int(f[4]) >= 30 and not ((flag & 1) and not (flag & 2))
            if not kept:
                continue
            if f[4] == b"30":
                seen["mapq30"].add(p)
            if f[10] == b"*":
                seen["qualstar"].add(p)
            if b"H" in f[5] or b"P" in f[5]:
                seen["hp"].add(p)
    assert seen["mapq30"] == {"conv", "staged", "global"}, seen
    assert {"conv", "staged"} <= seen["qualstar"] and {"conv", "staged"} <= seen["hp"], seen
    assert global_shifts >= 1


@pytest.mark.parametrize("name,seed,shift", [(n, s, 0) for n, s in FAMILY_CASES] + [("mixed", MIXED_SEED, k) for k in SHIFTS])
def test_restatement_matches_reference_on_shape_inputs(name, seed, shift, tmp_path, ref_dir):
    """Every input the GPU tests below compare with CHECKER: the restatement against the unmodified reference over the shim."""
    if ref_dir is None or not os.path.exists(sc.REF):
        pytest.skip("oracle/_ref/stochasticSpike is not built (STOCHASTICSIM_SRC): the GPU tests compare with the restatement")
    prefix, _, _ = _case(tmp_path, name, seed, shift)
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


def _cli_parity(prefix, outdir, env=None, sam=None):
    want = sc.run_cli(sc.CHECKER, prefix, os.path.join(outdir, "ora"), cmdname="stochasticSpike")
    saved = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        got = sc.run_cli(sc.PRODUCT, prefix, os.path.join(outdir, "gpu"), sam=sam)
    finally:
        for k, v in saved.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    assert want[0] == 0 and want[4] == b"", want[4]
    assert got[0] == 0, got[4]
    assert got[2] == want[2], "SAM differs: " + _first_diff(want[2], got[2])
    assert got[1] == want[1], "stats differ: %r vs %r" % (want[1], got[1])
    return want, got


@pytest.mark.gpu
@pytest.mark.parametrize("name,seed", FAMILY_CASES)
def test_shape_family_parity(name, seed, tmp_path, ctx):
    prefix, _, _ = _case(tmp_path, name, seed)
    want, got = _cli_parity(prefix, str(tmp_path))
    assert got[3] == want[3], "truth.vcf differs: " + _first_diff(want[3], got[3])


@pytest.mark.gpu
@pytest.mark.parametrize("shift", SHIFTS)
def test_every_line_through_every_tokeniser_path(shift, tmp_path, ctx):
    """The mixed case shifted against the 32 KiB tiles (see test_shifts_put_kept_lines_on_every_tokeniser_path)."""
    prefix, _, _ = _case(tmp_path, "mixed", MIXED_SEED, shift)
    want, got = _cli_parity(prefix, str(tmp_path))
    assert got[3] == want[3], "truth.vcf differs: " + _first_diff(want[3], got[3])


def _load(prefix):
    from stochasticsim_b200 import spike as sp
    sam = open(prefix + ".sam", "rb").read()
    hdr, body, names = sp.split_header(sam)
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    return hdr, body, names, seqs, targets


@pytest.mark.gpu
def test_chain_modes_agree(tmp_path, ctx, monkeypatch):
    """The one-warp serial chain, the chunked chain at small geometries, the tally_fast_kernel fallback (no exception list) and the
    8-byte end-order keys: same SAM (the checker's), same per-target results, draw count and SEQ_ERROR records."""
    from stochasticsim_b200 import spike as sp
    prefix, _, _ = _case(tmp_path, "mixed", MIXED_SEED)
    want = sc.run_cli(sc.CHECKER, prefix, str(tmp_path / "ora"), cmdname="stochasticSpike")
    assert want[0] == 0
    hdr, body, names, seqs, targets = _load(prefix)
    modes = [{"SSB_CHAIN_SERIAL": "1"}, {"SSB_CHAIN_CHUNK": "512", "SSB_CHAIN_GROUP": "4", "SSB_CHAIN_SLICE": "4096"},
             {"SSB_CHAIN_CHUNK": "96", "SSB_CHAIN_GROUP": "8", "SSB_CHAIN_SLICE": "3"}, {"SSB_NO_EXC_LIST": "1"}, {"SSB_SORT64": "1"}]
    key = lambda r: (r.status, r.at_tid, r.at_pos, r.filter, r.ref_cnt, r.mut_cnt, tuple(r.err_cnt), r.rng_offset, r.mutant_allele)
    se_key = lambda e: (e.tid, e.pos, e.locus_index, e.ref_cnt, tuple(e.err_cnt), e.ref_base)
    runs = []
    with sp.Spike(ctx, names, seqs) as s:
        for env in modes:
            with monkeypatch.context() as m:
                for k, v in env.items():
                    m.setenv(k, v)
                out, res, st = s.run_host(body, targets, 434)
            runs.append((env, out, [key(r) for r in res], st.rng_draws, st.chain_mode, [se_key(e) for e in s.seq_errors()]))
    base = runs[0]
    assert base[4] == 1
    assert any(r[4] > 1 for r in runs[1:3]), "expected the chunked chain to be used"
    assert len(base[5]) > 0 and any(r[0] == sp.T_HIT for r in base[2])
    for env, out, res, draws, mode, se in runs:
        assert hdr + out == want[2], "%s: SAM differs: %s" % (env, _first_diff(want[2], hdr + out))
        assert res == base[2], env
        assert draws == base[3], env
        assert se == base[5], env


@pytest.mark.gpu
def test_bam_input_of_the_mixed_case(tmp_path, ctx):
    """H, P, QUAL '*', RNAME '*' and RNEXT naming another @SQ through the BAM reader: same SAM, stats and truth.vcf body."""
    import bam_writer
    prefix, _, _ = _case(tmp_path, "mixed", MIXED_SEED)
    bam = tmp_path / "in.bam"
    bam.write_bytes(bam_writer.sam_to_bam(open(prefix + ".sam", "rb").read()))
    (tmp_path / "in.bam.bai").write_bytes(b"BAI\1")
    want, got = _cli_parity(prefix, str(tmp_path), sam=str(bam))
    strip = lambda v: b"\n".join(l for l in v.split(b"\n") if not l.startswith(b"##stochasticSpikeCommand="))
    assert strip(got[3]) == strip(want[3]), _first_diff(strip(want[3]), strip(got[3]))


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"SSB_SHARDS": "2", "SSB_HALO": "8000"}, {"SSB_SHARDS": "3", "SSB_HALO": "8000"}, {"SSB_STREAM_BYTES": "stream"}],
                         ids=["shards2", "shards3", "stream"])
def test_shards_and_streaming(env, tmp_path, ctx):
    """Coordinate shards (halo wider than the longest N skip) and a body streamed in a dozen pieces: supplementary alignments on the
    other contig and long skips cross the cuts."""
    prefix, _, _ = _case(tmp_path, "mixed", MIXED_SEED)
    if env.get("SSB_STREAM_BYTES") == "stream":
        body = _load(prefix)[1]
        env = {"SSB_STREAM_BYTES": str(len(body) // 12)}
    want, got = _cli_parity(prefix, str(tmp_path), env=env)
    assert got[3] == want[3], "truth.vcf differs: " + _first_diff(want[3], got[3])


@pytest.mark.gpu
def test_eight_same_name_reads_are_accepted(tmp_path, ctx):
    """Eight mutually overlapping alignments of one QNAME: the most tally_kernel takes (spike.cu, the cplx branch)."""
    d = tmp_path / "in"
    d.mkdir()
    prefix = sh.chain_case(str(d), 5, 8)
    want, got = _cli_parity(prefix, str(tmp_path))
    assert got[3] == want[3], "truth.vcf differs: " + _first_diff(want[3], got[3])


@pytest.mark.gpu
@pytest.mark.parametrize("size,seq_star", [(9, False), (2, True)], ids=["nine_same_name", "kept_seq_star"])
def test_documented_refusals(size, seq_star, tmp_path, ctx):
    """Nine mutually overlapping alignments of one QNAME, and a kept read whose SEQ is '*' (the reference would read outside the
    read's bases), are refused with SSB_E_FORMAT (exit status 3 from the main), never miscounted."""
    import stochasticsim_b200 as ssb
    from stochasticsim_b200 import spike as sp
    d = tmp_path / "in"
    d.mkdir()
    prefix = sh.chain_case(str(d), 5, size, seq_star=seq_star)
    got = sc.run_cli(sc.PRODUCT, prefix, str(tmp_path / "gpu"))
    assert got[0] == 3 and b"precondition" in got[4], (got[0], got[4])
    hdr, body, names, seqs, targets = _load(prefix)
    with sp.Spike(ctx, names, seqs) as s:
        with pytest.raises(ssb.SSBError) as e:
            s.run_host(body, targets, 434)
    assert e.value.code == -5
