"""Seeded spike inputs in the reference layouts real genomes have and tools/gen_synth.c and tests/shape_cases.py never make:
thousands of @SQ lines, names with '_', '*' and ':' that are prefixes of one another, runs of contigs without reads, a FASTA in
another order than @SQ (with contigs the header does not name, and without some it does), .spike tables in @SQ order and in
`sort -k1,1 -k2,2n` order, and the 32-bit boundary of the packed output-order keys (spike_run.cuh: tid_bits + pos_bits <= 32).

generate() writes <outdir>/in.{fa,sam,spike} like spike_cases.generate (so spike_cases.run_cli takes the prefix unchanged) and
returns (prefix, facts): what the builder placed.  The reads come from shape_cases._Builder (plain pairs, MAPQ, coverage
bookkeeping); the files are written here because the layouts need control over the FASTA order and the .spike order.
Every line is inside the pass-through envelope (DESIGN.md section 5), so a refusal is a bug, not an artefact of the input."""
import math
import os
import random
import re

import shape_cases as sh

LAYOUTS = ("grch38_like", "scaffolds", "key_boundary", "key_boundary_plus1")
ORDERS = ("sam", "lexicographic")
KEY_POS = 1 << 19                    # key_boundary: the largest kept end is KEY_POS - 1; key_boundary_plus1 adds one read ending at KEY_POS
_ACGT = bytes.maketrans(bytes(range(256)), b"ACGT" * 64)


def key_bits(n_sq, max_end):
    """tid_bits and pos_bits as run_shard chooses them for the output-order keys (spike_run.cuh, after the compaction)."""
    tid_bits = 0
    while (1 << tid_bits) < n_sq and tid_bits < 31:
        tid_bits += 1
    pos_bits = 1
    while pos_bits < 32 and (1 << pos_bits) <= max_end:
        pos_bits += 1
    return tid_bits, pos_bits


def _seq(rng, n):
    s = rng.randbytes(n).translate(_ACGT).decode()
    if n >= 2000:                                          # one soft-masked run and one N run
        a, l = rng.randrange(0, n - 400), rng.randrange(50, 400)
        s = s[:a] + s[a:a + l].lower() + s[a + l:]
        a, l = rng.randrange(300, n - 300), rng.randrange(5, 120)
        s = s[:a] + "N" * l + s[a + l:]
    return s


def _loguniform(rng, lo, hi):
    return max(lo, int(math.exp(rng.uniform(math.log(lo), math.log(hi)))))


# ------------------------------------------------------------------------------------------------ contig lists
def _grch38_names(rng):
    """The name kinds of GRCh38_full_analysis_set_plus_decoy_hla in its order: 25 primary, 42 _random, 127 chrUn_, chrEBV,
    261 _alt, 2,385 _decoy and 525 HLA contigs (3,366 @SQ lines)."""
    prim = ["chr%d" % i for i in range(1, 23)] + ["chrX", "chrY", "chrM"]
    karyo = prim[:24]
    acc = iter(range(270000, 272000))
    rnd = ["%s_KI%06dv1_random" % (karyo[i % 24], next(acc)) for i in range(39)] + ["chr1_KI270706v1_random", "chr17_GL000205v2_random", "chr22_KI270731v1_random"]
    rnd.sort(key=lambda n: karyo.index(n.split("_")[0]))
    un = ["chrUn_KI%06dv1" % next(acc) for _ in range(100)] + ["chrUn_GL%06dv1" % (226 + k) for k in range(27)]
    alt = ["%s_%s%06dv1_alt" % (karyo[i % 24], rng.choice(["KI", "GL"]), next(acc)) for i in range(261)]
    alt.sort(key=lambda n: karyo.index(n.split("_")[0]))
    decoy = ["chrUn_JTFH01%06dv1_decoy" % k for k in range(1, 2386)]
    hla, genes = [], ["A", "B", "C", "DQA1", "DQB1", "DRB1"]
    while len(hla) < 525:
        g = genes[len(hla) * len(genes) // 525]
        f = ["%02d" % rng.randrange(1, 58), "%02d" % rng.randrange(1, 40)] + ["%02d" % rng.randrange(1, 12) for _ in range(rng.randrange(0, 3))]
        n = "HLA-%s*%s%s" % (g, ":".join(f), rng.choice(["", "", "", "", "N", "Q"]))
        if n not in hla:
            hla.append(n)
    hla.sort(key=lambda n: (genes.index(n[4:n.index("*")]), n))
    return prim, rnd + un + ["chrEBV"] + alt + decoy + hla


def _cover_contig(b, tid, step, full=False):
    """Plain pairs along one contig (one every `step` bases), with its first and its last base covered; `full` covers every base."""
    n = len(b.contigs[tid][1])
    if full:
        for f in list(range(0, n - 200, 100)) + [n - 200]:
            b.pair(tid, f, [(100, "M")], [(100, "M")], 200)
        return
    for f in range(0, n, step):
        f = min(n - 1, f + b.rng.randrange(0, 40))
        L1, L2 = b.rng.randrange(60, 151), b.rng.randrange(60, 151)
        fl = b.rng.randrange(max(L1, L2), 450)
        if f + fl <= n:
            b.pair(tid, f, b.plain_ops(L1), b.plain_ops(L2), fl, mapq=b.rng.choice([(60, 60), (60, 60), (29, 60), (30, 30), (60, 0)]))
    b.pair(tid, 0, [(100, "M")], [(100, "M")], 260)
    b.pair(tid, n - 300, [(100, "M")], [(100, "M")], 300)


def _other_contig_mates(b, prim, others, count):
    """Pairs whose mates sit on two contigs (RNEXT names the other one): not proper, so the filter drops both, but both are parsed."""
    for _ in range(count):
        t1, t2 = b.rng.choice(prim), b.rng.choice(others)
        n1, n2 = len(b.contigs[t1][1]), len(b.contigs[t2][1])
        p1, p2 = b.rng.randrange(0, n1 - 150), b.rng.randrange(0, n2 - 150)
        name, L = b.qname(), b.rng.randrange(60, 151)
        b.add(name, 97, t1, p1, b.rng.choice([29, 30, 60]), [(L, "M")], b.contigs[t2][0], p2 + 1, 0)
        b.add(name, 145, t2, p2, b.rng.choice([0, 30, 60]), [(L, "M")], b.contigs[t1][0], p1 + 1, 0)


# ------------------------------------------------------------------------------------------------ layouts
def _grch38_like(rng, facts):
    prim, rest = _grch38_names(rng)
    contigs = [(n, _seq(rng, rng.randrange(8_000, 40_001))) for n in prim] + [(n, _seq(rng, _loguniform(rng, 400, 6000))) for n in rest]
    b = sh._Builder(rng, contigs)
    b.gaps = [(0, 0)] * len(contigs)
    covered = list(range(len(prim))) + sorted(rng.sample(range(len(prim), len(contigs)), (len(contigs) - len(prim)) // 7))
    full = set(rng.sample(covered[len(prim):], 12)) | {len(prim) - 1}                # chrM and a dozen small contigs, base to base
    for t in covered:
        _cover_contig(b, t, 100, full=t in full)
    far = [t for t in covered if t >= len(prim) and (b.contigs[t][0].endswith("_decoy") or b.contigs[t][0].startswith("HLA-"))]
    _other_contig_mates(b, list(range(len(prim))), far, 300)
    bare = [t for t in range(len(prim), len(contigs)) if t not in set(covered)]
    missing = set(rng.sample(bare, 6))
    fasta = sorted(n for k, (n, _) in enumerate(contigs) if k not in missing)
    extra = [("chrUn_JTFH01999001v1_decoy", _seq(rng, 900)), ("HLA-DRB1*99:01:01", _seq(rng, 1200)), ("chr1_KI279999v1_alt", _seq(rng, 700))]
    facts.update(full=sorted(full), missing=sorted(missing), extra=[n for n, _ in extra], rnext_other=300)
    return b, covered, fasta, extra


def _scaffolds(rng, facts):
    contigs = [("scaffold_%d" % (k + 1), _seq(rng, _loguniform(rng, 300, 3000))) for k in range(12_000)]
    b = sh._Builder(rng, contigs)
    b.gaps = [(0, 0)] * len(contigs)
    covered = sorted(rng.sample(range(len(contigs)), int(len(contigs) * 0.8)))
    full = set(rng.sample(covered, 100))
    for t in covered:
        _cover_contig(b, t, 500, full=t in full)
    facts.update(full=sorted(full), missing=[], extra=[], rnext_other=0)
    return b, covered, [n for n, _ in contigs], []


def _key_boundary(rng, facts):
    contigs = [("ctg%d" % (k + 1), _seq(rng, rng.randrange(300, 1201))) for k in range(4096)]
    contigs.append(("ctg4097", _seq(rng, KEY_POS + 3000)))                      # tid 4096: the top bit of a 13-bit tid
    b = sh._Builder(rng, contigs)
    b.gaps = [(0, 0)] * len(contigs)
    covered = sorted(rng.sample(range(4096), 2048))
    for t in covered:
        _cover_contig(b, t, 300)
    last, end = 4096, KEY_POS - 1
    for f in range(end - 4000, end - 450, 60):                                      # the last few kb below KEY_POS - 1
        L1, L2 = rng.randrange(60, 151), rng.randrange(60, 151)
        b.pair(last, f, b.plain_ops(L1), b.plain_ops(L2), rng.randrange(max(L1, L2), 450))
    b.pair(last, end - 300, [(100, "M")], [(100, "M")], 300)                         # the kept read that ends at KEY_POS - 1
    b.add(b.qname(), 1024, last, KEY_POS + 100, 60, [(100, "M")])                     # dropped (duplicate): its end does not count
    covered.append(last)
    facts.update(full=[], missing=[], extra=[], rnext_other=0)
    return b, covered, [n for n, _ in contigs], []


_LAYOUT = {"grch38_like": _grch38_like, "scaffolds": _scaffolds, "key_boundary": _key_boundary, "key_boundary_plus1": _key_boundary}


# ------------------------------------------------------------------------------------------------ targets
def _targets(b, covered, missing, unknown):
    """(name, pos, sort tid) of the targets: covered loci of many contigs, the first and last base of contigs, contigs without reads,
    @SQ contigs missing from the FASTA, and names not in @SQ."""
    rng, nc = b.rng, len(b.contigs)
    kinds = {"covered": set(), "contig_first": set(), "contig_last": set(), "no_reads": set(), "missing_fa": set(), "unknown_name": set()}
    cov = set(covered)
    for t in rng.sample(covered, min(len(covered), 400)):
        s = b.cover[t]
        for x in rng.sample(range(len(s)), 3):
            if s[x]:
                kinds["covered"].add((t, x))
    for t in rng.sample(range(nc), min(nc, 300)) + covered[:3] + covered[-3:]:
        kinds["contig_first"].add((t, 0))
        kinds["contig_last"].add((t, len(b.contigs[t][1]) - 1))
    bare = [t for t in range(nc) if t not in cov and t not in missing]
    for t in rng.sample(bare, min(len(bare), 60)):
        kinds["no_reads"].add((t, rng.randrange(len(b.contigs[t][1]))))
    for t in missing:
        kinds["missing_fa"].add((t, rng.randrange(len(b.contigs[t][1]))))
    out = {}
    for kind in kinds:
        for t, x in sorted(kinds[kind]):
            out.setdefault((b.contigs[t][0], x), (t, kind))
    for name in unknown:                                    # ordered in the @SQ table next to a random contig
        out[(name, rng.randrange(1, 5000))] = (rng.randrange(nc), "unknown_name")
        kinds["unknown_name"].add(name)
    recs = []
    for (name, x), (t, kind) in out.items():
        real = name in b.contigs.index_of and t not in missing
        ref = b.contigs[t][1][x].upper() if real else "N"
        alt = rng.choice([".", ".", ".", rng.choice([c for c in "ACGT" if c != ref])])
        af = rng.choice(["1", "%.3g" % rng.uniform(0.05, 0.95), "%.3g" % rng.uniform(0.3, 0.95)])
        recs.append((t, x, name, alt, af, kind))
    recs.sort()
    return [r[2:] + (r[0], r[1]) for r in recs], {k: len(v) for k, v in kinds.items()}


def spike_text(targets, order):
    """The .spike table: `sam` follows the @SQ order, `lexicographic` is `LC_ALL=C sort -k1,1 -k2,2n` of the same lines."""
    recs = [(name, pos, alt, af) for name, alt, af, kind, t, pos in targets]
    if order == "lexicographic":
        recs.sort(key=lambda r: (r[0].encode(), r[1]))
    elif order != "sam":
        raise ValueError(order)
    return "#CHROM\tPOS\tALT\tAF\n" + "".join("%s\t%d\t%s\t%s\n" % (n, p + 1, a, f) for n, p, a, f in recs)


# ------------------------------------------------------------------------------------------------ output
def _line_start(body, p):
    if p == 0:
        return 0
    q = body.find(b"\n", p - 1)
    return len(body) if q < 0 else q + 1


def _tail_line(k):
    return "\t".join(["SRR0742.0", "4", "*", "0", "0", "*", "*", "0", "0", "*", "*", "ZZ:Z:" + "x" * k]) + "\n"


def _align_cut(b, body):
    """An unplaced unmapped line at the end (dropped by the filter; it never cuts), sized so that ssb_spike_plan_shards' cut for two
    shards (the first line at or after half the body) is the first line of a contig that follows contigs without reads: that cut
    lies between contigs, inside a run of empty ones.  Returns (tail bytes, (tid before the cut, tid after it))."""
    starts = [0] + [i + 1 for i in range(len(body) - 1) if body[i] == 10]
    tids = [b.contigs.index_of[body[s:body.index(b"\n", s)].split(b"\t", 3)[2].decode()] for s in starts]
    base = len(_tail_line(0))
    for i in range(1, len(starts)):
        k0 = 2 * starts[i] - len(body) - base
        if tids[i] - tids[i - 1] < 2 or k0 < 4:
            continue
        for k in range(k0 - 4, k0 + 4):
            full = body + _tail_line(k).encode()
            if _line_start(full, len(full) // 2) == starts[i]:
                return _tail_line(k).encode(), (tids[i - 1], tids[i])
    raise AssertionError("no contig change to cut at")


class _Names(list):
    """[(name, sequence)] with an index by name."""
    def __init__(self, items):
        super().__init__(items)
        self.index_of = {n: i for i, (n, _) in enumerate(items)}


def generate(outdir, layout, seed, spike_order="sam"):
    """Writes <outdir>/in.{fa,sam,spike}; returns (prefix, facts).  facts: n_sq, names, covered (tids with reads), full (tids covered
    base to base), missing (@SQ tids absent from the FASTA), extra (FASTA names absent from @SQ), fasta_order, targets
    [(name, alt, af, kind, sort tid, pos)] in @SQ order, on (targets per kind), max_kept_end, cut (tids either side of the
    two-shard cut)."""
    rng = random.Random(seed)
    facts = {"layout": layout}
    b, covered, fasta, extra = _LAYOUT[layout](rng, facts)
    b.contigs = _Names(b.contigs)
    unknown = ["chr23", "chrUn_JTFH01999001v1_decoy", "HLA-A*99:99:99", "chr1_KI270706v1", "scaffold_0", "ctg0"]
    targets, on = _targets(b, covered, set(facts["missing"]), unknown)
    if layout == "key_boundary_plus1":
        b.rng = random.Random(seed + 1)
        b.pair(len(b.contigs) - 1, KEY_POS - 300, [(100, "M")], [(100, "M")], 300)   # the one kept read that ends at KEY_POS
    os.makedirs(outdir, exist_ok=True)
    prefix = os.path.join(outdir, "in")
    seqs = dict(b.contigs)
    seqs.update(extra)
    with open(prefix + ".fa", "w") as f:
        for name in fasta + [n for n, _ in extra]:
            s = seqs[name]
            f.write(">%s\n" % name + "\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + "\n")
    body = "".join(l[3] + "\n" for l in sorted(b.lines)).encode()
    tail, cut = _align_cut(b, body)
    with open(prefix + ".sam", "wb") as f:
        f.write(b"@HD\tVN:1.6\tSO:coordinate\n")
        f.write("".join("@SQ\tSN:%s\tLN:%d\n" % (n, len(s)) for n, s in b.contigs).encode())
        f.write(b"@RG\tID:grp1\tSM:LY%d\n@PG\tID:bwa\tPN:bwa\tVN:0.7.17\n" % seed)
        f.write(body + tail)
    with open(prefix + ".spike", "w") as f:
        f.write(spike_text(targets, spike_order))
    kept_end = max((p + sh.span(o) for p, o in _kept_alignments(b)), default=0)
    facts.update(n_sq=len(b.contigs), names=[n for n, _ in b.contigs], covered=covered, fasta_order=fasta + [n for n, _ in extra],
                 targets=targets, on=on, max_kept_end=kept_end, cut=cut)
    return prefix, facts


def _kept_alignments(b):
    """(pos, ops) of the lines read_bam's filter keeps, from the builder's own records."""
    for _, _, _, text in b.lines:
        f = text.split("\t")
        flag, mapq = int(f[1]), int(f[4])
        if f[2] != "*" and not (flag & 0x704) and mapq >= 30 and not ((flag & 1) and not (flag & 2)) and f[5] != "*":
            yield int(f[3]) - 1, [(int(n), op) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", f[5])]


def respike(prefix, facts, order, outdir):
    """The same input with the other .spike table: <outdir>/in.{fa,sam} link to `prefix`'s, in.spike is written in `order`."""
    os.makedirs(outdir, exist_ok=True)
    out = os.path.join(outdir, "in")
    for ext in (".fa", ".sam"):
        if not os.path.exists(out + ext):
            os.symlink(os.path.abspath(prefix + ext), out + ext)
    with open(out + ".spike", "w") as f:
        f.write(spike_text(facts["targets"], order))
    return out
