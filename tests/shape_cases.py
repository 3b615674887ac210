"""Seeded spike inputs in the alignment shapes real aligners (BWA-MEM, minimap2, STAR) write and tools/gen_synth.c never does:
M mixed with =/X, clips at both ends with H outside S, P, several indels per read (I next to D), I/D/N next to clips, short and
long (> 4096) N skips, single-end and supplementary reads, dropped flag kinds, placed unmapped reads, MAPQ 29/30/255, RNEXT
naming another @SQ, QUAL '*', and 3- to 8-read chains of one QNAME over one locus.

generate() writes <outdir>/in.{fa,sam,spike} like spike_cases.generate (so spike_cases.run_cli takes the prefix unchanged) and
returns (prefix, shapes, on_targets): how many times each shape was placed, and how many targets sit on each kind of spot.
Every line is inside the pass-through envelope (DESIGN.md section 5: canonical integers, RNEXT '=' for the same contig,
upper-case IUPAC SEQ), so a refusal is a bug, not an artefact of the input."""
import os
import random
from collections import Counter, defaultdict

FAMILIES = ("cigar", "flags", "chains", "qualstar")
TILE, OVERHANG, PARSERS = 32768, 3072, 96          # the tokeniser's tile, staged overhang and parsing threads (sam_parse.cuh)
QCH = "#+5:?AFFIII"
# shapes each family must place (the tests assert every count is non-zero)
FAMILY_SHAPES = {
    "cigar": ["M_mixed", "lead_S", "trail_S", "H_lead", "H_trail", "P", "multi_indel", "I_then_D", "D_then_I", "I_after_clip",
              "D_N_adjacent", "D_next_to_clip", "N_next_to_clip", "N_short", "N_long"],
    "flags": ["single_end_0", "single_end_16", "supp_same_contig", "supp_other_contig", "secondary", "duplicate", "qc_fail",
              "not_proper", "placed_unmapped", "mate_unmapped", "mapq_29", "mapq_30", "mapq_255", "rnext_other", "rnext_star",
              "long_line", "unplaced_unmapped"],
    "chains": ["chain_3", "chain_5", "chain_8"],
    "qualstar": ["qualstar_simple", "qualstar_nonsimple", "qualstar_mate_differs"],
}
# kinds of target spots each family must carry targets on
FAMILY_SPOTS = {
    "cigar": ["read_first", "read_last", "before_I", "after_I", "in_D", "next_to_D", "in_N"],
    "flags": ["supplementary", "mapq_30"],
    "chains": ["chain"],
    "qualstar": ["qualstar"],
}
COMMON_SPOTS = ["contig_first", "contig_last", "uncovered"]


def cigar_str(ops):
    return "".join("%d%s" % (n, op) for n, op in ops) if ops else "*"


def span(ops):
    return sum(n for n, op in ops if op in "M=XDN")


def qlen(ops):
    return sum(n for n, op in ops if op in "M=XIS")


class _Builder:
    def __init__(self, rng, contigs):
        self.rng = rng
        self.contigs = contigs                         # [(name, sequence)]
        self.lines = []                                # (tid or big, pos, serial, text)
        self.shapes = Counter()
        self.spots = defaultdict(set)                  # spot kind -> {(tid, pos)}
        self.gaps = []                                 # per contig: [a, b) that no read touches
        self.cover = [bytearray(len(s)) for _, s in contigs]
        self.serial = 0

    # ---------------------------------------------------------------- reads
    def qname(self):
        self.serial += 1
        return "SRR0742.%d" % (self.serial * 7 + self.rng.randrange(7))

    def free(self, tid, a, b):
        g0, g1 = self.gaps[tid]
        return 0 <= a and b <= len(self.contigs[tid][1]) and (b <= g0 or a >= g1)

    def seq_of(self, tid, pos, ops, sub=0.01, nrate=0.003):
        rng, ref, x, out = self.rng, self.contigs[tid][1], pos, []
        for n, op in ops:
            if op in "M=X":
                for _ in range(n):
                    b = ref[x].upper()
                    if b == "N":
                        b = rng.choice("ACGTN")
                    if op == "X" or (op == "M" and rng.random() < sub):
                        b = rng.choice([c for c in "ACGT" if c != b])
                    elif op == "M" and rng.random() < nrate:
                        b = "N"
                    out.append(b)
                    x += 1
            elif op in "IS":
                out += [rng.choice("ACGT") for _ in range(n)]
            elif op in "DN":
                x += n
        return out

    def qual_of(self, n, q0=0.02):
        rng = self.rng
        return ["!" if rng.random() < q0 else rng.choice(QCH) for _ in range(n)]

    def add(self, qname, flag, tid, pos, mapq, ops, rnext="*", pnext=0, tlen=0, seq=None, qual=None, tags=None):
        """One alignment line; seq/qual are made from the reference when not given ('*' for QUAL '*')."""
        if seq is None:
            seq = self.seq_of(tid, pos, ops) if ops else [self.rng.choice("ACGT") for _ in range(100)]
        if qual is None:
            qual = self.qual_of(len(seq))
        if tags is None:
            tags = ["NM:i:%d" % self.rng.randrange(6), "AS:i:%d" % self.rng.randrange(40, 151)]
        f = [qname, str(flag), self.contigs[tid][0] if tid >= 0 else "*", str(pos + 1 if tid >= 0 else 0), str(mapq), cigar_str(ops),
             rnext, str(pnext), str(tlen), "".join(seq) if seq != "*" else "*", "".join(qual) if qual != "*" else "*"] + list(tags)
        self.lines.append((tid if tid >= 0 else 1 << 30, pos if tid >= 0 else 0, len(self.lines), "\t".join(f)))
        if tid >= 0 and ops:
            e = pos + span(ops)
            self.cover[tid][pos:e] = b"\1" * (e - pos)
        return seq

    def spots_of(self, tid, pos, ops):
        """Reference loci next to the shapes of one alignment."""
        x, sp = pos, self.spots
        sp["read_first"].add((tid, pos))
        sp["read_last"].add((tid, pos + span(ops) - 1))
        for n, op in ops:
            if op == "I":
                sp["before_I"].add((tid, x - 1))
                sp["after_I"].add((tid, x))
            elif op == "D":
                sp["in_D"].update((tid, x + k) for k in range(n))
                sp["next_to_D"].update([(tid, x - 1), (tid, x + n)])
            elif op == "N":
                sp["in_N"].update([(tid, x), (tid, x + n // 2), (tid, x + n - 1)])
            if op in "M=XDN":
                x += n

    def pair(self, tid, f, ops1, ops2, fl, mapq=(60, 60), quals=(None, None), flags=None, qname=None, tags=(None, None)):
        """Two mates of one fragment [f, f + fl): the left one starts at f, the right one ends at f + fl."""
        s1, s2 = span(ops1), span(ops2)
        p1, p2 = f, max(f, f + fl - s2)
        lo, hi = min(p1, p2), max(p1 + s1, p2 + s2)
        if not (self.free(tid, lo, hi)):
            return None
        name = qname or self.qname()
        fl1, fl2 = flags or self.rng.choice([(99, 147), (163, 83)])
        tl = hi - lo
        self.add(name, fl1, tid, p1, mapq[0], ops1, "=", p2 + 1, tl, qual=quals[0], tags=tags[0])
        self.add(name, fl2, tid, p2, mapq[1], ops2, "=", p1 + 1, -tl if tl else 0, qual=quals[1], tags=tags[1])
        return name, p1, p2

    def plain_ops(self, L):
        r = self.rng.random()
        if r < 0.7:
            return [(L, "M")]
        if r < 0.85:
            return [(L, "=")]
        a = self.rng.randrange(5, L - 5)
        return [(a, "="), (1, "X"), (L - a - 1, "=")]

    def background(self, depth):
        for tid, (_, s) in enumerate(self.contigs):
            n = len(s)
            for f in range(0, n, max(1, 300 // depth)):
                f = min(n - 1, f + self.rng.randrange(0, 40))
                L1, L2 = self.rng.randrange(60, 151), self.rng.randrange(60, 151)
                fl = self.rng.randrange(max(L1, L2), 450)
                if f + fl <= n:
                    self.pair(tid, f, self.plain_ops(L1), self.plain_ops(L2), fl)
            # the first and the last base of the contig are covered
            self.pair(tid, 0, [(100, "M")], [(100, "M")], 260)
            self.pair(tid, n - 300, [(100, "M")], [(100, "M")], 300)

    # ---------------------------------------------------------------- families
    def cigar_family(self, count):
        rng = self.rng
        need = FAMILY_SHAPES["cigar"]
        for k in range(count):
            want = need[k % len(need)]
            ops, tags = self.shaped_ops(want)
            tid = rng.randrange(len(self.contigs))
            sp = span(ops)
            f = rng.randrange(0, len(self.contigs[tid][1]) - sp - 200)
            mate = self.plain_ops(rng.randrange(60, 151))
            fl = max(sp, span(mate)) + rng.randrange(0, 120)          # mates overlap: the mate's base is looked at inside D / N
            if rng.random() < 0.5:
                got = self.pair(tid, f, ops, mate, fl)
                pos = f
            else:
                got = self.pair(tid, f, mate, ops, fl)
                pos = None if got is None else got[2]
            if got is None:
                continue
            self.shapes.update(tags)
            self.spots_of(tid, pos, ops)

    def shaped_ops(self, want):
        """A CIGAR that has the shape `want` (and a few random others); returns (ops, shape tags)."""
        rng = self.rng
        blk = lambda: rng.randrange(12, 40)
        lead, trail, mid = [], [], []
        if want in ("lead_S", "I_after_clip", "D_next_to_clip", "N_next_to_clip") or rng.random() < 0.3:
            lead.append((rng.randrange(1, 20), "S"))
        if want == "H_lead" or rng.random() < 0.15:
            lead.insert(0, (rng.randrange(1, 60), "H"))
        if want == "trail_S" or rng.random() < 0.3:
            trail.append((rng.randrange(1, 20), "S"))
        if want == "H_trail" or rng.random() < 0.15:
            trail.append((rng.randrange(1, 60), "H"))
        events = {"I_then_D": [[("I", 0), ("D", 0)]], "D_then_I": [[("D", 0), ("I", 0)]], "D_N_adjacent": [[("D", 0), ("N", 0)] if rng.random() < 0.5 else [("N", 0), ("D", 0)]],
                  "N_short": [[("N", 0)]], "N_long": [[("N", 1)]], "P": [[("P", 0)]],
                  "multi_indel": [[(rng.choice("ID"), 0)] for _ in range(rng.randrange(2, 5))]}.get(want, [])
        for _ in range(rng.randrange(0, 3)):
            events.append([(rng.choice("IDDP"), 0)])
        rng.shuffle(events)
        events = events[:4]
        first = []
        if want == "I_after_clip" or (lead and rng.random() < 0.2):
            first = [(rng.randrange(1, 6), "I")]
        elif want in ("D_next_to_clip", "N_next_to_clip"):
            skip = (rng.randrange(1, 6), "D") if want == "D_next_to_clip" else (rng.randrange(30, 180), "N")
            if rng.random() < 0.5:
                first = [skip]                                           # right after the leading S
            else:
                if not trail or trail[0][1] != "S":
                    trail.insert(0, (rng.randrange(1, 20), "S"))
                trail.insert(0, skip)                                    # right before the trailing S
        mixed = want == "M_mixed" or rng.random() < 0.3
        for ev in [[]] + events:
            for op, longskip in ev:
                n = {"I": rng.randrange(1, 6), "D": rng.randrange(1, 6), "P": rng.randrange(1, 4),
                     "N": rng.randrange(4200, 6000) if longskip else rng.randrange(30, 199)}[op]
                mid.append((n, op))
            L = blk()
            if mixed and L > 8:
                a = rng.randrange(2, L - 4)
                mid += [(a, "M"), (1, "X"), (L - a - 1, "=")] if rng.random() < 0.5 else [(a, "="), (L - a, "M")]
            else:
                mid.append((L, "M"))
        ops = lead + first + mid + trail
        # adjacent ops of one kind merge (htslib would print them as they are; keep the CIGAR canonical anyway)
        out = []
        for n, op in ops:
            if out and out[-1][1] == op:
                out[-1] = (out[-1][0] + n, op)
            else:
                out.append((n, op))
        return out, self.tags_of(out)

    @staticmethod
    def tags_of(ops):
        t = set()
        kinds = [op for _, op in ops]
        if "M" in kinds and ("=" in kinds or "X" in kinds):
            t.add("M_mixed")
        if kinds[0] == "S" or kinds[:2] == ["H", "S"]:
            t.add("lead_S")
        if kinds[-1] == "S" or kinds[-2:] == ["S", "H"]:
            t.add("trail_S")
        if kinds[0] == "H":
            t.add("H_lead")
        if kinds[-1] == "H":
            t.add("H_trail")
        if "P" in kinds:
            t.add("P")
        if 2 <= sum(op in "ID" for op in kinds) <= 4:
            t.add("multi_indel")
        for a, b in zip(kinds, kinds[1:]):
            if (a, b) == ("I", "D"):
                t.add("I_then_D")
            if (a, b) == ("D", "I"):
                t.add("D_then_I")
            if {a, b} == {"D", "N"}:
                t.add("D_N_adjacent")
            if a in "HS" and b == "I":
                t.add("I_after_clip")
            if (a in "HS" and b == "D") or (a == "D" and b in "HS"):
                t.add("D_next_to_clip")
            if (a in "HS" and b == "N") or (a == "N" and b in "HS"):
                t.add("N_next_to_clip")
        for n, op in ops:
            if op == "N":
                t.add("N_long" if n > 4096 else "N_short")
        return t

    def flags_family(self, count):
        rng, nc = self.rng, len(self.contigs)
        for k in range(count):
            kind = FAMILY_SHAPES["flags"][k % len(FAMILY_SHAPES["flags"])]
            tid = rng.randrange(nc)
            n = len(self.contigs[tid][1])
            L = rng.randrange(60, 151)
            f = rng.randrange(0, n - 8000)
            mapq = rng.choice([29, 30, 30, 255, 60])
            if kind in ("single_end_0", "single_end_16", "mapq_29", "mapq_30", "mapq_255", "rnext_star"):
                if not self.free(tid, f, f + L):
                    continue
                mq = {"mapq_29": 29, "mapq_30": 30, "mapq_255": 255}.get(kind, mapq)
                fl = 16 if kind == "single_end_16" else (0 if kind == "single_end_0" else rng.choice([0, 16]))
                ops = rng.choice([[(L, "M")], [(5, "S"), (L - 5, "M")], [(L - 20, "M"), (20, "H")]])
                self.add(self.qname(), fl, tid, f, mq, ops)
                self.shapes.update(["single_end_%d" % fl, "mapq_%d" % mq, "rnext_star"])
                if mq == 30:
                    self.spots["mapq_30"].add((tid, f + rng.randrange(span(ops))))
            elif kind in ("supp_same_contig", "supp_other_contig", "rnext_other"):
                got = self.pair(tid, f, self.plain_ops(L), self.plain_ops(L), L + rng.randrange(20, 200))
                if got is None:
                    continue
                name, p1, p2 = got
                m = rng.randrange(30, L - 10)
                sops = [(m, "M"), (L - m, "H")] if rng.random() < 0.5 else [(L - m, "H"), (m, "M")]
                sflag = 2048 | rng.choice([99, 147, 163, 83, 97])          # 97: paired, not proper: dropped
                smq = rng.choice([30, 60, 29, 255])
                if kind == "supp_same_contig":
                    sp = p1 + rng.randrange(0, L // 2)                   # overlaps the pair
                    if not self.free(tid, sp, sp + m):
                        continue
                    self.add(name, sflag, tid, sp, smq, sops, "=", p2 + 1, 0)
                    self.spots["supplementary"].add((tid, sp + m // 2))
                else:
                    t2 = (tid + 1) % nc
                    sp = rng.randrange(0, len(self.contigs[t2][1]) - m)
                    if not self.free(t2, sp, sp + m):
                        continue
                    self.add(name, sflag, t2, sp, smq, sops, self.contigs[tid][0], p2 + 1, 0)
                    self.spots["supplementary"].add((t2, sp + m // 2))
                    self.shapes["rnext_other"] += 1
                self.shapes["supp_same_contig" if kind == "supp_same_contig" else "supp_other_contig"] += 1
            elif kind in ("secondary", "duplicate", "qc_fail", "not_proper"):
                bit = {"secondary": 256, "duplicate": 1024, "qc_fail": 512, "not_proper": 0}[kind]
                flags = (97, 145) if kind == "not_proper" else (99 | bit, 147 | bit)
                if self.pair(tid, f, self.plain_ops(L), self.plain_ops(L), L + 100, flags=flags) is not None:
                    self.shapes[kind] += 1
            elif kind in ("placed_unmapped", "mate_unmapped"):
                if not self.free(tid, f, f + L):
                    continue
                name = self.qname()
                fl1, fl2 = rng.choice([(73, 133), (89, 165), (137, 69), (153, 101)])
                self.add(name, fl1, tid, f, 60, [(L, "M")], "=", f + 1, 0)
                self.add(name, fl2, tid, f, 0, None, "=", f + 1, 0, seq=[rng.choice("ACGTN") for _ in range(L)])
                self.shapes.update(["placed_unmapped", "mate_unmapped"])
            elif kind == "long_line":
                # lines longer than the staged overhang: wherever they start near a tile's end, the global parser takes them
                L = rng.randrange(4500, 7000)
                for _ in range(40):
                    tid = rng.randrange(nc)
                    f = rng.randrange(0, len(self.contigs[tid][1]) - L)
                    if self.free(tid, f, f + L):
                        break
                else:
                    continue
                mq = rng.choice([29, 30, 30, 255])
                ops = [(L, "M")] if rng.random() < 0.5 else [(L - 30, "M"), (30, "H")]
                self.add(self.qname(), rng.choice([0, 16]), tid, f, mq, ops, qual="*" if rng.random() < 0.3 else None)
                self.shapes.update(["long_line", "mapq_%d" % mq])
                if mq == 30:
                    self.spots["mapq_30"].add((tid, f + rng.randrange(L)))
            elif kind == "unplaced_unmapped":
                self.add(self.qname(), 4, -1, 0, 0, None, seq=[rng.choice("ACGT") for _ in range(L)])
                self.shapes[kind] += 1

    def chain(self, tid, locus, size, qname=None):
        """`size` kept reads of one QNAME, all covering `locus`: a pair, then supplementary alignments."""
        rng = self.rng
        name = qname or self.qname()
        placed = []
        for i in range(size):
            L = rng.randrange(50, 120)
            p = locus - rng.randrange(0, L)
            ops = [(L, "M")] if i % 3 else [(rng.randrange(1, 9), "S"), (L, "M")] if i % 2 else [(L, "M"), (rng.randrange(5, 30), "H")]
            if not self.free(tid, p, p + L):
                return None
            placed.append((p, ops))
        ends = [p + span(o) for p, o in placed]
        (pa, oa), (pb, ob) = placed[0], placed[1]
        tl = max(ends[0], ends[1]) - min(pa, pb)
        self.add(name, 99, tid, pa, 60, oa, "=", pb + 1, tl if pa <= pb else -tl)
        self.add(name, 147, tid, pb, 60, ob, "=", pa + 1, -tl if pa <= pb else tl)
        for p, o in placed[2:]:
            self.add(name, 2048 | rng.choice([99, 147]), tid, p, rng.choice([30, 60, 255]), o, "=", pa + 1, 0)
        lo, hi = max(p for p, _ in placed), min(ends)
        self.spots["chain"].update((tid, x) for x in {locus, lo, hi - 1, locus + 1})
        return name

    def chains_family(self, count):
        rng = self.rng
        for k in range(count):
            size = (3, 5, 8)[k % 3]
            tid = rng.randrange(len(self.contigs))
            locus = rng.randrange(200, len(self.contigs[tid][1]) - 200)
            if self.chain(tid, locus, size) is not None:
                self.shapes["chain_%d" % size] += 1

    def qualstar_family(self, count):
        rng = self.rng
        tags = lambda: ["NM:i:%d" % rng.randrange(10), "MD:Z:%d" % rng.randrange(10, 150), "AS:i:%d" % rng.randrange(40, 151)]
        for k in range(count):
            tid = rng.randrange(len(self.contigs))
            n = len(self.contigs[tid][1])
            L = rng.randrange(60, 151)
            f = rng.randrange(0, n - 400)
            kind = k % 3
            if kind == 0:                                  # simple (M / = / X only), single-end or paired
                ops = self.plain_ops(L)
                if rng.random() < 0.5:
                    if self.free(tid, f, f + L):
                        self.add(self.qname(), rng.choice([0, 16]), tid, f, 60, ops, qual="*", tags=tags())
                        self.shapes["qualstar_simple"] += 1
                        self.spots["qualstar"].add((tid, f + rng.randrange(L)))
                    continue
                got = self.pair(tid, f, ops, self.plain_ops(L), L + rng.randrange(30, 200), quals=("*", None), tags=(tags(), None))
                if got:
                    self.shapes["qualstar_simple"] += 1
                    self.spots["qualstar"].add((tid, f + rng.randrange(L)))
            elif kind == 1:                                # with clips / indels
                ops, _ = self.shaped_ops(rng.choice(["multi_indel", "lead_S", "I_then_D", "N_short"]))
                sp = span(ops)
                got = self.pair(tid, f, ops, self.plain_ops(L), sp + rng.randrange(0, 100), quals=("*", None), tags=(tags(), None))
                if got:
                    self.shapes["qualstar_nonsimple"] += 1
                    self.spots["qualstar"].add((tid, f + rng.randrange(sp)))
                    self.spots_of(tid, f, ops)
            else:
                # overlapping mates that disagree: the QUAL '*' mate (BQ 255) outranks the other one (getBaseWithRPOcheck)
                fl = L + rng.randrange(10, L // 2)
                if not self.free(tid, f, f + fl):
                    continue
                name = self.qname()
                p2 = f + fl - L
                s1 = self.seq_of(tid, f, [(L, "M")], sub=0, nrate=0)
                s2 = self.seq_of(tid, p2, [(L, "M")], sub=0, nrate=0)
                q2 = self.qual_of(L, q0=0)
                for x in rng.sample(range(p2, f + L), min(6, f + L - p2)):
                    b = s2[x - p2]
                    s2[x - p2] = rng.choice([c for c in "ACGT" if c != b])
                    q2[x - p2] = "I"
                    self.spots["qualstar"].add((tid, x))
                star_first = rng.random() < 0.5
                tl = fl
                self.add(name, 99, tid, f, 60, [(L, "M")], "=", p2 + 1, tl, seq=s1, qual="*" if star_first else None, tags=tags())
                self.add(name, 147, tid, p2, 60, [(L, "M")], "=", f + 1, -tl, seq=s2, qual=q2 if star_first else "*", tags=tags())
                self.shapes["qualstar_mate_differs"] += 1

    # ---------------------------------------------------------------- output
    def targets(self, per_kind=10):
        rng = self.rng
        chosen = {}
        for kind in sorted(self.spots):
            pool = sorted(self.spots[kind])
            for t in rng.sample(pool, min(per_kind, len(pool))):
                chosen.setdefault(t, kind)
        for tid, (_, s) in enumerate(self.contigs):
            chosen.setdefault((tid, 0), "contig_first")
            chosen.setdefault((tid, len(s) - 1), "contig_last")
            self.spots["contig_first"].add((tid, 0))
            self.spots["contig_last"].add((tid, len(s) - 1))
            bare = [x for x in range(len(s)) if not self.cover[tid][x]]
            for x in rng.sample(bare, min(3, len(bare))):
                chosen.setdefault((tid, x), "uncovered")
                self.spots["uncovered"].add((tid, x))
        out = sorted(t for t in chosen if 0 <= t[1] < len(self.contigs[t[0]][1]))
        on = Counter()
        for t in out:
            for kind, pool in self.spots.items():
                if t in pool:
                    on[kind] += 1
        return out, on

    def write(self, outdir, shift, sm):
        prefix = os.path.join(outdir, "in")
        with open(prefix + ".fa", "w") as f:
            for name, s in self.contigs:
                f.write(">%s\n" % name + "\n".join(s[i:i + 70] for i in range(0, len(s), 70)) + "\n")
        lines = sorted(self.lines)
        if shift:
            # one duplicate-flagged line at POS 1 (dropped by the filter) moves every later byte by its length
            name, s = self.contigs[0]
            lines.insert(0, (0, 0, -1, "\t".join(["SRR0742.0", "1024", name, "1", "60", "10M", "*", "0", "0", s[:10].upper().replace("N", "A"),
                                                  "I" * 10, "ZZ:Z:" + "x" * shift])))
        with open(prefix + ".sam", "w") as f:
            f.write("@HD\tVN:1.6\tSO:coordinate\n")
            for name, s in self.contigs:
                f.write("@SQ\tSN:%s\tLN:%d\n" % (name, len(s)))
            f.write("@RG\tID:grp1\tSM:%s\n@PG\tID:bwa\tPN:bwa\tVN:0.7.17\n" % sm)
            f.write("".join(l[3] + "\n" for l in lines))
        return prefix


def _reference(rng, n_contigs):
    out = []
    for c in range(n_contigs):
        n = rng.randrange(10_000, 40_001)
        s = [rng.choice("ACGT") for _ in range(n)]
        for _ in range(rng.randrange(2, 5)):                 # soft-masked (lower-case) runs
            a, l = rng.randrange(0, n - 400), rng.randrange(50, 400)
            s[a:a + l] = [b.lower() for b in s[a:a + l]]
        for _ in range(rng.randrange(1, 3)):                 # N runs
            a, l = rng.randrange(300, n - 300), rng.randrange(5, 120)
            s[a:a + l] = ["N"] * l
        out.append(("chrS%d" % (c + 1), "".join(s)))
    return out


SIZES = {"cigar": 240, "flags": 400, "chains": 60, "qualstar": 150}


def generate(outdir, seed, families=FAMILIES, shift=0, depth=12):
    """Writes <outdir>/in.{fa,sam,spike}; returns (prefix, shapes placed, targets per spot kind)."""
    rng = random.Random(seed)
    b = _Builder(rng, _reference(rng, rng.choice([2, 3])))
    for _, s in b.contigs:
        g = rng.randrange(len(s) // 3, 2 * len(s) // 3)
        b.gaps.append((g, g + 300))
    b.background(depth)
    for fam in families:
        getattr(b, fam + "_family")(SIZES[fam])
    targets, on = b.targets()
    prefix = b.write(outdir, shift, "SH%d" % seed)
    with open(prefix + ".spike", "w") as f:
        f.write("#CHROM\tPOS\tALT\tAF\n")
        for tid, pos in targets:
            ref = b.contigs[tid][1][pos].upper()
            alt = rng.choice([".", ".", ".", rng.choice([c for c in "ACGT" if c != ref])])
            af = rng.choice(["1", "%.3g" % rng.uniform(0.05, 0.95), "%.3g" % rng.uniform(0.3, 0.95)])
            f.write("%s\t%d\t%s\t%s\n" % (b.contigs[tid][0], pos + 1, alt, af))
    return prefix, dict(b.shapes), dict(on)


def chain_case(outdir, seed, size, seq_star=False):
    """Plain pairs plus one chain of `size` mutually overlapping reads of one QNAME (and, with seq_star, one kept read whose SEQ is '*')."""
    rng = random.Random(seed)
    b = _Builder(rng, _reference(rng, 1))
    n = len(b.contigs[0][1])
    b.gaps.append((n, n))
    b.background(8)
    b.chain(0, n // 2, size)
    if seq_star:
        b.add(b.qname(), 0, 0, n // 3, 60, [(80, "M")], seq="*", qual="*")
    targets, _ = b.targets()
    prefix = b.write(outdir, 0, "SH%d" % seed)
    with open(prefix + ".spike", "w") as f:
        f.write("#CHROM\tPOS\tALT\tAF\n" + "".join("%s\t%d\t.\t0.5\n" % (b.contigs[t][0], p + 1) for t, p in targets))
    return prefix


def tokeniser_paths(body: bytes):
    """Which route through parse_kernel's two line parsers (sam_parse.cuh) each line of `body` takes: 'conv' (the common-shape
    parser; a line it objects to goes on to the careful parser over the staged tile), 'staged' (the careful parser over the
    staged tile: lines beyond the first PARSERS of a tile) or 'global' (the careful parser over global memory: lines that end
    past the tile's overhang).
    Returns [(line start, path)]."""
    n = len(body)
    starts = [0] + [i + 1 for i in range(n) if body[i] == 10 and i + 1 < n]
    out, per_tile = [], Counter()
    for s in starts:
        t = s // TILE
        li = per_tile[t]
        per_tile[t] += 1
        e = body.find(b"\n", s)
        e = n if e < 0 else e
        T0 = t * TILE
        stage_end = T0 + TILE + OVERHANG if T0 + TILE + OVERHANG <= n else n
        if e > stage_end:
            out.append((s, "global"))
        else:
            out.append((s, "conv" if li < PARSERS else "staged"))
    return out
