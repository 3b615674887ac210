"""Seeded FASTA inputs shared by the oracle tests (CPU) and the parity tests (GPU)."""
import random

import numpy as np

# SURVEY.md App. B known answers: produced by running the reference's own compiled binary.
KAT = [
    (b">c1\nACGT\nGGCC\n", {"ACG": 2, "CCA": 1, "GCC": 2}),
    (b">c1\nACGTGGCC\n", {"ACG": 2, "CCA": 1, "GCC": 2, "GTG": 1}),
    (b">c1\nAC\nNNNN\nGT\n", {"ACG": 1}),
    (b">c1\nACG\n>c2\nTTA\n", {"ACG": 1, "GTT": 1, "TTA": 1}),
    (b">c1\nACg\nacgt\nTTA\n", {"TTA": 1}),
    (b">c1\nACGT", {"ACG": 2}),
    (b">c1\nACGT\r\nGGCC\r\n", {"ACG": 2, "GCC": 2}),
    (b"A\nC\nG\nT\n", {}),
    (b">c1\nACNGT\nANA\n", {}),
]

EDGE = [
    b"", b"\n", b"\n\n\n", b">", b">\n", b"A", b"AC", b"ACG", b"ACG\n", b"\nACG", b">ACGT\nACGT\n",
    b"ACGT\n>ACGTA\nCGTA\n", b"ACGT\n>hdrA\nCG\n", b"ACGN\nACGT\n", b"NNNN\nACGT\n", b"ACGT\n\n\nACGT\n",
    b"ACGT\nN\nACGT\n", b"A\nCG\n", b"AC\nG\nT\nAC\n", b">x\n>y\n>z\nAC\nGT\n", b"ACGT\n>A", b"ACGT\n>AAAA\nCC",
    b"acgt\nAC\n", b"ACGT\nacgt\nACGT\n", b"ACGT\nNNNN\nnnnn\n>h\nNN\nGGT\n", b"T\n>ACGT\nGG\n",
]


def random_fasta(rng: random.Random, max_lines=14) -> bytes:
    alph = rng.choice(["ACGT", "ACGTN", "ACGTacgtN", "ACGTN\r>", "AC", "ACGT" * 5 + "N"])
    parts = []
    for _ in range(rng.randint(0, max_lines)):
        r = rng.random()
        if r < 0.15:
            parts.append(">" + "".join(rng.choice("chrACGT 12") for _ in range(rng.randint(0, 8))))
        elif r < 0.25:
            parts.append("")
        elif r < 0.35:
            parts.append(rng.choice("Nn") * rng.randint(1, 5))
        else:
            parts.append("".join(rng.choice(alph) for _ in range(rng.randint(1, rng.choice([1, 2, 3, 5, 10, 33, 70])))))
    s = "\n".join(parts)
    if parts and rng.random() < 0.8:
        s += "\n"
    return s.encode()


def genome_like(rng: random.Random, n_bases: int, width=60, n_block=None, lower_runs=0, contigs=1) -> bytes:
    """Fixed-width FASTA with optional N block, soft-masked runs and several contigs."""
    out = []
    per = n_bases // contigs
    for c in range(contigs):
        seq = bytearray(rng.choices(b"ACGT", k=per))
        if n_block:
            a, b = n_block
            seq[a:b] = b"N" * (min(b, per) - a)
        for _ in range(lower_runs):
            a = rng.randrange(0, max(1, per - 300))
            seq[a:a + 300] = bytes(seq[a:a + 300]).lower()
        out.append(b">chr%d some description\n" % (c + 1))
        for i in range(0, per, width):
            out.append(bytes(seq[i:i + width]) + b"\n")
    return b"".join(out)


def shard_counts_with_carry(data: bytes, lo: int, hi: int):
    """Counts of data[lo:hi] given everything before lo, via the oracle: counts(data[:hi]) - counts(data[:lo]) is NOT
    what a rank can compute, so emulate the device contract instead: prepend the minimal context the carried state
    stands for and subtract its own windows."""
    import oracle_bind as ob
    import stochasticsim_b200 as ssb
    st = ssb.tnc.carry_after(np.frombuffer(data, dtype=np.uint8)[:lo]) if lo else None
    piece = data[lo:hi]
    if st is None:
        return ob.tnc_counts(piece)
    # context equivalent to the state: the carried last byte of the nearest kept line, then the fragment of the current line
    started, prev, carry, frag_nonempty, frag_first, frag_has_base = st.as_tuple()
    ctx = b""
    if carry:
        ctx += b"A" + bytes([carry]) + b"\n"          # a kept line ending in `carry` ("A" makes it kept, adds no window by itself)
    j = data.rfind(b"\n", 0, lo) + 1                     # the current line's fragment before the cut, verbatim
    frag = data[j:lo]
    base = ob.tnc_counts(ctx + frag) if (ctx or frag) else np.zeros(64, dtype=np.int64)
    return ob.tnc_counts(ctx + frag + piece) - base
