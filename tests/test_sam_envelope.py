"""The tokeniser refuses the same lines on each of its routes (sam_parse.cuh).  parse_kernel meets a line through one of:
- 'conv': the common-shape parser, for the first PARSERS lines of a tile; a line it objects to goes on to the careful parser;
- 'staged': the careful parser over the staged tile, for the lines beyond the first PARSERS;
- 'global': the careful parser over global memory, for lines that end past the tile's staged overhang.

A short-read body (~270 lines per 32 KiB tile) gets one line changed in place so that one field lies just outside what htslib
prints back unchanged.  The line keeps its place, so the sortedness check cannot answer first.  That line is placed on each
route: early in a tile, late in a tile, and padded with a ~4 KiB ZZ:Z: tag while it starts in the last line of a tile (once
in the middle of the body, once as the body's last line without its final newline).

CPU: each placement puts the line on the route it names (shape_cases.tokeniser_paths).
GPU (marked `gpu`): every mutation on every route is refused with SSB_E_FORMAT; the unmutated body runs to completion."""
import pytest

import shape_cases as sh
import spike_cases as sc
import stochasticsim_b200 as ssb
from stochasticsim_b200 import spike as sp

TILE_NO = 2                                       # the tile the placed line sits in (the body has ~9)
PAD = b"\tZZ:Z:" + b"A" * 4096                    # longer than the overhang: the line ends past the staged window
SSB_E_FORMAT = -5


def _field(i, new):
    return lambda f: f[:i] + [new(f[i])] + f[i + 1:]


def _tag(t):
    return lambda f: f + [t]


QNAME, FLAG, RNAME, POS, MAPQ, CIGAR, RNEXT, PNEXT, TLEN, SEQ, QUAL = range(11)
MUTATIONS = {
    "flag_leading_zero": _field(FLAG, lambda v: b"0" + v),
    "flag_65536": _field(FLAG, lambda v: b"65536"),
    "pos_leading_zero": _field(POS, lambda v: b"0" + v),
    "pos_2147483648": _field(POS, lambda v: b"2147483648"),
    "mapq_256": _field(MAPQ, lambda v: b"256"),
    "rname_not_in_header": _field(RNAME, lambda v: b"chrQ"),
    "cigar_leading_zero": _field(CIGAR, lambda v: b"0" + v),
    "cigar_unknown_op": _field(CIGAR, lambda v: v[:-1] + b"Q"),
    "cigar_trailing_digits": _field(CIGAR, lambda v: v + b"5"),
    "cigar_query_length_not_seq_length": _field(CIGAR, lambda v: v + b"1S"),
    "rnext_own_contig_spelled_out": lambda f: f[:RNEXT] + [f[RNAME]] + f[RNEXT + 1:],
    "rnext_not_in_header": _field(RNEXT, lambda v: b"chrQ"),
    "tlen_minus_zero": _field(TLEN, lambda v: b"-0"),
    "seq_lower_case": _field(SEQ, lambda v: v[:1].lower() + v[1:]),
    "seq_one_base_short": _field(SEQ, lambda v: v[:-1]),
    "qual_0x20": _field(QUAL, lambda v: b"\x20" + v[1:]),
    "qual_0x7f": _field(QUAL, lambda v: v[:-1] + b"\x7f"),
    "qname_255_bytes": _field(QNAME, lambda v: v + b"q" * (255 - len(v))),
    "qname_0x7f": _field(QNAME, lambda v: v[:-1] + b"\x7f"),
    "aux_unknown_type": _tag(b"XX:q:1"),
    "aux_int_leading_zero": _tag(b"XX:i:01"),
    "aux_array_leading_zero": _tag(b"XX:B:c,01"),
    "aux_hex_odd_length": _tag(b"XX:H:ABC"),
    "aux_char_two_bytes": _tag(b"XX:A:ab"),
    "aux_float_trailing_zero": _tag(b"XX:f:1.50"),     # judged by aux_float_kernel
}
# placement -> (the route tokeniser_paths must report, how it is made)
ROUTES = {"conv": "conv", "staged": "staged", "global": "global", "global_last_no_newline": "global"}


@pytest.fixture(scope="module")
def base(tmp_path_factory):
    """(names, sequences, targets, body) of a 36 bp read body: ~270 lines per tile, so tiles have lines beyond PARSERS."""
    d = str(tmp_path_factory.mktemp("envelope"))
    prefix = sc.generate("plain", d, contigs="chr19:3000", read_len=36, frag_mean=60, frag_sd=6, coverage=30, spikes=10)
    hdr, body, names = sp.split_header(open(prefix + ".sam", "rb").read())
    seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
    targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    return names, seqs, targets, body


def _placed(body, placement, mutation):
    """(body with the mutated line on `placement`, start of that line)."""
    lines = body.split(b"\n")[:-1]
    starts, s = [], 0
    for l in lines:
        starts.append(s)
        s += len(l) + 1
    in_tile = [i for i, s in enumerate(starts) if s // sh.TILE == TILE_NO]
    assert len(in_tile) > 2 * sh.PARSERS
    k = {"conv": in_tile[sh.PARSERS // 2], "staged": in_tile[2 * sh.PARSERS]}.get(placement, in_tile[-1])
    line = lines[k] + (PAD if placement.startswith("global") else b"")
    if mutation is not None:
        line = b"\t".join(MUTATIONS[mutation](line.split(b"\t")))
    if placement == "global_last_no_newline":
        return b"\n".join(lines[:k] + [line]), starts[k]
    return b"\n".join(lines[:k] + [line] + lines[k + 1:]) + b"\n", starts[k]


@pytest.mark.parametrize("placement", sorted(ROUTES))
def test_placements_reach_their_route(placement, base):
    body = base[3]
    for mutation in [None] + sorted(MUTATIONS):
        b, s = _placed(body, placement, mutation)
        assert dict(sh.tokeniser_paths(b))[s] == ROUTES[placement], (placement, mutation)
        if placement == "global_last_no_newline":
            assert not b.endswith(b"\n") and b.rfind(b"\n") == s - 1
        if placement.startswith("global"):
            assert sh.TILE - s % sh.TILE <= 200, (placement, mutation)


@pytest.fixture(scope="module")
def spike(base):
    ctx = ssb.Context(0)
    with sp.Spike(ctx, base[0], base[1]) as s:
        yield s
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("placement", sorted(ROUTES))
def test_unmutated_line_runs_on_every_route(placement, base, spike):
    body, _ = _placed(base[3], placement, None)
    out, _, st = spike.run_host(body, base[2], 434)
    assert st.alignmentCount == out.count(b"\n") > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mutation", sorted(MUTATIONS))
@pytest.mark.parametrize("placement", sorted(ROUTES))
def test_mutated_line_is_refused_on_every_route(placement, mutation, base, spike):
    body, _ = _placed(base[3], placement, mutation)
    with pytest.raises(ssb.SSBError) as e:
        spike.run_host(body, base[2], 434)
    assert e.value.code == SSB_E_FORMAT
