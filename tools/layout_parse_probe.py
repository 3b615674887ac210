"""Tokeniser time (stats.ms_parse) on a many-contig header against one contig, same lines.

name_lookup (sam_parse.cuh) rescans every earlier @SQ name for each line's RNAME hint and scans them all for a spelled-out RNEXT,
so its cost per line may grow with the tid.  This builds the `scaffolds` layout of tests/layout_cases.py (12,000 @SQ lines) and a
twin body in which every scaffold is laid end to end on one contig (RNAME, POS and PNEXT rewritten, everything else the same
bytes), runs both through ssb_spike_run_host alternately and prints one JSON line with the median ms_parse of each.

    python tools/layout_parse_probe.py [--reps 9]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def one_contig(body, names, seqs, targets, one="scaffold_00000"):
    """The same lines on one contig made of all contigs end to end, and the targets moved with them."""
    off, at = {}, 0
    for n in names:
        off[n] = at
        at += len(seqs[n])
    out = []
    for line in body.split(b"\n"):
        if not line:
            continue
        f = line.split(b"\t")
        name = f[2].decode()
        if name != "*":
            f[2], f[3] = one.encode(), b"%d" % (int(f[3]) + off[name])
            if f[6] == b"=" and int(f[7]) > 0:
                f[7] = b"%d" % (int(f[7]) + off[name])
        out.append(b"\t".join(f) + b"\n")
    moved = [(one, 0, locus + off[c], base, af) for c, t, locus, base, af in targets if t >= 0]
    return b"".join(out), [one], {one: b"".join(seqs[n] for n in names)}, moved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    import layout_cases as lc
    import stochasticsim_b200 as ssb
    from stochasticsim_b200 import spike as sp

    with tempfile.TemporaryDirectory() as d:
        prefix, _ = lc.generate(d, "scaffolds", 1)
        _, body, names, = sp.split_header(open(prefix + ".sam", "rb").read())
        seqs = sp.parse_fasta(open(prefix + ".fa", "rb").read())
        targets = sp.parse_spike(open(prefix + ".spike", "rb").read(), names)
    inputs = {"scaffolds": (body, names, seqs, targets), "one_contig": one_contig(body, names, seqs, targets)}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    ms = {k: [] for k in inputs}
    with ssb.Context(0) as ctx:
        spikes = {k: sp.Spike(ctx, v[1], v[2]) for k, v in inputs.items()}
        outs = {}
        for rep in range(args.reps + 2):                       # two warm-up passes, then alternate the two inputs
            for k, (b, _, _, t) in inputs.items():
                out, _, st = spikes[k].run_host(b, t, 434)
                outs[k] = (len(out), st.n_lines, st.n_kept)
                if rep >= 2:
                    ms[k].append(st.ms_parse)
        for s in spikes.values():
            s.close()
    res = {"gpu": gpu, "reps": args.reps}
    for k, (b, n, _, _) in inputs.items():
        res[k] = {"contigs": len(n), "body_bytes": len(b), "lines": outs[k][1], "kept": outs[k][2],
                  "ms_parse_median": round(statistics.median(ms[k]), 4), "ms_parse_min": round(min(ms[k]), 4), "ms_parse_max": round(max(ms[k]), 4)}
    res["ratio"] = round(res["scaffolds"]["ms_parse_median"] / res["one_contig"]["ms_parse_median"], 3)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
