"""Times ssb_tnc_count_intervals_device (per-interval trinucleotide counts) on the GRCh38-shaped FASTA of bench.py's C3 workload
(3.1 GB, device-resident), for three BED shapes:

  exome   about 200 k seeded intervals of 100-300 bp over sequence without N (one item per interval, plain-add flush)
  tile1k  a 1 kb tiling of every contig: about 3.1 M rows, 1.6 GB of rows (one item per interval)
  tile1m  a 1 Mb tiling of every contig: about 3.1 k rows, each split into about 490 items over many warps (atomic flush)

For each shape: the call's time (CUDA events around the call, which includes copying the intervals to the device) and the kernel's
time (profiling slot SSB_PROF_TNC_INTERVALS), both as interval bases/s, after one warm-up call; and a spot check of sampled rows against
the numpy closed form of tests/interval_cases.py.  For the exome shape it also times ssb_tnc_count_bed_device on the same intervals.
The FASTA is far larger than L2, so the tilings read it from HBM; the exome shape touches about 40 MB of it.  Prints one JSON line
with the card's name and power limit.  Needs a GPU: without one it fails.

    python tools/tnc_intervals_probe.py [--reps 5] [--samples 300] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
import interval_cases as ic  # noqa: E402
import stochasticsim_b200 as ssb  # noqa: E402
from stochasticsim_b200 import tnc  # noqa: E402
from tnc_shape_probe import card  # noqa: E402

PROF_INTERVALS, PROF_SCAN, PROF_FIXUP = 7, 0, 1


def exome(host, idx, n, seed=11):
    """n intervals of 100-300 bp that hold no N, placed at random (contigs weighted by length), in BED order."""
    g = np.random.default_rng(seed)
    lens = np.array([c.len for _, c in idx], dtype=np.int64)
    geo = np.array([(c.seq_off, c.line_bases, c.line_bytes) for _, c in idx], dtype=np.int64)
    out = np.zeros((0, 3), dtype=np.int64)
    while len(out) < n:
        ci = g.choice(len(idx), size=n, p=lens / lens.sum())
        ln = g.integers(100, 301, size=n)
        a = (g.random(n) * (lens[ci] - ln)).astype(np.int64)
        p = a[:, None] + np.minimum(np.arange(300)[None, :], ln[:, None] - 1)     # the bases of each candidate (the last one repeated)
        off, lb, lbytes = geo[ci, 0:1], geo[ci, 1:2], geo[ci, 2:3]
        has_n = (host[off + p + (p // lb) * (lbytes - lb)] == ord("N")).any(axis=1)
        out = np.concatenate([out, np.stack([ci, a, a + ln], axis=1)[~has_n]])
    out = out[:n]
    return out[np.lexsort((out[:, 1], out[:, 0]))]


def tiling(idx, size):
    parts = []
    for ci, (_, c) in enumerate(idx):
        a = np.arange(0, c.len, size, dtype=np.int64)
        parts.append(np.stack([np.full_like(a, ci), a, np.minimum(a + size, c.len)], axis=1))
    return np.concatenate(parts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--samples", type=int, default=300)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    L = ssb.lib()
    L.ssb_tnc_count_intervals_device.restype = C.c_int
    L.ssb_tnc_count_intervals_device.argtypes = tnc._IV_ARGS
    L.ssb_tnc_count_bed_device.restype = C.c_int
    L.ssb_tnc_count_bed_device.argtypes = tnc._IV_ARGS
    res = {"probe": "tnc_intervals"}
    with ssb.Context(0) as ctx:                        # raises without an sm_100 device
        res["card"], res["power_limit"] = card(ctx)
        fasta, n_bases = bench.tnc_make_fasta_device(torch, 0)
        n = fasta.numel()
        host = fasta.cpu().numpy()
        idx = tnc.fasta_index(host)
        res["fasta"] = {"bytes": n, "bases": n_bases, "contigs": len(idx)}
        ctx.profile_enable(True)
        g = np.random.default_rng(5)
        for name, iv in (("exome", exome(host, idx, 200_000)), ("tile1k", tiling(idx, 1000)), ("tile1m", tiling(idx, 1_000_000))):
            carr, civ = tnc._index_and_intervals(idx, iv)
            rows = torch.zeros((len(iv), 64), dtype=torch.int64, device="cuda")
            iv_bases = int((iv[:, 2] - iv[:, 1]).sum())

            def call():
                ssb.check(L.ssb_tnc_count_intervals_device(ctx.handle, fasta.data_ptr(), n, carr, len(idx), civ, len(iv), 0, len(iv), rows.data_ptr()), ctx.handle)

            rows.zero_()
            call()                                      # warm-up; its rows are the ones checked
            ctx.sync()
            pick = g.choice(len(iv), size=min(a.samples, len(iv)), replace=False)
            got = rows.cpu().numpy()
            ok = all(np.array_equal(got[i], ic.interval_row(host, idx[iv[i, 0]][1], iv[i, 1], iv[i, 2])) for i in pick)
            ctx.profile_read(PROF_INTERVALS)
            call_ms = []
            for _ in range(a.reps):
                rows.zero_()
                ctx.sync()
                ctx.timer_start()
                call()
                call_ms.append(ctx.timer_stop())
            k_ms, k_n = ctx.profile_read(PROF_INTERVALS)
            k_avg = k_ms / max(1, k_n)
            med = float(np.median(call_ms))
            r = {"rows": len(iv), "interval_bases": iv_bases, "call_ms": [round(x, 3) for x in call_ms], "call_ms_median": round(med, 3),
                 "call_bases_per_s": iv_bases / (med / 1e3), "kernel_ms_avg": round(k_avg, 4), "kernel_bases_per_s": iv_bases / (k_avg / 1e3),
                 "kernel_text_gb_per_s": None, "rows_gb": len(iv) * 512 / 1e9, "sampled_rows_match_closed_form": bool(ok), "sampled": len(pick)}
            if name != "exome":                         # a tiling reads the whole text once (plus the 2-base halos)
                r["kernel_text_gb_per_s"] = n / (k_avg / 1e3) / 1e9 if k_avg else None
            else:
                total = torch.zeros(64, dtype=torch.int64, device="cuda")

                def bed():
                    ssb.check(L.ssb_tnc_count_bed_device(ctx.handle, fasta.data_ptr(), n, carr, len(idx), civ, len(iv), 0, len(iv), total.data_ptr()), ctx.handle)

                bed()
                ctx.sync()
                ctx.profile_read(PROF_SCAN)
                ctx.profile_read(PROF_FIXUP)
                bed_ms = []
                for _ in range(a.reps):
                    total.zero_()
                    ctx.sync()
                    ctx.timer_start()
                    bed()
                    bed_ms.append(ctx.timer_stop())
                s_ms, s_n = ctx.profile_read(PROF_SCAN)
                bmed = float(np.median(bed_ms))
                r["bed_mode"] = {"call_ms": [round(x, 3) for x in bed_ms], "call_ms_median": round(bmed, 3), "call_bases_per_s": iv_bases / (bmed / 1e3),
                                 "scan_kernel_ms_per_call": round(s_ms / a.reps, 4), "scan_launches_per_call": s_n / a.reps}
                del total
            res[name] = r
            del rows
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
