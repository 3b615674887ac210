"""Times one count_device call on a 1 GiB 60-column FASTA and on the same bases written as unwrapped contigs (one line each).

The state-out task and resolve_carry in csrc/tnc.cu walk back one 32-byte step per iteration in a single warp, so for a contig
written as one line they take one step per 32 bytes of the line.  This measures what that costs at genome scale.  Prints one
JSON line with the card's name and power limit.  Needs a GPU: without one it fails.

    python tools/tnc_shape_probe.py [--gib 1] [--contigs 8] [--reps 3] [--check]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import stochasticsim_b200 as ssb  # noqa: E402


def layouts(total, contigs, seed=1):
    """(60-column text, unwrapped text) of the same `contigs` contigs, about `total` bytes each."""
    rng = np.random.default_rng(seed)
    per = total // contigs - 64
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    wrapped, unwrapped = [], []
    for k in range(contigs):
        n = per * 60 // 61
        seq = lut[rng.integers(0, 4, n, dtype=np.uint8)]
        hdr = b">chr%d\n" % (k + 1)
        rows = -(-n // 60)
        arr = np.full((rows, 61), ord("\n"), dtype=np.uint8)
        flat = np.zeros(rows * 60, dtype=np.uint8)
        flat[:n] = seq
        arr[:, :60] = flat.reshape(rows, 60)
        wrapped += [hdr, arr.reshape(-1)[:n + (n - 1) // 60].tobytes(), b"\n"]
        unwrapped += [hdr, seq.tobytes(), b"\n"]
    return b"".join(wrapped), b"".join(unwrapped)


def card(ctx):
    name = ctx.info()["name"]
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(0), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return name, q.stdout.strip()
    except OSError:
        return name, "power limit not readable"


def time_call(ctx, data, reps):
    n = len(data)
    d = ctx.dev_alloc(n + 64)
    dc = ctx.dev_alloc(64 * 8)
    host = np.frombuffer(data, dtype=np.uint8)
    ctx.h2d(d, host.ctypes.data, n)
    ctx.sync()
    times, counts = [], np.zeros(64, dtype=np.int64)
    for it in range(reps + 1):                          # the first call warms up
        ctx.memset(dc, 0, 64 * 8)
        ctx.sync()
        t0 = time.perf_counter()
        ssb.tnc.count_device(ctx, d, n, dc)            # returns after a stream synchronise
        dt = time.perf_counter() - t0
        if it:
            times.append(dt * 1e3)
    ctx.d2h(counts.ctypes.data, dc, 64 * 8)
    ctx.sync()
    ctx.dev_free(d)
    ctx.dev_free(dc)
    return times, counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--contigs", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", action="store_true", help="also compare both counts with the CPU oracle")
    a = ap.parse_args()
    wrapped, unwrapped = layouts(int(a.gib * (1 << 30)), a.contigs)
    res = {}
    with ssb.Context(0) as ctx:                        # raises without an sm_100 device
        res["card"], res["power_limit"] = card(ctx)
        for name, data in (("60-column", wrapped), ("unwrapped", unwrapped)):
            times, counts = time_call(ctx, data, a.reps)
            r = {"bytes": len(data), "ms": [round(t, 3) for t in times], "median_ms": round(float(np.median(times)), 3)}
            if a.check:
                import oracle_bind as ob
                r["matches_oracle"] = bool(np.array_equal(counts, ob.tnc_counts(data)))
            res[name] = r
    res["contigs"] = a.contigs
    print(json.dumps(res))


if __name__ == "__main__":
    main()
