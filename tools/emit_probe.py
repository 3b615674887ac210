"""Emit against the copy ceiling (GPU box): one JSON line on stdout.

    python tools/emit_probe.py [--tree DIR] [--reps N] [--short-mb MB]

Times, with CUDA events and the library's emit profile slot (3), on the card it runs on:
  copy_aligned / copy_phase1   device-to-device copy of the C2 body's byte count, source and destination aligned, and 1 byte out of
                               phase (torch copy_ on offset views): the rate a copy of emit's size can reach
  c2_emit                      the emit group of ssb_spike_run_device on C2 (bench.py's flagship input)
  short_emit                   the emit group on a stand-in for aligner output, where the output order leaves the input order every
                               few lines: the C2 generator with 10 % soft clips, 2 % indels, 3 % ref-skips, 5 % filtered pairs
Rates count bytes read + bytes written (2 x out_bytes for emit).  `--tree` imports stochasticsim_b200 from another checkout, so that
two builds can be compared in one session."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001 -- reported, not guessed
        return {"error": str(e)}


def median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def emit_ms(ctx, S, d_in, n, d_out, tarr, n_targets, reps, sp):
    """(median ms of the emit group per pass, out_bytes) over `reps` passes after two warm-up passes."""
    res = (sp.TargetResult * max(1, n_targets))()
    st = sp.Stats()
    for _ in range(2):
        out = S.run_device(d_in, n, d_out, n + 1, tarr, n_targets, 434, res, st)
    ctx.sync()
    ctx.profile_read(3)
    times = []
    for _ in range(reps):
        out = S.run_device(d_in, n, d_out, n + 1, tarr, n_targets, 434, res, st)
        ctx.sync()
        ms, k = ctx.profile_read(3)
        assert k == 1, k
        times.append(ms)
    return median(times), min(times), max(times), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT, help="checkout whose stochasticsim_b200 build is timed")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--short-mb", type=float, default=4.0, help="contig length of the short-segment shape, in Mb (at 100x)")
    args = ap.parse_args()
    tree = os.path.abspath(args.tree)
    sys.path.insert(0, ROOT)
    sys.path.insert(0, tree)
    import numpy as np
    import torch
    import bench_spike as bs
    import stochasticsim_b200 as ssb
    from stochasticsim_b200 import spike as sp
    assert os.path.dirname(os.path.abspath(ssb.__file__)).startswith(tree), ssb.__file__
    log = lambda *a: print(*a, file=sys.stderr, flush=True)
    out = {"tree": tree, "card": card()}
    L = bs.synth_lib()

    # ---- C2
    ref, parts, n_reads, spike_text = bs.make_workload(L, 2, bs.CHR19, 100.0, 10_000, log=log)
    n = sum(b.size for b in parts)
    src = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    dst = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    off = 0
    for b in parts:
        src[off:off + b.size].copy_(torch.from_numpy(b))
        off += b.size
    del parts
    torch.cuda.synchronize()

    def copy_ms(d, s):
        d.copy_(s)
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            d.copy_(s)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        return median(times), min(times), max(times)

    for key, d, s in (("copy_aligned", dst[:n], src[:n]), ("copy_phase1", dst[1:n + 1], src[:n])):
        m, lo, hi = copy_ms(d, s)
        out[key] = {"bytes": n, "ms": m, "ms_min": lo, "ms_max": hi, "tb_s": 2 * n / m / 1e9}
        log(key, out[key])

    ctx = ssb.Context(0)
    ctx.profile_enable(True)
    targets = sp.parse_spike(spike_text, ["chr19"])
    with sp.Spike(ctx, ["chr19"], {"chr19": ref.tobytes()}) as S:
        tarr = S.make_targets(targets)
        m, lo, hi, ob = emit_ms(ctx, S, src.data_ptr(), n, dst.data_ptr(), tarr, len(targets), args.reps, sp)
    out["c2_emit"] = {"reads": n_reads, "sam_bytes": n, "out_bytes": ob, "ms": m, "ms_min": lo, "ms_max": hi, "tb_s": 2 * ob / m / 1e9}
    log("c2_emit", out["c2_emit"])
    del src, dst
    torch.cuda.empty_cache()

    # ---- short segments
    clen = int(args.short_mb * 1e6)
    p = bs.c2_params(L, 7, 100.0)
    p.softclip_rate, p.indel_rate, p.refskip_rate, p.filt_rate = 0.1, 0.02, 0.03, 0.05
    ref = np.empty(clen + 1, dtype=np.uint8)
    L.synth_ref_contig(C.byref(p), 0, clen, 0, clen, 0, ref.ctypes.data)
    need = L.synth_sam_range(C.byref(p), 0, b"chr19", ref.ctypes.data, clen, 0, clen, 0, clen, None, 0, None)
    body = np.empty(need, dtype=np.uint8)
    nr = C.c_int64()
    L.synth_sam_range(C.byref(p), 0, b"chr19", ref.ctypes.data, clen, 0, clen, 0, clen, body.ctypes.data, need, C.byref(nr))
    ns = max(8, clen * 10_000 // bs.CHR19)
    sn = L.synth_spike_table(C.byref(p), 0, b"chr19", 0, clen, ns, 1, 0.01, 0.5, None, 0)
    sb = C.create_string_buffer(sn + 1)
    L.synth_spike_table(C.byref(p), 0, b"chr19", 0, clen, ns, 1, 0.01, 0.5, sb, sn)
    targets = sp.parse_spike(sb.raw[:sn], ["chr19"])
    src = torch.empty(need + 64, dtype=torch.uint8, device="cuda")
    dst = torch.empty(need + 64, dtype=torch.uint8, device="cuda")
    src[:need].copy_(torch.from_numpy(body))
    torch.cuda.synchronize()
    with sp.Spike(ctx, ["chr19"], {"chr19": ref[:clen].tobytes()}) as S:
        tarr = S.make_targets(targets)
        m, lo, hi, ob = emit_ms(ctx, S, src.data_ptr(), need, dst.data_ptr(), tarr, len(targets), max(args.reps, 15), sp)
    out["short_emit"] = {"contig_bp": clen, "reads": nr.value, "sam_bytes": need, "out_bytes": ob, "ms": m, "ms_min": lo, "ms_max": hi,
                         "tb_s": 2 * ob / m / 1e9}
    log("short_emit", out["short_emit"])
    ctx.close()
    out["copy_phase1_over_c2_emit"] = out["c2_emit"]["ms"] / out["copy_phase1"]["ms"]
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
