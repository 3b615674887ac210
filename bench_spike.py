"""Spike workload of bench.py (BASELINE.json configs[1], SURVEY.md 8d C2): chr19-length reference, 150 bp paired
reads at 100x (39.1 M reads, ~14 GB of SAM text), 10,000 SBS spike loci, seed 434.

At N GPUs the input is ONE coordinate-sorted SAM over N chr19-sized contigs (the shape of C4: one generator seed, one
`.spike` table with N x 10,000 loci, one rand() stream), cut by coordinate range: rank g holds the reads that start on
contig g and runs as shard g of a cooperative group (ssb_spike_run_shard_device over an NCCL exchange).  The shards hand
the exact rand() offset on (8 bytes, rank 0 -> 1 -> ...) after simulating the window of offsets they can be entered with;
the concatenated outputs are what one GPU (or the reference) makes of the whole file (tests/test_spike_shards.py).

The synthetic input comes from tools/gen_synth.c (counter based, so any coordinate range can be generated on its
own: ranks and host threads build their shards independently).  All compute goes through the C ABI
(ssb_spike_run[_shard]_device for `value`, ssb_spike_run[_shard]_host for `e2e`)."""
import ctypes as C
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
CHR19 = 58_617_616
SPIKE_SEED = 434                       # bin/spikeIn.bash:41


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("read_len", C.c_int), ("frag_mean", C.c_double), ("frag_sd", C.c_double),
                ("coverage", C.c_double), ("sub_rate", C.c_double), ("indel_rate", C.c_double), ("n_rate", C.c_double),
                ("q0_rate", C.c_double), ("softclip_rate", C.c_double), ("refskip_rate", C.c_double), ("filt_rate", C.c_double),
                ("fa_width", C.c_int), ("lower_frac", C.c_double), ("aux_tags", C.c_int)]


def synth_lib():
    so = os.path.join(ROOT, "tools", "_build", "libsynth.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-s", "-C", ROOT, "tools"], check=True)
    L = C.CDLL(so)
    L.synth_default_params.argtypes = [C.POINTER(SynthParams)]
    L.synth_ref_contig.argtypes = [C.POINTER(SynthParams), C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_void_p]
    L.synth_sam_range.restype = C.c_int64
    L.synth_sam_range.argtypes = [C.POINTER(SynthParams), C.c_int, C.c_char_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                  C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    L.synth_spike_table.restype = C.c_int64
    L.synth_spike_table.argtypes = [C.POINTER(SynthParams), C.c_int, C.c_char_p, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                    C.c_double, C.c_double, C.c_void_p, C.c_int64]
    return L


def c2_params(L, seed, coverage):
    p = SynthParams()
    L.synth_default_params(C.byref(p))
    p.seed, p.read_len, p.frag_mean, p.frag_sd, p.coverage = seed, 150, 350.0, 35.0, coverage
    p.sub_rate, p.indel_rate = 0.001, 0.0001
    p.aux_tags = int(os.environ.get("SSB_BENCH_AUX", "0"))          # development only: NM:i / RG:Z fields on every line
    return p


def spike_table(L, seed, coverage, contig_len, n_spikes, name=b"chr19", cidx=0):
    p = c2_params(L, seed, coverage)
    sn = L.synth_spike_table(C.byref(p), cidx, name, 0, contig_len, n_spikes, 1, 0.01, 0.5, None, 0)
    sb = C.create_string_buffer(sn + 1)
    L.synth_spike_table(C.byref(p), cidx, name, 0, contig_len, n_spikes, 1, 0.01, 0.5, sb, sn)
    return sb.raw[:sn]


def make_workload(L, seed, contig_len, coverage, n_spikes, name=b"chr19", threads=None, log=None, cidx=0, lo=0, hi=None):
    """Returns (ref bytes ndarray, body chunks list[bytes-like ndarray], n_reads, spike text bytes) of contig `cidx`; only the reads that
    start in [lo, hi) when a range is given (the generator is counter based: any range can be made on its own)."""
    p = c2_params(L, seed, coverage)
    ref = np.empty(contig_len + 1, dtype=np.uint8)
    L.synth_ref_contig(C.byref(p), cidx, contig_len, 0, contig_len, 0, ref.ctypes.data)
    step = 200_000
    hi = contig_len if hi is None else hi
    ranges = [(a, min(hi, a + step)) for a in range(lo, hi, step)]
    per_pos = coverage / 150.0 * 420.0 * 1.25 + 64          # generous bytes per reference position

    def gen(rg):
        lo, hi = rg
        cap = int((hi - lo) * per_pos) + (1 << 16)
        buf = np.empty(cap, dtype=np.uint8)
        nr = C.c_int64()
        need = L.synth_sam_range(C.byref(p), cidx, name, ref.ctypes.data, contig_len, 0, contig_len, lo, hi, buf.ctypes.data, cap, C.byref(nr))
        if need > cap:
            buf = np.empty(need, dtype=np.uint8)
            L.synth_sam_range(C.byref(p), cidx, name, ref.ctypes.data, contig_len, 0, contig_len, lo, hi, buf.ctypes.data, need, C.byref(nr))
        return buf[:need], nr.value

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads or min(32, os.cpu_count() or 8)) as ex:
        parts = list(ex.map(gen, ranges))
    n_reads = sum(nr for _, nr in parts)
    if log:
        log(f"[bench] generated {n_reads} reads, {sum(b.size for b, _ in parts)} SAM bytes in {time.perf_counter() - t0:.1f} s")
    return ref[:contig_len], [b for b, _ in parts], n_reads, spike_table(L, seed, coverage, contig_len, n_spikes, name, cidx)


def header_for(name, contig_len):
    return ("@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:%s\tLN:%d\n@PG\tID:gen_synth\tPN:gen_synth\n" % (name, contig_len)).encode()


# ---- where to cut ONE input of N contigs into N coordinate shards so that every GPU finishes at the same time.  Timeline of a shard
# of length l (in contigs) over the contig range [x0, x1): everything up to the pileup entries (PRE * l), then the output branch (OUT * l:
# emit + tallies, which needs nothing from the other shards), then -- not before EVERY shard has reached the exchange of expected draw
# counts, time A = PRE * the longest shard -- phase 1 of the RNG chain, whose windows widen with the square root of the loci in front of
# the shard (P1_LIN * l + P1_GROW * (x1^1.5 - x0^1.5): the rand() offset there is only known to +-4 sigma while the shards work side by
# side), then the composition, phase 3 and the patches (POST * l).  Constants: ms per C2 contig, measured on B200 (DESIGN.md section 8).
PRE, OUT, P1_LIN, P1_GROW, POST = 22.8, 9.0, 8.2, 4.5, 3.3


def shard_finish(x0, x1, a_all):
    ln = x1 - x0
    return max((PRE + OUT) * ln, a_all) + P1_LIN * ln + P1_GROW * (x1 ** 1.5 - x0 ** 1.5) + POST * ln


def balanced_cuts(n_shards, n_contigs, balance=True):
    """Cut positions x_0 = 0 < x_1 < ... < x_N = n_contigs in contig units."""
    if not balance or n_shards == 1:
        return [n_contigs * g / n_shards for g in range(n_shards + 1)]

    def cuts_for(t, a_all):
        x, cuts = 0.0, [0.0]
        for _g in range(n_shards):
            a, b = x, float(n_contigs) + 1.0
            for _ in range(60):                      # the longest shard from x that is done by t
                m = (a + b) / 2
                if shard_finish(x, m, a_all) <= t:
                    a = m
                else:
                    b = m
            x = a
            cuts.append(x)
        return cuts

    a_all, cuts = 0.0, None
    for _ in range(12):                              # fixed point on the time of the exchange
        lo_t, hi_t = 0.0, 1e5
        for _ in range(60):                          # bisection on the common finishing time
            t = (lo_t + hi_t) / 2
            if cuts_for(t, a_all)[-1] >= n_contigs:
                hi_t = t
            else:
                lo_t = t
        cuts = cuts_for(hi_t, a_all)
        a_all = PRE * max(cuts[i + 1] - cuts[i] for i in range(n_shards))
    cuts[-1] = float(n_contigs)
    return cuts


def traffic_from_profile(scale):
    """dram__bytes_read.sum + dram__bytes_write.sum per step, summed over every kernel of one pass, from the committed ncu capture of
    this exact workload (profiles/r02_spike_traffic.json, written by tools/ncu_traffic.py); None when there is none."""
    p = os.path.join(ROOT, "profiles", "r02_spike_traffic.json")
    if scale != 1.0 or not os.path.exists(p):
        return None, None
    try:
        import json
        j = json.load(open(p))
        return float(j["dram_bytes_per_step"]), j.get("per_kernel")
    except Exception:
        return None, None


DUMP_BLOCK = 1 << 16                   # bytes of spiked SAM per entry of spike_sam_block_sums (on one rank)
DUMP_WINDOWS, DUMP_WINDOW = 64, 1 << 16
# the Stats fields that are results of the pass (the counters of the reference's stats block, the rand() draws); timings and
# scheduling counters (chain chunks, streamed pieces, window retries) may differ between builds that compute the same thing
DUMP_STATS = ("alignmentCount", "numberOfLociCovered", "totalFoldCoverage", "maxDepth", "n_lines", "n_kept", "in_bytes", "out_bytes",
              "n_hits", "rng_draws", "rng_k_in", "rng_k_out")


def dump_spike(args, D, ctx, d_out, out_bytes, res, n_targets, st):
    """--dump-outputs for one spike pass: what a caller of ssb_spike_run[_shard]_device receives.  The spiked SAM body is too large to
    store, so it goes as the byte sum of every block (the whole body) plus windows of 64 KiB at seeded offsets, byte for byte; the
    targets go as one row per target this rank owns (target index first).  On N ranks the blocks are N x 64 KiB long and each rank
    writes 64 / N windows, so the files of all ranks together stay near the size of one rank's at N = 1 (about 19 MB at C2)."""
    if not args.dump_outputs:
        return
    from bench import dump
    from stochasticsim_b200 import spike as sp
    block = DUMP_BLOCK * D.world
    chunk = block * max(1, (1 << 28) // block)
    buf = np.empty(chunk, dtype=np.uint8)
    sums = []
    for c0 in range(0, out_bytes, chunk):
        m = min(chunk, out_bytes - c0)
        ctx.d2h(buf.ctypes.data, d_out + c0, m)
        ctx.sync()
        full = m // block * block
        sums.append(buf[:full].reshape(-1, block).sum(axis=1, dtype=np.uint64))
        if full < m:
            sums.append(buf[full:m].sum(dtype=np.uint64, keepdims=True))
    dump(args, D, "spike_sam_block_sums", np.concatenate(sums) if sums else np.zeros(0))
    w, nw = min(DUMP_WINDOW, out_bytes), max(1, DUMP_WINDOWS // D.world)
    offs = np.sort(np.random.default_rng(434).integers(0, out_bytes - w + 1, size=nw))
    win = np.empty((nw, w), dtype=np.uint8)
    for i, o in enumerate(offs):
        ctx.d2h(win[i].ctypes.data, d_out + int(o), w)
    ctx.sync()
    dump(args, D, "spike_sam_window_offsets", offs)
    dump(args, D, "spike_sam_windows", win, np.float32)
    tr = []
    for i in range(n_targets):
        r = res[i]
        if r.status != sp.T_ELSEWHERE:
            tr.append([i, r.status, r.at_tid, r.at_pos, r.locus_index, r.ref_base, r.mutant_allele, r.filter, r.ref_cnt, r.mut_cnt,
                       *r.err_cnt, r.rng_offset])
    dump(args, D, "spike_targets", np.array(tr, dtype=np.float64).reshape(len(tr), 15))
    dump(args, D, "spike_stats", [getattr(st, k) for k in DUMP_STATS])


def run(args, D):
    import torch
    import stochasticsim_b200 as ssb
    from stochasticsim_b200 import spike as sp
    from bench import ClockSampler, measured_peaks, log
    peak, peak_src = measured_peaks()
    torch.cuda.set_device(D.local)
    L = synth_lib()
    coverage = 100.0 * args.scale
    contig_len = CHR19
    n_spikes = 10_000
    N = D.world
    names = ["chr19"] if N == 1 else ["chr19.%d" % g for g in range(N)]
    # ONE input: N contigs of the same generator seed, cut into N coordinate ranges of equal expected finishing time (SSB_BENCH_BALANCE=0: one contig each).
    # default: one contig per shard.  Cuts for equal finishing time (SSB_BENCH_BALANCE=1: later shards simulate wider windows, so they get fewer reads) were
    # measured at N=4: 57.4 ms against 57.0 -- the shards meet at three exchanges before phase 1 (loci per shard, the target reduction, the expected
    # draws), so a shard with fewer reads only waits longer there (DESIGN.md section 8)
    balance = os.environ.get("SSB_BENCH_BALANCE", "0") != "0"
    cuts = balanced_cuts(N, N, balance)
    HALO = 1024                                               # bases: 150 bp reads with a few indels span < 200
    def to_pos(x):                                            # contig units -> (contig, position)
        c = int(x)
        p = int(round((x - c) * contig_len))
        if p >= contig_len:
            c, p = c + 1, 0
        return c, p

    x0, x1 = cuts[D.rank], cuts[D.rank + 1]
    (c_lo, p_lo), (c_hi, p_hi) = to_pos(x0), to_pos(x1)     # the shard owns (c_lo, p_lo) <= (contig, pos) < (c_hi, p_hi)
    refs, parts, n_reads, halo_bytes = {}, [], 0, 0
    if p_lo > 0:                                              # the lines of the previous shard that can reach into this one
        _, hp_parts, _, _ = make_workload(L, 2, contig_len, coverage, n_spikes, name=names[c_lo].encode(), cidx=c_lo, lo=max(0, p_lo - HALO), hi=p_lo)
        parts += hp_parts
        halo_bytes = sum(b.size for b in hp_parts)
    for c in range(c_lo, min(c_hi, N - 1) + 1):
        a = p_lo if c == c_lo else 0
        b = p_hi if c == c_hi else contig_len
        if b <= a:
            continue
        ref_c, prt, nr, _ = make_workload(L, 2, contig_len, coverage, n_spikes, name=names[c].encode(), log=log, cidx=c, lo=a, hi=b)
        refs[names[c]] = ref_c.tobytes()
        parts += prt
        n_reads += nr
    spike_text = b"".join(spike_table(L, 2, coverage, contig_len, n_spikes, names[g].encode(), g) for g in range(N))
    n = sum(b.size for b in parts)
    ctx = ssb.Context(D.local)
    ctx.profile_enable(True)
    # pinned host copy (e2e input) and the device-resident copy (`value` input)
    hp = ctx.host_alloc(n + 64)
    off = 0
    for b in parts:
        C.memmove(hp + off, b.ctypes.data, b.size)
        off += b.size
    del parts
    hout = ctx.host_alloc(n + 64)
    d_in = ctx.dev_alloc(n + 64)
    d_out = ctx.dev_alloc(n + 64)
    ctx.h2d(d_in, hp, n)
    ctx.sync()
    targets = sp.parse_spike(spike_text, names)
    S = sp.Spike(ctx, names, refs)                            # a shard only ever touches the contigs of its range
    tarr = S.make_targets(targets)
    res = (sp.TargetResult * len(targets))()
    st = sp.Stats()
    shard, xc, comm = None, None, None
    if N > 1:
        hi_tid, hi_pos = (0x7fffffff, 0) if D.rank == N - 1 else (c_hi, p_hi)
        shard = sp.Shard(index=D.rank, count=N, lo_tid=c_lo, hi_tid=hi_tid, lo_pos=p_lo, hi_pos=hi_pos, halo_bytes=halo_bytes)
        comm = D.ssb_comm(ctx)
        x = C.c_void_p()
        ssb.check(sp._bind().ssb_exchange_nccl_create(ctx.handle, comm, D.rank, N, C.byref(x)), ctx.handle)
        xc = x
    log(f"[bench rank {D.rank}] shard [{x0:.4f}, {x1:.4f}) of {N} contigs = ({c_lo}, {p_lo}) .. ({c_hi}, {p_hi}): {n_reads} reads, {n} bytes ({halo_bytes} halo)")

    def step():
        return S.run_shard_device(shard, xc, d_in, n, d_out, n + 1, tarr, len(targets), SPIKE_SEED, res, st)

    for _ in range(args.warmup):
        out_bytes = step()
    ctx.sync()
    for slot in range(2, 7):
        ctx.profile_read(slot)
    l0 = ctx.launches()
    D.barrier()
    torch.cuda.synchronize()
    stage_ms = {}
    with ClockSampler(D.local) as clk:
        ctx.timer_start()
        for _ in range(args.steps):
            out_bytes = step()
            for k, v in st.as_dict().items():
                if k.startswith("ms_"):
                    stage_ms[k] = stage_ms.get(k, 0.0) + v
        ms = ctx.timer_stop()
    torch.cuda.synchronize()
    D.barrier()
    launches = ctx.launches() - l0
    prof = {name: ctx.profile_read(slot) for name, slot in (("parse", 2), ("emit", 3), ("chain", 4), ("other", 5), ("tally", 6))}
    ms = D.max(ms)
    total_reads = D.sum(float(n_reads))
    total_bytes = D.sum(float(n + out_bytes))
    stats = st.as_dict()
    # one stream over all shards: every rank starts where its predecessor stopped
    chain = D.gather([stats["rng_k_in"], stats["rng_k_out"], stats["n_hits"], stats["chain_mode"],
                      stage_ms.get("ms_chain", 0.0) / args.steps, stage_ms.get("ms_phase1", 0.0) / args.steps,
                      stage_ms.get("ms_handoff_wait", 0.0) / args.steps, stage_ms.get("ms_exchange", 0.0) / args.steps,
                      (stage_ms.get("ms_parse", 0.0) + stage_ms.get("ms_sort", 0.0) + stage_ms.get("ms_cover", 0.0) + stage_ms.get("ms_gather", 0.0)) / args.steps,
                      stage_ms.get("ms_patch", 0.0) / args.steps, stage_ms.get("ms_total", 0.0) / args.steps, float(stats["n_window_retries"]), float(n_reads)])
    if D.rank == 0:
        for a, b in zip(chain, chain[1:]):
            assert int(a[1]) == int(b[0]), "rand() offset hand-off broken: %r" % (chain,)
        assert int(chain[0][0]) == 0
    dump_spike(args, D, ctx, d_out, out_bytes, res, len(targets), st)

    # ---- e2e: pinned host SAM body in, spiked SAM body back on the host
    e2e_steps = args.steps
    outn = C.c_size_t()
    Lb = sp._bind()

    def e2e_step():
        if shard is None:       # one GPU: the body is streamed through the device in coordinate pieces, both directions of the host link busy
            ssb.check(Lb.ssb_spike_run_host(S.handle, hp, n, hout, n + 1, tarr, len(targets), SPIKE_SEED, res, C.byref(st), C.byref(outn)), ctx.handle)
        else:
            ssb.check(Lb.ssb_spike_run_shard_host(S.handle, C.byref(shard), xc, hp, n, hout, n + 1, tarr, len(targets), SPIKE_SEED,
                                                  res, C.byref(st), C.byref(outn)), ctx.handle)

    e2e_step()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = D.max(time.perf_counter() - t0)
    assert outn.value == out_bytes
    e2e_pieces = int(st.n_forwarded) if shard is None else 0
    # the streamed output must be the device-resident run's output, byte for byte (checked on a sample of 64 MiB windows)
    if shard is None:
        import torch
        dev = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
        host = np.empty(64 << 20, dtype=np.uint8)
        step()
        for w0 in range(0, int(out_bytes), 1 << 30):
            w = min(64 << 20, int(out_bytes) - w0)
            ctx.d2h(host.ctypes.data, d_out + w0, w)
            ctx.sync()
            got = np.ctypeslib.as_array((C.c_uint8 * w).from_address(hout + w0))
            assert np.array_equal(got, host[:w]), "streamed e2e output differs from the device-resident run at offset %d" % w0
        del dev

    # size-independent properties at full size: every read of the ONE input is written exactly once (by the shard that owns its last
    # base: a shard also parses the few lines of its predecessor that reach into its range, and leaves its own last ones to its successor)
    written = D.sum(float(stats["alignmentCount"]))
    assert int(written) == int(total_reads), (written, total_reads)
    assert out_bytes == stats["out_bytes"]
    if N == 1:
        assert stats["alignmentCount"] == stats["n_kept"]
    emit_ms, emit_n = prof["emit"]
    parse_ms, parse_n = prof["parse"]
    chain_ms, chain_n = prof["chain"]
    traffic, traffic_per_kernel = traffic_from_profile(args.scale)
    whole = total_bytes * args.steps / (ms / 1e3) / 1e9 / N          # per GPU
    res_json = {
        "metric": "sam_reads_spiked_per_s", "value": total_reads * args.steps / (ms / 1e3), "unit": "reads/s",
        "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": ("C2 chr19 full-length synthetic 150bp paired reads at %gx with 10k SBS spike loci" % coverage if N == 1 else
                                "ONE coordinate-sorted SAM over %d chr19-sized contigs (C2 per contig: 150bp paired reads at %gx, 10k SBS spike loci each; one seed, one "
                                ".spike table, one rand() stream), cut by coordinate range, shard g on GPU g" % (N, coverage))
                               + ("" if args.scale == 1.0 else f" (depth scaled x{args.scale})"),
                   "cuts_in_contigs": [round(c, 4) for c in cuts], "cut_rule": ("equal expected finishing time per shard (a shard further down the stream simulates wider windows of rand() offsets in phase 1, so it gets fewer reads)" if balance and N > 1 else "one contig per shard"),
                   "reads_on_rank0": n_reads, "sam_bytes_on_rank0": n, "covered_loci_on_rank0": stats["numberOfLociCovered"], "spike_seed": SPIKE_SEED,
                   "targets": len(targets), "targets_hit_on_rank0": stats["n_hits"], "l2": "input (%.2f GB) larger than L2, no flush" % (n / 1e9),
                   "collective": "none" if N == 1 else
                   "NCCL over NVLink, inside the timed region: all-gather of 5 scalars per shard, max-reduction of one int64 per .spike record (%d), "
                   "all-gather of the expected draw counts, the exact rand() offset as an 8-byte send/recv from shard g to g+1, all-gather of the verdict; "
                   "no alignment text moves" % len(targets)},
        "e2e": {"value": total_reads * e2e_steps / e2e_s, "unit": "reads/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": int(out_bytes),
                "steps": e2e_steps, "api": "ssb_spike_run%s_host (pinned host SAM body -> spiked SAM body on the host)" % ("" if N == 1 else "_shard"),
                "streamed_pieces": e2e_pieces},
        "gpu_launches": launches,
        # the whole pass is the unit the north star's "sustained" bandwidth means; the kernels below explain it
        "roofline": {"bound": "hbm", "kernel": "whole pass (every kernel of one step, per GPU)", "achieved": whole,
                     "peak": peak, "unit": "GB/s", "frac": whole / peak, "traffic": traffic,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": n + out_bytes, "kernel_ms_avg": ms / args.steps,
                     "kernel_share_of_step": 1.0,
                     "emit_kernel": {"achieved": 2.0 * out_bytes * args.steps / (emit_ms / 1e3) / 1e9 if emit_ms else None, "kernel_ms_avg": emit_ms / max(1, emit_n),
                                     "algorithmic_bytes_per_launch": 2 * out_bytes, "frac": 2.0 * out_bytes * args.steps / (emit_ms / 1e3) / 1e9 / peak if emit_ms else None,
                                     "note": "the kernel that moves the most bytes (2 x out_bytes)"},
                     "parse_kernel": {"achieved": n * args.steps / (parse_ms / 1e3) / 1e9 if parse_ms else None, "kernel_ms_avg": parse_ms / max(1, parse_n),
                                      "algorithmic_bytes_per_launch": n, "frac": n * args.steps / (parse_ms / 1e3) / 1e9 / peak if parse_ms else None},
                     "chain_kernels": {"ms_per_step": chain_ms / args.steps, "note": "phase 1 + compose + boundaries + phase 3: issue bound, no credited bytes"},
                     "traffic_per_kernel": traffic_per_kernel},
        "stages_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
        "kernel_groups_ms_per_step": {k: v[0] / args.steps for k, v in prof.items()},
        "chain_chunks": stats["chain_mode"],
        "rng_chain": {"ms_per_step": stage_ms.get("ms_chain", 0.0) / args.steps, "phase1_ms_per_step": stage_ms.get("ms_phase1", 0.0) / args.steps,
                      "draws_after_last_shard": int(chain[-1][1]) if D.rank == 0 else None,
                      "per_shard": [{"k_in": int(c[0]), "k_out": int(c[1]), "hits": int(c[2]), "chunks": int(c[3]), "chain_ms": c[4], "phase1_ms": c[5],
                                     "handoff_wait_ms": c[6], "exchange_ms": c[7], "before_chain_ms": c[8], "after_chain_ms": c[9], "host_total_ms": c[10],
                                     "window_retries_last_step": int(c[11]), "reads": int(c[12])} for c in chain] if D.rank == 0 else None,
                      "note": "one glibc rand() stream consumed at every covered locus (stochasticSpike.c:1197): window maps per shard, exact 8-byte hand-off"},
        "clocks": clk.summary(),
    }
    # ---- CPU baseline + parity of the sample (rank 0)
    if D.rank == 0 and not args.no_cpu_baseline:
        res_json["cpu_baseline"] = cpu_baseline(L, S_ctx=(ctx, sp), target_s=15.0)
    if xc is not None:
        sp.exchange_destroy(xc)
    S.close()
    for p_ in (hp, hout):
        ctx.host_free(p_)
    ctx.dev_free(d_in)
    ctx.dev_free(d_out)
    return res_json, ctx


def cpu_exe():
    exe = os.path.join(ROOT, "oracle", "_ref", "stochasticSpike")
    if os.path.exists(exe):
        return exe, "reference", "unmodified stochasticSpike.c -O2 over oracle/shim (htslib I/O + pileup restated, SAM text in)"
    exe = os.path.join(ROOT, "oracle", "_build", "spike_oracle")
    if not os.path.exists(exe):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
    return exe, "port", "oracle/spike_oracle.c -O2"


def write_sample(L, td, contig_len, coverage, n_spikes, seed=2):
    ref, parts, n_reads, spike_text = make_workload(L, seed, contig_len, coverage, n_spikes, threads=4)
    with open(os.path.join(td, "s.fa"), "wb") as f:
        f.write(b">chr19\n")
        r = ref.tobytes()
        for i in range(0, len(r), 60):
            f.write(r[i:i + 60] + b"\n")
    with open(os.path.join(td, "s.sam"), "wb") as f:
        f.write(header_for("chr19", contig_len))
        for b in parts:
            f.write(b.tobytes())
    open(os.path.join(td, "s.spike"), "wb").write(spike_text)
    return n_reads


def cpu_run(td):
    exe, kind, what = cpu_exe()
    t0 = time.perf_counter()
    r = subprocess.run([exe, "s.sam", "s.fa", "s.spike", str(SPIKE_SEED), "out.sam"], cwd=td, capture_output=True,
                       env=dict(os.environ, SPIKE_ORACLE_CMDNAME="stochasticSpike"))
    if r.returncode != 0:
        raise RuntimeError("CPU reference failed: " + r.stderr.decode()[:500])
    return time.perf_counter() - t0, kind, what


def cpu_baseline(L, S_ctx=None, target_s=15.0):
    """The reference's CPU code on a bounded sample of the same shape (a sub-region of chr19 at 100x)."""
    with tempfile.TemporaryDirectory() as td:
        n_reads = write_sample(L, td, 40_000, 100.0, 8)
        t, kind, what = cpu_run(td)
        rate = n_reads / t
        region = int(min(3_000_000, max(40_000, rate * target_s / (100.0 / 150.0 / 2 * 2))))
        region = int(min(3_000_000, max(40_000, rate * target_s * 1.5)))         # reads ~ region * 100/150
        n_reads = write_sample(L, td, region, 100.0, max(8, region * 10_000 // CHR19))
        t, kind, what = cpu_run(td)
        out = {"value": n_reads / t, "unit": "reads/s", "cores": 1, "kind": kind, "host_cores_available": os.cpu_count(),
               "sample": f"{n_reads} reads over a {region} bp region at 100x (same generator, same spike density) in {t:.2f} s; {what}; single-threaded as the reference is"}
        if S_ctx is not None:
            ctx, sp = S_ctx
            sam = open(os.path.join(td, "s.sam"), "rb").read()
            hdr, body, names = sp.split_header(sam)
            seqs = sp.parse_fasta(open(os.path.join(td, "s.fa"), "rb").read())
            targets = sp.parse_spike(open(os.path.join(td, "s.spike"), "rb").read(), names)
            with sp.Spike(ctx, names, seqs) as S2:
                got, _, _ = S2.run_host(body, targets, SPIKE_SEED)
            same = (hdr + got) == open(os.path.join(td, "out.sam"), "rb").read()
            out["sample_parity"] = "bit-exact SAM" if same else "MISMATCH"
            assert same, "GPU SAM differs from the CPU reference on the sample"
    return out


def run_reference(args, D):
    if D.rank != 0:
        return None
    L = synth_lib()
    budget = 150.0 / max(1, args.steps + args.warmup)
    with tempfile.TemporaryDirectory() as td:
        n_reads = write_sample(L, td, 40_000, 100.0, 8)
        t, kind, what = cpu_run(td)
        region = int(min(3_000_000, max(40_000, n_reads / t * budget * 1.5)))
        n_reads = write_sample(L, td, region, 100.0, max(8, region * 10_000 // CHR19))
        for _ in range(args.warmup):
            cpu_run(td)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_run(td)
        s = time.perf_counter() - t0
    v = n_reads * args.steps / s
    cb = {"value": v, "unit": "reads/s", "cores": 1, "kind": kind, "host_cores_available": os.cpu_count(),
          "sample": f"{n_reads} reads over a {region} bp region at 100x per step; {what}; single-threaded as the reference is"}
    return {"impl": "reference", "metric": "sam_reads_spiked_per_s", "value": v, "unit": "reads/s", "n_gpus": D.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "C2 chr19 synthetic 150bp paired reads at 100x with 10k SBS spike loci (bounded sub-region sample)"},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


# ------------------------------------------------------------------------------------------------------------ C5: deep panel
def make_panel(L, n_intervals, depth, seed=5, log=None):
    """BASELINE configs[4] (SURVEY 8d C5) in the shape one of 8 GPUs gets when n_intervals = 625: 1 kb panel intervals (1.5 kb windows so that
    the core reaches the full depth) on 22 contigs, 150 bp pairs with fragments N(200, 20) -- ~40 % of the pairs overlap --, a target on every
    50th core base with AF U(0.005, 0.05).  Returns (names, {name: ref bytes}, body parts, n_reads, spike text)."""
    p = SynthParams()
    L.synth_default_params(C.byref(p))
    p.seed, p.read_len, p.frag_mean, p.frag_sd, p.coverage = seed, 150, 200.0, 20.0, depth
    p.sub_rate, p.indel_rate = 0.001, 0.0001
    names = ["chr%d" % (i + 1) for i in range(22)]
    per = (n_intervals + 21) // 22
    pitch, win, core0, core = 10_000, 1_500, 250, 1_000
    contig_len = per * pitch + 2_000
    refs, jobs = {}, []
    for c, nm in enumerate(names):
        ref = np.empty(contig_len + 1, dtype=np.uint8)
        L.synth_ref_contig(C.byref(p), c, contig_len, 0, contig_len, 0, ref.ctypes.data)
        refs[nm] = ref
        for i in range(per):
            if c * per + i < n_intervals:
                jobs.append((c, 1_000 + i * pitch))
    jobs.sort()

    def gen(job):
        c, w0 = job
        cap = int(depth / 150.0 * 420.0 * win * 1.3) + (1 << 16)
        buf = np.empty(cap, dtype=np.uint8)
        nr = C.c_int64()
        need = L.synth_sam_range(C.byref(p), c, names[c].encode(), refs[names[c]].ctypes.data, contig_len, w0, w0 + win, w0, w0 + win, buf.ctypes.data, cap, C.byref(nr))
        if need > cap:
            buf = np.empty(need, dtype=np.uint8)
            L.synth_sam_range(C.byref(p), c, names[c].encode(), refs[names[c]].ctypes.data, contig_len, w0, w0 + win, w0, w0 + win, buf.ctypes.data, need, C.byref(nr))
        return buf[:need], nr.value

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 8)) as ex:
        parts = list(ex.map(gen, jobs))
    rng = np.random.default_rng(seed)
    lines = []
    for c, w0 in jobs:
        for x in range(w0 + core0, w0 + core0 + core, 50):
            lines.append("%s\t%d\t.\t%.4g\n" % (names[c], x + 1, rng.uniform(0.005, 0.05)))
    n_reads = sum(nr for _, nr in parts)
    if log:
        log(f"[bench] panel: {len(jobs)} intervals, {n_reads} reads, {sum(b.size for b, _ in parts)} SAM bytes, {len(lines)} targets in {time.perf_counter() - t0:.1f} s")
    return names, {k: v[:contig_len].tobytes() for k, v in refs.items()}, [b for b, _ in parts], n_reads, "".join(lines).encode()


def run_panel(args, D):
    """--workload panel: the deep-panel shape (C5).  One GPU's share of the 8-GPU split by default (625 of the 5,000 intervals); --scale 8 = all of C5."""
    import torch
    import stochasticsim_b200 as ssb
    from stochasticsim_b200 import spike as sp
    from bench import ClockSampler, measured_peaks, log
    peak, peak_src = measured_peaks()
    torch.cuda.set_device(D.local)
    L = synth_lib()
    n_intervals = max(1, int(round(625 * args.scale)))
    names, refs, parts, n_reads, spike_text = make_panel(L, n_intervals, 2000.0, log=log)
    n = sum(b.size for b in parts)
    ctx = ssb.Context(D.local)
    ctx.profile_enable(True)
    hp = ctx.host_alloc(n + 64)
    off = 0
    for b in parts:
        C.memmove(hp + off, b.ctypes.data, b.size)
        off += b.size
    del parts
    d_in, d_out = ctx.dev_alloc(n + 64), ctx.dev_alloc(n + 64)
    ctx.h2d(d_in, hp, n)
    ctx.sync()
    targets = sp.parse_spike(spike_text, names)
    S = sp.Spike(ctx, names, refs)
    tarr = S.make_targets(targets)
    res = (sp.TargetResult * len(targets))()
    st = sp.Stats()
    steps, warm = args.steps, 1
    for _ in range(warm):
        out_bytes = S.run_device(d_in, n, d_out, n + 1, tarr, len(targets), SPIKE_SEED, res, st)
    ctx.sync()
    stage_ms = {}
    with ClockSampler(D.local) as clk:
        ctx.timer_start()
        for _ in range(steps):
            out_bytes = S.run_device(d_in, n, d_out, n + 1, tarr, len(targets), SPIKE_SEED, res, st)
            for k, v in st.as_dict().items():
                if k.startswith("ms_"):
                    stage_ms[k] = stage_ms.get(k, 0.0) + v
        ms = ctx.timer_stop()
    stats = st.as_dict()
    dump_spike(args, D, ctx, d_out, out_bytes, res, len(targets), st)
    entries = sum(r.ref_cnt + r.mut_cnt + sum(r.err_cnt) for r in res if r.status == sp.T_HIT)
    ms_step = ms / steps
    out = {
        "metric": "sam_reads_spiked_per_s", "value": n_reads * steps / (ms / 1e3), "unit": "reads/s", "n_gpus": 1, "steps": steps, "warmup": warm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "C5 deep panel: %d of 5,000 1 kb intervals at 2000x (150 bp pairs, fragments N(200,20)), a target on every 50th base, AF 0.5-5 %%"
                               % n_intervals + (" = one GPU's share of the 8-GPU split" if n_intervals == 625 else ""),
                   "reads": n_reads, "sam_bytes": n, "targets": len(targets), "targets_hit": stats["n_hits"], "max_depth": stats["maxDepth"],
                   "pileup_entries_tallied": int(entries), "spike_seed": SPIKE_SEED, "l2": "input (%.2f GB) larger than L2, no flush" % (n / 1e9)},
        "roofline": {"bound": "hbm", "kernel": "whole pass", "achieved": (n + out_bytes) / (ms_step / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": (n + out_bytes) / (ms_step / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                     "note": "bound by the serial RNG chain over the pileups of the targets (one warp, entries staged in shared memory), not by HBM"},
        "stages_ms_per_step": {k: v / steps for k, v in stage_ms.items()},
        "rng_chain": {"ms_per_step": stage_ms.get("ms_chain", 0.0) / steps, "chunks": stats["chain_mode"], "draws": stats["rng_draws"],
                      "ns_per_pileup_entry": stage_ms.get("ms_chain", 0.0) / steps * 1e6 / max(1, entries)},
        "clocks": clk.summary(),
    }
    S.close()
    ctx.host_free(hp)
    ctx.dev_free(d_in)
    ctx.dev_free(d_out)
    ctx.close()
    return out
