#!/usr/bin/env python
"""bench.py -- the judged harness (one JSON line on stdout, see the contract in DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload spike|tnc] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of a hot path over one batch of synthetic input that is already resident in HBM
(`value`), or that starts in pinned host memory and ends with the results back on the host (`e2e`).
Both go through the C ABI of libssb200.so (ctypes, plain pointers): torch is used only to create the
synthetic input on the device, for torch.distributed (barrier, max over ranks) and for nothing else.

Workloads (BASELINE.json configs; SURVEY.md 8d):
  spike  C2: chr19-length reference, 150 bp paired reads, 10k spike loci (--reads scales the depth)
  tnc    C3: whole-FASTA trinucleotide scan of a GRCh38-shaped 24-contig 60-column FASTA (3.14 GB)

`--impl reference` times the reference's own CPU code (oracle/_ref, the UNMODIFIED reference sources
compiled by oracle/Makefile; falls back to the restated oracle when that binary is absent) on a bounded
sample of the same workload.  oracle/ is never on the product path: it is executed only for this arm,
for the `cpu_baseline` object and for the parity check of the sample.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GRCH38 = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717,
          133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285,
          58617616, 64444167, 46709983, 50818468, 156040895, 57227415]
GRCH38_NAMES = ["chr%d" % i for i in range(1, 23)] + ["chrX", "chrY"]
assert sum(GRCH38) == 3088269832


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump(args, D, name, arr, dtype=None, replicated=False):
    """--dump-outputs: writes one output of the timed path as DIR/<name>.npy (float64 unless `dtype` says float32), so that two builds
    can be compared output for output on the same seeded input.  When several ranks run, an output every rank holds alike
    (`replicated`) is written by rank 0 alone; any other goes to DIR/<name>.rank<r>.npy."""
    import numpy as np
    if not args.dump_outputs or (replicated and D.rank != 0):
        return
    os.makedirs(args.dump_outputs, exist_ok=True)
    if D.on and not replicated:
        name = "%s.rank%d" % (name, D.rank)
    np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(arr, dtype=dtype or np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.thread = [], set(), False, None
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # NVML missing: report that rather than inventing numbers
            self.nv = None
            self.err = str(e)

    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
             0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.NAMES.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def __enter__(self):
        if self.nv:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        if self.thread:
            self.thread.join()

    def summary(self):
        if not self.nv or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------ distributed
class Dist:
    def __init__(self, gpus):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.on = self.world > 1
        if self.on:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(self.local)
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.on:
            self.dist.barrier()

    def max(self, x):
        if not self.on:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x):
        if not self.on:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def gather(self, row):
        """list of float64 rows, one per rank, in rank order (on every rank)."""
        if not self.on:
            return [list(map(float, row))]
        import torch
        t = torch.tensor(list(map(float, row)), dtype=torch.float64, device="cuda")
        out = [torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [o.cpu().tolist() for o in out]

    def ssb_comm(self, ctx):
        """The library's own NCCL communicator over the ranks of this job (ssb_nccl_unique_id on rank 0, the 128 bytes broadcast
        through torch.distributed, ssb_nccl_comm_init_rank everywhere): what the product collectives and the spike exchange run on."""
        if getattr(self, "_comm", None) is not None:
            return self._comm
        import torch
        import stochasticsim_b200 as ssb
        from stochasticsim_b200 import spike as sp
        L = sp._bind()
        idt = torch.zeros(128, dtype=torch.uint8)
        if self.rank == 0:
            buf = (C.c_uint8 * 128)()
            ssb.check(L.ssb_nccl_unique_id(buf))
            idt = torch.tensor(list(buf), dtype=torch.uint8)
        idt = idt.cuda()
        self.dist.broadcast(idt, 0)
        raw = bytes(idt.cpu().tolist())
        comm = C.c_void_p()
        ssb.check(L.ssb_nccl_comm_init_rank(ctx.handle, self.world, self.rank, raw, C.byref(comm)), ctx.handle)
        self._comm = comm
        return comm

    def close(self):
        if self.on:
            if getattr(self, "_comm", None) is not None:
                from stochasticsim_b200 import spike as sp
                sp._bind().ssb_nccl_comm_destroy(self._comm)
            self.dist.destroy_process_group()


# ------------------------------------------------------------------------------------- TNC workload
def tnc_make_fasta_device(torch, rank, scale=1.0):
    """GRCh38-shaped FASTA on the device: 24 contigs, 60 columns, 10 kb telomere + 3 Mb centromere N blocks,
    5 % soft-masked lower-case runs (SURVEY.md 8d C3).  Returns (uint8 tensor, n_bases)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(3 + 1000 * rank)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    parts, n_bases = [], 0
    for name, ln in zip(GRCH38_NAMES, GRCH38):
        ln = max(600, int(ln * scale))
        lines = (ln + 59) // 60
        body = lut[torch.randint(0, 4, (lines * 60,), generator=g, device="cuda", dtype=torch.uint8).long()]
        # soft-masked runs: blocks of 256 bases, 5 % of them lower case
        nb = (lines * 60 + 255) // 256
        low = (torch.rand(nb, generator=g, device="cuda") < 0.05).repeat_interleave(256)[: lines * 60]
        body = torch.where(low, body | 0x20, body)
        tel = min(10_000, ln // 10)
        cen0, cen1 = ln // 2, min(ln, ln // 2 + min(3_000_000, ln // 10))
        body[:tel] = ord("N")
        body[ln - tel:ln] = ord("N")
        body[cen0:cen1] = ord("N")
        arr = torch.full((lines, 61), ord("\n"), dtype=torch.uint8, device="cuda")
        arr[:, :60] = body.view(lines, 60)
        flat = arr.view(-1)
        last = ln - (lines - 1) * 60                     # bases on the last line
        flat = torch.cat([flat[: (lines - 1) * 61 + last], flat[-1:]])
        hdr = torch.tensor(list((">%s synthetic\n" % name).encode()), dtype=torch.uint8, device="cuda")
        parts += [hdr, flat]
        n_bases += ln
        del body, arr, low
    return torch.cat(parts), n_bases


def run_tnc(args, D, ctx=None):
    """C3: whole-FASTA trinucleotide scan.  At N > 1 ONE FASTA is cut by byte range (rank g takes [g n / N, (g+1) n / N)), every rank gets
    the scanner state at its cut from ssb_tnc_carry_after, and the 64 counters are combined by ssb_tnc_allreduce INSIDE the timed region
    (the path's only collective).  `value` is whole-job bases/s: the FASTA is the same at every N (strong scaling)."""
    import numpy as np
    import torch
    import stochasticsim_b200 as ssb
    peak, peak_src = measured_peaks()
    torch.cuda.set_device(D.local)
    own_ctx = ctx is None
    if own_ctx:
        ctx = ssb.Context(D.local)
    ctx.profile_enable(True)
    fasta, n_bases = tnc_make_fasta_device(torch, 0, args.scale)       # the same file on every rank
    n_all = fasta.numel()
    torch.cuda.synchronize()
    N = D.world
    lo = (n_all * D.rank // N) & ~31
    hi = n_all if D.rank == N - 1 else (n_all * (D.rank + 1) // N) & ~31
    piece = fasta[lo:hi]
    n = hi - lo
    carry = None
    L = ssb.lib()
    if lo:
        # scanner state at the cut from the bytes before it (host, counts nothing); the last 16 MiB are far more than it ever looks at here
        tail0 = max(0, lo - (16 << 20))
        tail = fasta[tail0:lo].cpu().numpy()
        carry = ssb.tnc.carry_after(tail)
    comm = D.ssb_comm(ctx) if D.on else None
    d_counts = torch.zeros(64, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    log(f"[bench rank {D.rank}] tnc: bytes [{lo}, {hi}) of a {n_all}-byte FASTA ({n_bases} bases) resident in HBM")

    def step():
        ctx.memset(d_counts.data_ptr(), 0, 512)
        ssb.tnc.count_device(ctx, piece.data_ptr(), n, d_counts.data_ptr(), carry_in=carry)
        if comm is not None:
            ssb.check(L.ssb_tnc_allreduce(ctx.handle, comm, d_counts.data_ptr()), ctx.handle)

    for _ in range(args.warmup):
        step()
    ctx.sync()
    ctx.profile_read(0)
    ctx.profile_read(1)
    l0 = ctx.launches()
    D.barrier()
    torch.cuda.synchronize()
    with ClockSampler(D.local) as clk:
        ctx.timer_start()
        for _ in range(args.steps):
            step()
        ms = ctx.timer_stop()
    torch.cuda.synchronize()
    D.barrier()
    launches = ctx.launches() - l0
    scan_ms, scan_n = ctx.profile_read(0)
    fix_ms, fix_n = ctx.profile_read(1)
    ms = D.max(ms)
    counts = d_counts.cpu().numpy().copy()                                 # after the all-reduce: the whole file's counts on every rank
    dump(args, D, "tnc_counts", counts, replicated=True)

    # the sharded counts must equal the one-GPU counts of the whole file (rank 0 checks, outside the timed region)
    if D.on and D.rank == 0:
        d_whole = torch.zeros(64, dtype=torch.int64, device="cuda")
        ssb.tnc.count_device(ctx, fasta.data_ptr(), n_all, d_whole.data_ptr())
        ctx.sync()
        assert np.array_equal(d_whole.cpu().numpy(), counts), "sharded TNC counts differ from the single-GPU counts"

    # ---- e2e: host buffers through ssb_tnc_count_host (H2D inside the timed region, counts back on the host, all-reduce included)
    e2e_steps = args.steps
    hp = ctx.host_alloc(max(n, 1))
    ctx.d2h(hp, piece.data_ptr(), n)
    ctx.sync()
    out = np.zeros(64, dtype=np.int64)

    def e2e_step():
        ssb.check(L.ssb_tnc_count_host(ctx.handle, hp, n, C.byref(carry) if carry is not None else None, None, out.ctypes.data_as(C.POINTER(C.c_int64))), ctx.handle)
        if comm is not None:
            ctx.h2d(d_counts.data_ptr(), out.ctypes.data, 512)
            ssb.check(L.ssb_tnc_allreduce(ctx.handle, comm, d_counts.data_ptr()), ctx.handle)
            ctx.d2h(out.ctypes.data, d_counts.data_ptr(), 512)
            ctx.sync()

    e2e_step()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = D.max(time.perf_counter() - t0)
    assert np.array_equal(out, counts), "device-resident and host-streamed counts differ"
    ctx.host_free(hp)

    scan_gbs = n * args.steps / (scan_ms / 1e3) / 1e9 if scan_ms else None
    res = {
        "metric": "tnc_ref_bases_per_s", "value": n_bases * args.steps / (ms / 1e3), "unit": "bases/s",
        "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong" if D.on else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "C3 tncCountsProfile whole-FASTA scan, ONE GRCh38-shaped 24-contig 60-col FASTA"
                               + (" cut by byte range over %d GPUs" % N if D.on else "") + ("" if args.scale == 1.0 else f" (scaled x{args.scale})"),
                   "fasta_bytes": n_all, "fasta_bytes_per_gpu": n, "bases": n_bases, "l2": "input (%.2f GB per GPU) larger than L2, no flush" % (n / 1e9),
                   "collective": "ssb_tnc_allreduce: one NCCL all-reduce of 64 int64 over NVLink, inside the timed region" if D.on else "none"},
        "e2e": {"value": n_bases * e2e_steps / e2e_s, "unit": "bases/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": 512,
                "steps": e2e_steps, "api": "ssb_tnc_count_host (pinned host FASTA -> 64 host counters)" + (" + ssb_tnc_allreduce" if D.on else "")},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": "tnc_scan_kernel", "achieved": scan_gbs,
                     "peak": peak, "unit": "GB/s", "frac": (scan_gbs / peak) if scan_gbs else None,
                     "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": n * args.steps // max(1, scan_n),
                     "kernel_ms_avg": scan_ms / max(1, scan_n), "kernel_share_of_step": scan_ms / ms if ms else None,
                     "fixup_kernel_ms_avg": fix_ms / max(1, fix_n),
                     "whole_path": {"achieved": n * args.steps / (ms / 1e3) / 1e9, "frac": n * args.steps / (ms / 1e3) / 1e9 / peak}},
        "clocks": clk.summary(),
    }
    del fasta, piece
    torch.cuda.empty_cache()
    if own_ctx:
        ctx.close()
    return res, counts


# --------------------------------------------------------------------------- CPU side (oracle / _ref)
def tnc_sample_fasta(n_bases, seed=3):
    import numpy as np
    rng = np.random.default_rng(seed)
    lines = n_bases // 60
    body = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=lines * 60, dtype=np.uint8)]
    low = np.repeat(rng.random((lines * 60 + 255) // 256) < 0.05, 256)[: lines * 60]
    body = np.where(low, body | 0x20, body).astype(np.uint8)
    body[: 10_000] = ord("N")
    arr = np.full((lines, 61), ord("\n"), dtype=np.uint8)
    arr[:, :60] = body.reshape(lines, 60)
    return b">chr1 synthetic sample\n" + arr.tobytes()


def tnc_cpu_run(path):
    """Runs the reference's tncCountsProfile (unmodified source, -O2 build in oracle/_ref) on a file; returns
    (seconds, stdout, kind)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "tncCountsProfile")
    kind = "reference"
    if not os.path.exists(exe):
        exe = os.path.join(ROOT, "oracle", "_build", "tnc_oracle")
        kind = "port"
        if not os.path.exists(exe):
            subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
    t0 = time.perf_counter()
    out = subprocess.run([exe, path], capture_output=True, check=True).stdout
    return time.perf_counter() - t0, out, kind


def tnc_cpu_baseline(target_s=12.0):
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "probe.fa")
        open(p, "wb").write(tnc_sample_fasta(6_000_000))
        t, _, kind = tnc_cpu_run(p)
        rate = 6_000_000 / t
        nb = int(min(400_000_000, max(6_000_000, rate * target_s))) // 60 * 60
        data = tnc_sample_fasta(nb)
        open(p, "wb").write(data)
        t, out, kind = tnc_cpu_run(p)
    return {"value": nb / t, "unit": "bases/s", "cores": 1, "kind": kind,
            "sample": f"{nb} bases ({len(data)} B, 60-col, 5% lower case, one N block) in {t:.2f} s, "
                      + ("unmodified tncCountsProfile.c -O2" if kind == "reference" else "oracle/tnc_oracle.c -O2"),
            "host_cores_available": os.cpu_count()}, data, out


def run_tnc_reference(args, D):
    """--impl reference for the TNC workload: each step is one run of the CPU binary over a bounded sample."""
    if D.rank != 0:
        return None
    budget = 150.0 / (args.steps + args.warmup)
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "probe.fa")
        open(p, "wb").write(tnc_sample_fasta(3_000_000))
        t, _, kind = tnc_cpu_run(p)
        nb = int(min(400_000_000, max(3_000_000, 3_000_000 / t * budget))) // 60 * 60
        open(p, "wb").write(tnc_sample_fasta(nb))
        for _ in range(args.warmup):
            tnc_cpu_run(p)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            tnc_cpu_run(p)
        s = time.perf_counter() - t0
    v = nb * args.steps / s
    cb = {"value": v, "unit": "bases/s", "cores": 1, "kind": kind, "host_cores_available": os.cpu_count(),
          "sample": f"{nb} bases per step (60-col FASTA), single-threaded as the reference is"}
    return {"impl": "reference", "metric": "tnc_ref_bases_per_s", "value": v, "unit": "bases/s", "n_gpus": D.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": s / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "C3 tncCountsProfile whole-FASTA scan (bounded sample of the same shape)"},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


# ---------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("SSB_BENCH_WORKLOAD", "auto"), choices=["auto", "spike", "tnc", "panel"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (development only; the judged run uses 1.0)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tnc", action="store_true", help="spike workload only (development)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # only the JSON line may reach stdout: libraries (NCCL prints its version there) go to stderr meanwhile
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    D = Dist(args.gpus)
    workload = args.workload
    if workload == "auto":
        try:
            import bench_spike  # noqa: F401  (present once the spike path is benchable)
            workload = "spike"
        except ImportError:
            workload = "tnc"

    if args.impl == "reference":
        if workload == "spike":
            import bench_spike
            res = bench_spike.run_reference(args, D)
        else:
            res = run_tnc_reference(args, D)
        if D.rank == 0:
            emit(res)
        D.close()
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback (use --impl reference for the CPU arm)")
    import numpy as np
    import stochasticsim_b200 as ssb
    if workload == "panel":
        import bench_spike
        res = bench_spike.run_panel(args, D)
        if D.rank == 0:
            emit(res)
        D.close()
        return
    if workload == "spike":
        import bench_spike
        res, ctx = bench_spike.run(args, D)
        # the other hot path rides in the same line (BASELINE's metric names both)
        if not args.no_tnc:
            tnc, counts = run_tnc(args, D, ctx)
            if D.rank == 0 and not args.no_cpu_baseline:
                tnc["cpu_baseline"] = tnc_parity_baseline(ctx)
            res["tnc"] = tnc
        ctx.close()
    else:
        res, counts = run_tnc(args, D)
        if D.rank == 0 and not args.no_cpu_baseline:
            with ssb.Context(D.local) as ctx:
                res["cpu_baseline"] = tnc_parity_baseline(ctx)
    if D.rank == 0:
        emit(res)
    D.close()


def tnc_parity_baseline(ctx):
    """The reference binary on a bounded sample, and the GPU path against its stdout on that sample."""
    import numpy as np
    import stochasticsim_b200 as ssb
    cb, data, ref_out = tnc_cpu_baseline()
    got = ssb.tnc.format_counts(ssb.tnc.count_host(ctx, np.frombuffer(data, dtype=np.uint8)))
    cb["sample_parity"] = "bit-exact" if got.encode() == ref_out else "MISMATCH"
    assert got.encode() == ref_out, "GPU counts differ from the reference binary on the CPU sample"
    return cb


if __name__ == "__main__":
    main()
