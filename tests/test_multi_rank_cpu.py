"""CPU, world_size 2 over gloo: the N>1 plumbing of the TNC path -- cut the FASTA by byte range, give every rank the
scanner state at its cut (ssb_tnc_carry_after, host only), count the shards independently, all-reduce the 64
counters.  On this GPU-less box the per-shard counting is done by the CHECKER (oracle) seeded with the same state
semantics, which is exactly what makes the test meaningful: the sum over ranks must equal the whole-file counts."""
import os
import random
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))


def _worker(rank, world, port, data, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n = len(data)
    lo, hi = (n * rank // world) & ~31, n if rank == world - 1 else (n * (rank + 1) // world) & ~31
    import fasta_cases as fc
    c = torch.from_numpy(fc.shard_counts_with_carry(data, lo, hi).astype(np.int64))
    dist.all_reduce(c)                                   # the path's only collective: 64 int64 counters
    if rank == 0:
        out_q.put(c.numpy().tolist())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_two_ranks_sum_to_whole_file(seed):
    import fasta_cases as fc
    import oracle_bind as ob
    rng = random.Random(seed)
    data = fc.genome_like(rng, 40_000, width=rng.choice([60, 61, 70]), n_block=(5_000, 9_000), lower_runs=6, contigs=3)
    want = ob.tnc_counts(data)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + seed
    procs = [ctx.Process(target=_worker, args=(r, 2, port, data, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = np.array(q.get(timeout=120), dtype=np.int64)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert np.array_equal(got, want)
