"""Digests of the unmodified reference's answers on the inputs of the restatement tests (tests/test_spike_oracle.py,
tests/test_tnc_oracle.py).  Where the reference binaries (oracle/_ref/, built from the upstream sources STOCHASTICSIM_SRC
points to) are absent, those tests compare the restatements with tests/golden/reference_digests.json instead; where they are
present, the tests compare with the binaries themselves.  tests/golden/make_reference_digests.py writes the file."""
import hashlib
import json
import os
import random

import fasta_cases as fc

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
TNC_FUZZ_SEED, TNC_FUZZ_N = 11, 300


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def load():
    return json.load(open(PATH))


def tnc_fuzz_inputs():
    """The FASTAs of test_fuzz_against_compiled_reference: fasta_cases.EDGE, then seeded random ones."""
    rng = random.Random(TNC_FUZZ_SEED)
    return [fc.EDGE[i] if i < len(fc.EDGE) else fc.random_fasta(rng) for i in range(TNC_FUZZ_N)]


def spike_inputs(prefix):
    """[length, sha256] of <prefix>.{sam,fa,spike}: shows that the seeded generator still makes the input a digest belongs to."""
    out = {}
    for ext in ("sam", "fa", "spike"):
        b = open(prefix + "." + ext, "rb").read()
        out[ext] = [len(b), sha(b)]
    return out


def spike_outputs(run, prefix):
    """Exit status and [length, sha256] of stdout, out.sam and truth.vcf of a spike_cases.run_cli result on the input at `prefix`.
    truth.vcf's ##stochasticSpikeCommand line names the input files, so their directory is replaced by a fixed token first."""
    d = os.path.dirname(prefix).encode()
    out = {"rc": run[0]}
    for key, b in (("stdout", run[1]), ("out.sam", run[2]), ("truth.vcf", run[3])):
        out[key] = None if b is None else [len(b.replace(d, b"<in>")), sha(b.replace(d, b"<in>"))]
    return out
