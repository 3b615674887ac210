"""CPU: pins the TNC restatement (oracle/tnc_oracle.c) against the reference's own answers."""
import json
import os
import random
import subprocess

import numpy as np
import pytest

import fasta_cases as fc
import oracle_bind as ob
import reference_digests as rd

HERE = os.path.dirname(os.path.abspath(__file__))


def nonzero(text):
    return {l.split("\t")[0]: int(l.split("\t")[1]) for l in text.splitlines() if not l.endswith("\t0")}


@pytest.mark.parametrize("data,expect", fc.KAT)
def test_known_answers_app_b(data, expect):
    assert nonzero(ob.tnc_text(ob.tnc_counts(data))) == expect


def test_golden_fixture():
    """tests/golden/tnc_golden.json was produced by the compiled reference (make_golden.py)."""
    gold = json.load(open(os.path.join(HERE, "golden", "tnc_golden.json")))
    assert len(gold) >= 40
    for case in gold:
        data = bytes.fromhex(case["hex"])
        assert ob.tnc_text(ob.tnc_counts(data)) == case["stdout"], case["hex"]


def test_sum_rule_60col():
    """App. B last row: 59 of every 60 windows outside the N block are counted (independent of the bases)."""
    rng = random.Random(5)
    n, w = 600_000, 60
    data = fc.genome_like(rng, n, width=w, n_block=(99_960, 105_000))
    total = int(ob.tnc_counts(data).sum())
    # two runs of bases, [0,99960) and [105000,600000), both made of whole lines; the all-N lines
    # between them are invisible, so the two runs are joined by one more straddling window
    def run(length):
        lines = length // w
        return lines * (w - 2) + (lines - 1)          # in-line windows + one straddle per line pair
    assert total == run(99_960) + run(495_000) + 1


def test_nul_rejected():
    with pytest.raises(ValueError):
        ob.tnc_counts(b"ACGT\x00ACGT\n")


def test_fuzz_against_compiled_reference(ref_dir, tmp_path):
    """Against oracle/_ref/tncCountsProfile when it is built, else against the digests of its stdout on the same inputs
    (tests/golden/reference_digests.json)."""
    gold = rd.load()["tnc_fuzz"] if ref_dir is None else None
    inputs = rd.tnc_fuzz_inputs()
    assert gold is None or len(gold) == len(inputs)
    for i, data in enumerate(inputs):
        got = ob.tnc_text(ob.tnc_counts(data))
        if gold is not None:
            assert [len(data), rd.sha(data)] == gold[i][:2], "input %d is not the one the digest was recorded on" % i
            assert rd.sha(got.encode()) == gold[i][2], data
            continue
        p = tmp_path / "f.fa"
        p.write_bytes(data)
        ref = subprocess.run([os.path.join(ref_dir, "tncCountsProfile"), str(p)], capture_output=True).stdout.decode()
        assert got == ref, data


def test_missing_file_exit_status(ref_dir):
    exe = os.path.join(ob.ROOT, "oracle", "_build", "tnc_oracle")
    assert subprocess.run([exe, "/nonexistent"], capture_output=True).returncode == 1
    assert subprocess.run([exe], capture_output=True).returncode == 1
