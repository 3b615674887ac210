"""CPU: pins the spike restatement (oracle/spike_oracle.c).

 * against oracle/_ref/stochasticSpike = the UNMODIFIED reference source compiled over oracle/shim/ (only the
   htslib I/O + pileup layer is restated there; "reference logic over shimmed htslib"), byte for byte on SAM,
   truth.vcf and stdout -- or, where that binary is not built, against the digests of its answers on the same inputs
   (tests/golden/reference_digests.json);
 * against the committed golden fixture tests/golden/spike_toy/ (made by tests/golden/make_spike_golden.py with
   that same reference binary), which needs no reference binary;
 * against the glibc rand() known answers of SURVEY.md App. C."""
import os

import numpy as np
import pytest

import oracle_bind as ob
import reference_digests as rd
import spike_cases as sc

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "spike_toy")


def _matches_reference(key, prefix, seed, tmp_path, ref_dir):
    """The restatement against the reference over the shim on one input: byte for byte against oracle/_ref/stochasticSpike when it
    is built, else against the digests of that binary's answers in tests/golden/reference_digests.json."""
    b = sc.run_cli(sc.ORACLE, prefix, str(tmp_path / "ora"), seed=seed, cmdname="stochasticSpike")
    if ref_dir is not None and os.path.exists(sc.REF):
        a = sc.run_cli(sc.REF, prefix, str(tmp_path / "ref"), seed=seed)
        assert a[0] == b[0] == 0
        assert a[2] == b[2], "SAM differs"
        assert a[3] == b[3], "truth.vcf differs"
        assert a[1] == b[1], "stdout differs"
        return
    gold = rd.load()["spike"][key]
    assert gold["seed"] == seed
    assert rd.spike_inputs(prefix) == gold["inputs"], "the generator no longer makes the input the digests were recorded on"
    got = rd.spike_outputs(b, prefix)
    assert got["rc"] == gold["outputs"]["rc"] == 0
    assert got["out.sam"] == gold["outputs"]["out.sam"], "SAM differs"
    assert got["truth.vcf"] == gold["outputs"]["truth.vcf"], "truth.vcf differs"
    assert got["stdout"] == gold["outputs"]["stdout"], "stdout differs"


def reference_case(family, name, outdir):
    """(input prefix, seed) of one input of the two parametrized tests below."""
    if family == "shim":
        return sc.generate(name, outdir), 434
    if name in LONG_READS:
        from test_spike_gpu import _long_read_case
        return _long_read_case(outdir, LONG_READS[name]), 435
    return sc.generate("plain", outdir, **EXTRA_CASES[name]), 435


@pytest.mark.parametrize("name", sorted(sc.CASES))
def test_restatement_matches_reference_over_shim(name, tmp_path, ref_dir):
    prefix, seed = reference_case("shim", name, str(tmp_path))
    _matches_reference("shim/" + name, prefix, seed, tmp_path, ref_dir)


def _gold(name):
    return open(os.path.join(GOLD, name), "rb").read()


def test_golden_fixture_bytes(tmp_path):
    import shutil
    for f in ("in.sam", "in.fa", "in.spike"):
        shutil.copy(os.path.join(GOLD, f), tmp_path / f)
    import subprocess
    env = dict(os.environ, SPIKE_ORACLE_CMDNAME="stochasticSpike")
    r = subprocess.run([sc.ORACLE, "in.sam", "in.fa", "in.spike", "434", "out.sam"], cwd=tmp_path, capture_output=True, env=env)
    assert r.returncode == 0
    assert (tmp_path / "out.sam").read_bytes() == _gold("out.sam")
    assert (tmp_path / "truth.vcf").read_bytes() == _gold("truth.vcf")
    assert r.stdout == _gold("stdout.txt")


def test_simple_spike_fixture_has_no_valid_target():
    """toyExample/simple.spike separates POS and ALT with spaces: strtok("\\t") sees 3 fields, every record is skipped (SURVEY D10)."""
    import stochasticsim_b200.spike as sp
    text = _gold("simple.spike")
    assert sp.parse_spike(text, ["chr19"]) == []


def test_glibc_rand_kat():
    r = ob.glibc_rand(434, 0, 5)
    assert list(r) == [43521843, 555289354, 711778510, 1948175914, 749459303]
    assert int(ob.glibc_rand(434, 10**6, 1)[0]) == 1066614699


def test_usage_exit_status():
    import subprocess
    r = subprocess.run([sc.ORACLE], capture_output=True)
    assert r.returncode == 0 and b"Usage" in r.stderr


def _fuzz_args(k):
    """The generator settings of tests/test_spike_gpu.py::test_fuzz_configs (same seeded draws)."""
    import random
    rng = random.Random(1000 + k)
    rl = rng.choice([36, 50, 76, 100, 151])
    return dict(seed=2000 + k, contigs=rng.choice(["c1:9000", "chrA:6000,chrB:5000", "chr1:4000,chr2:4000,chr3:3000"]),
                coverage=rng.choice([3, 12, 40, 150]), read_len=rl, frag_mean=int(rl * rng.choice([1.05, 1.4, 2.2, 3.0])), frag_sd=rng.choice([3, 15, 40]),
                sub=rng.choice([0.0, 0.002, 0.03]), indel=rng.choice([0.0, 0.01, 0.08]), nrate=rng.choice([0.0, 0.005]), q0=rng.choice([0.0, 0.02]),
                softclip=rng.choice([0.0, 0.1]), refskip=rng.choice([0.0, 0.04]), filt=rng.choice([0.0, 0.1]), lower=rng.choice([0.0, 0.2]),
                spikes=rng.choice([5, 60, 400]), alt_mode=rng.choice([0, 1]), aux=rng.choice([0, 1]), af=rng.choice(["0.01:0.5", "0.3:1.0", "0.001:0.02"]))


EXTRA_CASES = {
    "short36": dict(contigs="chr19:20000", read_len=36, frag_mean=60, frag_sd=6, coverage=60, spikes=80),
    "error_rich": dict(contigs="chr19:12000", coverage=40, sub=0.15, q0=0.1, nrate=0.02, spikes=60),
}
EXTRA_CASES.update({"fuzz%d" % k: _fuzz_args(k) for k in range(8)})
LONG_READS = {"long5k": [5000] * 150, "long_mix": [40000] * 12 + [5000] * 40 + [150] * 300, "long100k": [100000, 90000, 70000]}


@pytest.mark.parametrize("name", sorted(EXTRA_CASES) + sorted(LONG_READS))
def test_restatement_matches_reference_on_gpu_test_inputs(name, tmp_path, ref_dir):
    """Every input family the GPU parity tests use beyond spike_cases.CASES: the restatement must agree with the unmodified
    reference over the shim there too, or those GPU tests would pin nothing."""
    prefix, seed = reference_case("gpu_inputs", name, str(tmp_path))
    _matches_reference("gpu_inputs/" + name, prefix, seed, tmp_path, ref_dir)
