"""Writes tests/golden/reference_digests.json: the answers of the unmodified reference (oracle/_ref/, built by `make ref` from the
upstream sources STOCHASTICSIM_SRC points to) on every input of the restatement tests, as lengths and SHA-256 digests.

    python tests/golden/make_reference_digests.py
    python tests/golden/make_reference_digests.py --from-restatement "<why the restatements' answers are the reference's>"

The second form records the restatements' answers instead, for where the upstream sources are not at hand.  It is only valid at a
commit whose tests compared the restatements with the reference on these same inputs, and the note must name that commit."""
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import json  # noqa: E402

import oracle_bind as ob  # noqa: E402
import reference_digests as rd  # noqa: E402
import spike_cases as sc  # noqa: E402
import test_spike_oracle as tso  # noqa: E402


def main():
    from_restatement = len(sys.argv) == 3 and sys.argv[1] == "--from-restatement"
    if not from_restatement and len(sys.argv) != 1:
        raise SystemExit(__doc__)
    subprocess.run(["make", "-s", "-C", ROOT, "all", "oracle"], check=True, stdout=subprocess.DEVNULL)
    tnc_ref = os.path.join(ROOT, "oracle", "_ref", "tncCountsProfile")
    if not from_restatement and not (os.path.exists(sc.REF) and os.path.exists(tnc_ref)):
        raise SystemExit("oracle/_ref is not built: set STOCHASTICSIM_SRC and run `make ref REFERENCE=$STOCHASTICSIM_SRC`")
    out = {"recorded_with": sys.argv[2] if from_restatement else "oracle/_ref (the unmodified reference)", "spike": {}, "tnc_fuzz": []}
    with tempfile.TemporaryDirectory() as td:
        fams = [("shim", n) for n in sorted(sc.CASES)] + [("gpu_inputs", n) for n in sorted(tso.EXTRA_CASES) + sorted(tso.LONG_READS)]
        for fam, name in fams:
            d = os.path.join(td, fam, name)
            os.makedirs(d)
            prefix, seed = tso.reference_case(fam, name, d)
            if from_restatement:
                run = sc.run_cli(sc.ORACLE, prefix, os.path.join(d, "out"), seed=seed, cmdname="stochasticSpike")
            else:
                run = sc.run_cli(sc.REF, prefix, os.path.join(d, "out"), seed=seed)
            assert run[0] == 0, run[4]
            out["spike"][fam + "/" + name] = {"seed": seed, "inputs": rd.spike_inputs(prefix), "outputs": rd.spike_outputs(run, prefix)}
        p = os.path.join(td, "f.fa")
        for data in rd.tnc_fuzz_inputs():
            if from_restatement:
                text = ob.tnc_text(ob.tnc_counts(data)).encode()
            else:
                open(p, "wb").write(data)
                text = subprocess.run([tnc_ref, p], capture_output=True, check=True).stdout
            out["tnc_fuzz"].append([len(data), rd.sha(data), rd.sha(text)])
    with open(rd.PATH, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print("%s: %d spike inputs, %d TNC inputs" % (rd.PATH, len(out["spike"]), len(out["tnc_fuzz"])))


if __name__ == "__main__":
    main()
