#!/usr/bin/env python
"""Run the unmodified reference binaries (oracle/_ref, built by oracle/Makefile where the reference sources exist) on every
scenario the parity tests compare against, and store what they wrote as tests/golden/reference_outputs.json:

  inputs[scenario]  SHA-256 of each read file the scenario generates (the records are only valid for exactly these reads)
  runs[key]         SHA-256 of every pregraph output file (and of the `contig -R` outputs where a test checks them), the
                    counter lines of the log (util.counter_lines) and the order pass 1 opened the read files in

The tests look records up by util.ref_key(scenario, flavour127, K, P, extra); a test case missing here fails with that key.
Usage: python scripts/make_reference_golden.py [-j JOBS]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from soapdenovo2_b200 import synth  # noqa: E402
from tests import util  # noqa: E402

SCENARIOS = {
    "se": synth.scenario_se_fasta,
    "pe": synth.scenario_pe_fastq,
    "multilib": synth.scenario_multilib,
    "mid": util.scenario_midsize,
    "c1": synth.config_c1,
    "c2": synth.config_c2,
    "c5": synth.config_c5,
}
for _crlf, _k in ((False, 31), (True, 31), (True, 63)):
    SCENARIOS[util.adversarial_name(_crlf, _k)] = (lambda c, k: lambda d: synth.scenario_adversarial(d, crlf=c, K_hint=k))(_crlf, _k)

R, A1 = ("-R",), ("-a", "1")
# (scenario, flavour127, K, P, extra, run the contig stage too)
CASES = [
    # tests/test_oracle_vs_ref.py
    *[("se", 0, 31, P, ("-R", *x), False) for P, x in [(1, ()), (3, ()), (8, ()), (3, A1), (8, ("-d", "1")), (8, ("-d", "3", "-a", "1"))]],
    ("pe", 0, 63, 8, R, False), ("pe", 0, 63, 4, A1, False),
    ("pe", 1, 127, 3, R, False), ("pe", 1, 91, 8, (), False), ("pe", 1, 127, 1, ("-a", "3"), False),
    ("pe", 0, 63, 8, ("-d", "2", "-R"), False), ("pe", 0, 45, 5, ("-d", "1", "-a", "1", "-R"), False), ("pe", 0, 23, 2, (), False),
    ("multilib", 1, 99, 4, ("-R", "-d", "1"), False), ("multilib", 0, 63, 8, R, False),
    ("se", 0, 30, 2, (), False), ("se", 0, 7, 2, (), False),
    (util.adversarial_name(False, 31), 0, 31, 3, R, False), (util.adversarial_name(True, 31), 0, 31, 8, ("-a", "1", "-d", "2"), False),
    (util.adversarial_name(True, 63), 0, 63, 4, ("-a", "1", "-R"), False),
    # tests/test_host_logic.py
    ("multilib", 0, 31, 2, (), False),
    # tests/test_gpu_full.py, tests/test_gpu_edge.py
    ("se", 0, 31, 3, ("-a", "1", "-R"), False), ("se", 0, 31, 8, ("-a", "1", "-d", "1", "-R"), False), ("se", 0, 31, 1, A1, False),
    ("se", 0, 21, 5, ("-a", "1", "-d", "3"), False),
    ("pe", 0, 63, 8, ("-a", "1", "-R"), False),
    ("pe", 1, 127, 3, ("-a", "1", "-R"), False), ("pe", 1, 91, 8, A1, False), ("pe", 1, 63, 2, ("-a", "1", "-R"), False),
    ("multilib", 0, 63, 8, ("-a", "1", "-R"), True),
    ("mid", 0, 63, 8, ("-a", "2", "-R"), False),
    ("se", 0, 31, 3, R, False), ("se", 0, 31, 8, (), False), ("se", 0, 31, 1, ("-d", "1"), False),
    ("pe", 1, 127, 4, R, False),
    (util.adversarial_name(False, 31), 0, 13, 2, ("-a", "1", "-R"), False),
    # tests/test_gpu_pass1.py
    ("multilib", 0, 63, 8, A1, False),
    # tests/test_gpu_configs.py
    ("c1", 0, 31, 8, A1, False), ("c2", 0, 63, 8, ("-a", "2", "-R"), False), ("c5", 0, 63, 8, ("-a", "4", "-R"), True),
]


def _fuzz_cases():
    """tests/test_oracle_fuzz.py, tests/test_gpu_fuzz.py: the run options synth.scenario_fuzz draws for each seed."""
    out = []
    with tempfile.TemporaryDirectory() as d:
        for seed in util.FUZZ_SEEDS:
            SCENARIOS[f"fuzz{seed}"] = (lambda s: lambda dd: synth.scenario_fuzz(dd, s)[0])(seed)
            _cfg, K, flavour127, P, extra, _env = synth.scenario_fuzz(d, seed)
            out.append((f"fuzz{seed}", flavour127, K, P, extra, False))
    return out


CASES += _fuzz_cases()


def record(work, scenario, flavour127, K, P, extra, contig):
    ref = util.REF127 if flavour127 else util.REF63
    d = tempfile.mkdtemp(dir=work)
    cfg = SCENARIOS[scenario](d)
    out = os.path.join(d, "ref")
    log = util.run([ref, "pregraph", "-s", cfg, "-K", str(K), "-p", str(P), "-o", out, *extra], timeout=3600)
    rec = {"files": {s: util.sha256(f"{out}.{s}") for s in util.SUFFIXES_R if os.path.exists(f"{out}.{s}")},
           "counters": util.counter_lines(log), "open_order": util.open_order(log)}
    if contig:
        util.run([ref, "contig", "-g", out, "-R"], timeout=3600)
        rec["files"].update({s: util.sha256(f"{out}.{s}") for s in util.CONTIG_SUFFIXES})
    inputs = util.cfg_inputs(cfg)
    subprocess.run(["rm", "-rf", d], check=True)
    print("recorded", util.ref_key(scenario, flavour127, K, P, extra), flush=True)
    return scenario, util.ref_key(scenario, flavour127, K, P, extra), rec, inputs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("-j", "--jobs", type=int, default=4)
    args = ap.parse_args()
    if not util.have_ref():
        raise SystemExit("oracle/_ref/SOAPdenovo-{63,127}mer missing: build them with `make -C oracle ref` where the reference sources are")
    uniq = {util.ref_key(*c[:5]): c for c in CASES}
    with tempfile.TemporaryDirectory() as work, ThreadPoolExecutor(args.jobs) as ex:
        results = list(ex.map(lambda c: record(work, *c), uniq.values()))
    golden = {"inputs": {}, "runs": {}}
    for scenario, key, rec, inputs in results:
        assert golden["inputs"].setdefault(scenario, inputs) == inputs, f"{scenario}: read set not reproducible"
        golden["runs"][key] = rec
    with open(util.GOLDEN_REF, "w") as f:
        json.dump(golden, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
