#!/usr/bin/env python
"""Fuzz the CPU oracle (oracle/pregraph_model.c) against the unmodified reference binary on the seeded random scenarios of
synth.scenario_fuzz: read formats, libraries, ragged / long / truncated reads, CRLF, unusual bytes, K, -p, -a, -d, -R, 63- and
127-mer builds.  CPU only; `python scripts/fuzz_oracle.py [n_cases] [seed0] [-j jobs]`.
Prints one line per case and the mismatching suffixes, exit code 1 if any case differs."""
import argparse
import filecmp
import os
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from soapdenovo2_b200 import synth   # noqa: E402
from tests import util               # noqa: E402


def one_case(seed: int):
    with tempfile.TemporaryDirectory() as d:
        cfg, K, big, P, extra, _env = synth.scenario_fuzz(d, seed)
        ref_bin, mod_bin = (util.REF127, util.MODEL127) if big else (util.REF63, util.MODEL63)
        ref, mod = os.path.join(d, "ref"), os.path.join(d, "mod")
        util.run_ref(ref_bin, cfg, ref, K, P, extra)
        util.run_model(mod_bin, cfg, mod, K, P, extra)
        sfx = util.SUFFIXES_R if "-R" in extra else util.SUFFIXES
        bad = [s for s in sfx if not filecmp.cmp(f"{ref}.{s}", f"{mod}.{s}", shallow=False)]
    return f"seed {seed} {'127' if big else '63'}mer K {K} P {P} {' '.join(extra)}", bad


def checked(seed: int):
    try:
        return one_case(seed)
    except Exception as e:   # a crash of either binary is a finding too
        return f"seed {seed}", [f"EXCEPTION {str(e)[-300:]}"]


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=40)
    ap.add_argument("seed0", type=int, nargs="?", default=1000)
    ap.add_argument("-j", "--jobs", type=int, default=1)
    args = ap.parse_args()
    util.build_oracle()
    fails = 0
    with ThreadPoolExecutor(args.jobs) as ex:
        for desc, bad in ex.map(checked, range(args.seed0, args.seed0 + args.n)):
            print(desc, "OK" if not bad else f"DIFF {bad}", flush=True)
            fails += bool(bad)
    sys.exit(1 if fails else 0)
