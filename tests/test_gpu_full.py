"""GPU parity, whole stage: `pregraph-b200-{63,127}mer pregraph ...` must write the same bytes as the reference binary for all
seven files, and print the same counters.  The reference's outputs are the SHA-256 digests and counter lines stored in
tests/golden/reference_outputs.json (scripts/make_reference_golden.py)."""
import os
import subprocess

import pytest

from soapdenovo2_b200 import api, synth
from tests import util

pytestmark = pytest.mark.gpu


def _oracle(scenario, cfg, flavour127, K, P, extra):
    """The reference's record for this run (output digests, counter lines)."""
    return util.golden(scenario, flavour127, K, P, extra, cfg=cfg)


def _suffixes(extra):
    return util.SUFFIXES_R if "-R" in extra else util.SUFFIXES


def _engine(flavour127, cfg, out, K, P, extra, env=None):
    exe = api.BIN127 if flavour127 else api.BIN63
    r = subprocess.run([exe, "pregraph", "-s", cfg, "-K", str(K), "-p", str(P), "-o", out, *extra], capture_output=True, text=True,
                       env=dict(os.environ, **(env or {})), timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return r.stderr


@pytest.fixture(scope="module")
def se_cfg(tmp_path_factory):
    return synth.scenario_se_fasta(str(tmp_path_factory.mktemp("se")))


@pytest.fixture(scope="module")
def pe_cfg(tmp_path_factory):
    return synth.scenario_pe_fastq(str(tmp_path_factory.mktemp("pe")))


@pytest.mark.parametrize("K,P,extra", [(31, 3, ("-a", "1", "-R")), (31, 8, ("-a", "1", "-d", "1", "-R")), (31, 1, ("-a", "1")), (21, 5, ("-a", "1", "-d", "3"))])
def test_se_fasta(se_cfg, tmp_path, K, P, extra):
    gpu = str(tmp_path / "gpu")
    rec = _oracle("se", se_cfg, 0, K, P, extra)
    lg = _engine(0, se_cfg, gpu, K, P, extra)
    util.compare_golden(gpu, rec, _suffixes(extra))
    assert rec["counters"] == util.counter_lines(lg)


@pytest.mark.parametrize("P,extra", [(8, ("-a", "1", "-R")), (4, ("-a", "1"))])
def test_pe_fastq_k63(pe_cfg, tmp_path, P, extra):
    gpu = str(tmp_path / "gpu")
    rec = _oracle("pe", pe_cfg, 0, 63, P, extra)
    _engine(0, pe_cfg, gpu, 63, P, extra)
    util.compare_golden(gpu, rec, _suffixes(extra))


@pytest.mark.parametrize("K,P,extra", [(127, 3, ("-a", "1", "-R")), (91, 8, ("-a", "1")), (63, 2, ("-a", "1", "-R"))])
def test_127mer_flavour(pe_cfg, tmp_path, K, P, extra):
    gpu = str(tmp_path / "gpu")
    rec = _oracle("pe", pe_cfg, 1, K, P, extra)
    _engine(1, pe_cfg, gpu, K, P, extra)
    util.compare_golden(gpu, rec, _suffixes(extra))


def test_multilib_k63_small_chunks(tmp_path):
    """4 libraries (FASTA/FASTQ, SE/PE, rd_len_cutoff, reverse_seq, N's, lower case, ignored asm_flags=2 lib); 1 MB host chunks."""
    cfg = synth.scenario_multilib(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = _oracle("multilib", cfg, 0, 63, 8, ("-a", "1", "-R"))
    _engine(0, cfg, gpu, 63, 8, ("-a", "1", "-R"), env={"PGB200_CHUNK_MB": "1", "PGB200_TABLE_SLOTS": "4096"})
    util.compare_golden(gpu, rec, util.SUFFIXES_R)


def test_multilib_k63_aggregated_pass1(tmp_path):
    """The same multi-library case with pass 1 forced through the aggregated path (super-k-mer records, skm.cu), several chunks."""
    cfg = synth.scenario_multilib(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = _oracle("multilib", cfg, 0, 63, 8, ("-a", "1", "-R"))
    _engine(0, cfg, gpu, 63, 8, ("-a", "1", "-R"), env={"PGB200_SKM": "1", "PGB200_CHUNK_MB": "1", "PGB200_TABLE_SLOTS": "4096"})
    util.compare_golden(gpu, rec, util.SUFFIXES_R)


def test_downstream_contig_consumes_gpu_output(tmp_path):
    """configs[4]: the reference's own `contig` stage must produce identical contigs from both pregraph outputs.  The contig
    stage is a deterministic function of the pregraph files, so byte identity with the reference's pregraph files carries over to
    the contigs the golden record holds; where the reference binary is built, its `contig` runs on the GPU output as well."""
    cfg = synth.scenario_multilib(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = _oracle("multilib", cfg, 0, 63, 8, ("-a", "1", "-R"))
    _engine(0, cfg, gpu, 63, 8, ("-a", "1", "-R"))
    util.compare_golden(gpu, rec, util.SUFFIXES_R)
    if util.have_ref():
        util.run([util.REF63, "contig", "-g", gpu, "-R"])
        util.compare_golden(gpu, rec, util.CONTIG_SUFFIXES)


def test_midsize_pe_k63_vs_reference(tmp_path):
    """2 Mbp genome, 30x, 150 bp PE FASTQ, K=63, -p 8 -a 2 -R (17.6 M k-mer instances): exercises many tip rounds, long edges."""
    cfg = util.scenario_midsize(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = _oracle("mid", cfg, 0, 63, 8, ("-a", "2", "-R"))
    lg = _engine(0, cfg, gpu, 63, 8, ("-a", "2", "-R"))
    util.compare_golden(gpu, rec, util.SUFFIXES_R)
    assert rec["counters"] == util.counter_lines(lg)
    # and with the aggregated pass 1 (forced: the CLI feeds host text, which defaults to per-chunk inserts)
    gpu2 = str(tmp_path / "gpu2")
    _engine(0, cfg, gpu2, 63, 8, ("-a", "2", "-R"), env={"PGB200_SKM": "1"})
    util.compare_golden(gpu2, rec, util.SUFFIXES_R)


@pytest.mark.parametrize("K,P,extra", [(31, 3, ("-R",)), (31, 8, ()), (31, 1, ("-d", "1"))])
def test_dynamic_tables_no_a(se_cfg, tmp_path, K, P, extra):
    """f1: without -a the reference's sets grow (in-place rehash with displacement chains); the engine replays the growth history."""
    gpu = str(tmp_path / "gpu")
    rec = _oracle("se", se_cfg, 0, K, P, extra)
    _engine(0, se_cfg, gpu, K, P, extra)
    util.compare_golden(gpu, rec, _suffixes(extra))


def test_dynamic_tables_no_a_pe_127(pe_cfg, tmp_path):
    gpu = str(tmp_path / "gpu")
    rec = _oracle("pe", pe_cfg, 1, 127, 4, ("-R",))
    _engine(1, pe_cfg, gpu, 127, 4, ("-R",))
    util.compare_golden(gpu, rec, util.SUFFIXES_R)
