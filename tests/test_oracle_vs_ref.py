"""Pin the CPU restatement (oracle/pregraph_model.c) against the UNMODIFIED reference binary.  The reference ships no tests or
golden vectors (SURVEY.md section 4), so byte identity of all seven pregraph outputs on the Appendix-B scenarios is the pin: the
reference's outputs are stored as SHA-256 digests in tests/golden/reference_outputs.json (scripts/make_reference_golden.py runs
the reference binaries that oracle/Makefile builds).  CPU only."""
import os

import pytest

from soapdenovo2_b200 import synth
from tests import util


@pytest.fixture(scope="module", autouse=True)
def _build():
    util.build_oracle()


@pytest.fixture(scope="module")
def se_cfg(tmp_path_factory):
    return synth.scenario_se_fasta(str(tmp_path_factory.mktemp("se")))


@pytest.fixture(scope="module")
def pe_cfg(tmp_path_factory):
    return synth.scenario_pe_fastq(str(tmp_path_factory.mktemp("pe")))


def _model_vs_ref(scenario, cfg, tmp_path, flavour127, K, P, extra):
    """The model's files must be the reference's, byte for byte (all seven with -R)."""
    rec = util.golden(scenario, flavour127, K, P, extra, cfg=cfg)
    mod = str(tmp_path / "mod")
    util.run_model(util.MODEL127 if flavour127 else util.MODEL63, cfg, mod, K, P, extra)
    util.compare_golden(mod, rec, util.SUFFIXES_R if "-R" in extra else util.SUFFIXES)


@pytest.mark.parametrize("P,extra", [(1, ()), (3, ()), (8, ()), (3, ("-a", "1")), (8, ("-d", "1")), (8, ("-d", "3", "-a", "1"))])
def test_se_fasta_k31(se_cfg, tmp_path, P, extra):
    _model_vs_ref("se", se_cfg, tmp_path, 0, 31, P, ("-R", *extra))


@pytest.mark.parametrize("P,extra", [(8, ("-R",)), (4, ("-a", "1"))])
def test_pe_fastq_k63(pe_cfg, tmp_path, P, extra):
    _model_vs_ref("pe", pe_cfg, tmp_path, 0, 63, P, extra)


@pytest.mark.parametrize("K,P,extra", [(127, 3, ("-R",)), (91, 8, ()), (127, 1, ("-a", "3"))])
def test_pe_fastq_127mer_build(pe_cfg, tmp_path, K, P, extra):
    _model_vs_ref("pe", pe_cfg, tmp_path, 1, K, P, extra)


@pytest.mark.parametrize("K,P,extra", [(63, 8, ("-d", "2", "-R")), (45, 5, ("-d", "1", "-a", "1", "-R")), (23, 2, ())])
def test_pe_fastq_more_k_and_cutoffs(pe_cfg, tmp_path, K, P, extra):
    """-d together with -R at K = 63 (delow before the edges and the read paths), an odd K between the word sizes, the default K."""
    _model_vs_ref("pe", pe_cfg, tmp_path, 0, K, P, extra)


def test_multilib_127mer_build(tmp_path):
    _model_vs_ref("multilib", synth.scenario_multilib(str(tmp_path)), tmp_path, 1, 99, 4, ("-R", "-d", "1"))


def test_multilib_k63(tmp_path):
    _model_vs_ref("multilib", synth.scenario_multilib(str(tmp_path)), tmp_path, 0, 63, 8, ("-R",))


def test_k_fixups(se_cfg, tmp_path):
    """even K -> K+1, K<13 -> 13 (pregraph.c:71-97)."""
    for k in (30, 7):
        os.makedirs(tmp_path / f"k{k}")
        _model_vs_ref("se", se_cfg, tmp_path / f"k{k}", 0, k, 2, ())


@pytest.mark.parametrize("crlf,K,P,extra", [(False, 31, 3, ("-R",)), (True, 31, 8, ("-a", "1", "-d", "2")), (True, 63, 4, ("-a", "1", "-R"))])
def test_adversarial_inputs(tmp_path, crlf, K, P, extra):
    """ragged lengths (< K+1, == K+1), N / '.' / lower case, poly-A saturation, tandem repeat, palindrome, CRLF."""
    cfg = synth.scenario_adversarial(str(tmp_path), crlf=crlf, K_hint=K)
    _model_vs_ref(util.adversarial_name(crlf, K), cfg, tmp_path, 0, K, P, extra)
