"""GPU parity on the edge cases the reference's own code paths distinguish (there are no reference tests to borrow from):
reads shorter than / exactly K+1, N / '.' / lower case, CRLF, poly-A counter saturation (links 63, coverage 255 under heavy
same-slot contention), tandem repeats, a reverse-complement palindrome (bal_edge = 0), truncation, empty input pieces."""
import os
import subprocess

import pytest

from soapdenovo2_b200 import api, synth
from tests import util
from tests.test_gpu_full import _engine, _oracle, _suffixes

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("crlf,K,P,extra", [(False, 31, 3, ("-R",)), (True, 31, 8, ("-a", "1", "-d", "2")), (True, 63, 4, ("-a", "1", "-R")),
                                            (False, 13, 2, ("-a", "1", "-R"))])
def test_adversarial_inputs(tmp_path, crlf, K, P, extra):
    cfg = synth.scenario_adversarial(str(tmp_path), crlf=crlf, K_hint=max(K, 31))
    gpu = str(tmp_path / "gpu")
    rec = _oracle(util.adversarial_name(crlf, max(K, 31)), cfg, 0, K, P, extra)
    _engine(0, cfg, gpu, K, P, extra)
    util.compare_golden(gpu, rec, _suffixes(extra))


def test_saturation_under_contention():
    """2e5 identical poly-A reads: one k-mer receives 1.4e7 concurrent updates; the entry must end exactly saturated."""
    eng = api.PregraphEngine(K=31, P=1, initG=1, max_rd_len=100)
    rec = b">a\n" + b"A" * 100 + b"\n"
    eng.feed_text(rec * 200000, fastq=False)
    st = eng.finish_pass1()
    assert st.distinct == 1 and st.instances == 200000 * 70
    hist, lin, _ = eng.sweeps()
    assert hist[255] == 1 and sum(hist) == 1 and lin == 1
    eng.build_layout()
    d = eng.dump_nodes()
    # canonical AAAA..A (all zero) vs TTTT..T: A-mer is smaller; left link A (code 0) and right link A saturate at 63
    assert d[:16] == bytes(16) and d[16] == 63 and d[20] == 63 and d[24] == 255 and d[25] & 1 == 0
    eng.close()


def test_short_and_empty_pieces():
    """reads shorter than K+1 are skipped (prlHashReads.c:504); an empty feed is a no-op; a chunk that is not whole records errors."""
    eng = api.PregraphEngine(K=31, P=2, initG=1, max_rd_len=100)
    assert eng.feed_text(b"", fastq=True) == 0
    n = eng.feed_text(b"@s\n" + b"ACGT" * 7 + b"\n+\n" + b"I" * 28 + b"\n" + b"@t\n" + b"ACGTACGA" * 4 + b"\n+\n" + b"I" * 32 + b"\n", fastq=True)
    assert n == 2
    st = eng.finish_pass1()
    assert st.reads_kept == 1 and st.instances == 2          # 28 < K+1 skipped; 32 = K+1 -> 2 k-mers
    with pytest.raises(api.EngineError):
        eng.feed_text(b"@x\nACGT\n+\n", fastq=True)
    eng.close()


@pytest.mark.parametrize("text,fastq", [
    (b">a\nACGTACGTAC\nGGGTTTAAAC\n>b\nACGTACGTAC\nGGGTTTAAAC\n", False),     # multi-line FASTA whose line count is a multiple of 2
    (b"@a\nACGT\n+\nIIII\n\n@b\nACGT\n+\nIIII\n\n\n\n", True),                # stray blank lines, line count a multiple of 4
    (b"@a\nACGT\n-\nIIII\n", True),                                        # separator line does not start with '+'
])
def test_malformed_records_are_rejected(text, fastq):
    """Header lines must start with '>' / '@' and FASTQ separators with '+': the engine must not hash header letters as bases
    (the reference's readseqInBuf keys on '>'; multi-line FASTA is out of scope, so it has to fail loudly)."""
    eng = api.PregraphEngine(K=13, P=2, initG=1, max_rd_len=100)
    with pytest.raises(api.EngineError):
        eng.feed_text(text, fastq=fastq)
        eng.finish_pass1()
    eng.close()


def test_truncation_and_reverse_via_api(tmp_path):
    """maxlen truncation and reverse_seq give the same table as feeding the pre-truncated / pre-reversed reads."""
    import numpy as np
    g = synth.genome(5000, 4)
    r = synth.se_reads(g, 300, 100, 0.0, 5)
    fa = b"".join(b">r\n" + x.tobytes() + b"\n" for x in r)
    comp = {65: 84, 67: 71, 71: 67, 84: 65}
    rc = b"".join(b">r\n" + bytes(comp[c] for c in x.tobytes()[:80][::-1]) + b"\n" for x in r)
    a = api.PregraphEngine(K=31, P=2, initG=1, max_rd_len=100)
    a.feed_text(fa, fastq=False, maxlen=80, reverse_seq=1)
    b = api.PregraphEngine(K=31, P=2, initG=1, max_rd_len=100)
    b.feed_text(rc, fastq=False)
    for e in (a, b):
        e.finish_pass1(); e.sweeps(); e.build_layout()
    assert a.dump_nodes() == b.dump_nodes()
    a.close(); b.close()
