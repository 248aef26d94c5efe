"""CPU: the host-side read-stream plan (config parsing, library sort, file-type order, truncation) against the ORDER in which the
unmodified reference binary opens the files (its "Import reads from file:" stderr lines, stored in tests/golden/reference_outputs.json)."""
import os
import subprocess

import pytest

from soapdenovo2_b200 import api, synth
from tests import util


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-j8", "-C", os.path.join(util.ROOT, "soapdenovo2_b200", "csrc")], check=True)


def test_multilib_plan_matches_reference_open_order(tmp_path):
    cfg = synth.scenario_multilib(str(tmp_path))
    mrl, plan = api.plan_files(cfg)
    assert mrl == 150
    assert [os.path.dirname(p[4]) for p in plan] == [str(tmp_path)] * len(plan)
    assert [os.path.basename(p[4]) for p in plan] == util.golden("multilib", 0, 31, 2)["open_order"]
    by = {os.path.basename(p[4]): p for p in plan}
    assert by["m_a1.fa"][:4] == (0, 0, 0, 150) and by["m_a2.fa"][:4] == (1, 0, 0, 150)
    assert by["m_s.fa"][:4] == (-1, 0, 0, 140) and by["m_q1.fq"][:4] == (0, 1, 0, 140)       # rd_len_cutoff=140
    assert by["m_rq.fq"][:4] == (-1, 1, 1, 150)                                                  # reverse_seq=1
    assert "m_ig.fa" not in by                                                                   # asm_flags=2 is not used by pregraph


def test_config_quirks(tmp_path):
    """max_rd_len only counts before the first [LIB]; '#' lines and unknown keys are ignored; q before f inside a library is
    still opened after f1/f2 and q1/q2; default max_rd_len is 100.  The reference opens the files of this config in the order
    asserted here (a run of the unmodified binary: "Import reads from file:" z1.fq, z2.fq, x.fa, y.fq)."""
    d = str(tmp_path)
    g = synth.genome(3000, 2)
    for name, fq in (("x.fa", False), ("y.fq", True), ("z1.fq", True), ("z2.fq", True)):
        r = synth.se_reads(g, 40, 60, 0.0, hash(name) % 1000)
        (synth.write_fastq if fq else synth.write_fasta)(os.path.join(d, name), r)
    cfg = os.path.join(d, "q.cfg")
    with open(cfg, "w") as f:
        f.write("#a comment\nfoo=bar\n[LIB]\navg_ins=300\nmax_rd_len=50\nq=%s/y.fq\nf=%s/x.fa\nq1=%s/z1.fq\nq2=%s/z2.fq\nasm_flags=1\n" % (d, d, d, d))
    mrl, plan = api.plan_files(cfg)
    assert mrl == 100
    assert [p[4] for p in plan] == [os.path.join(d, n) for n in ("z1.fq", "z2.fq", "x.fa", "y.fq")]


def _fq(n, qual=None, eol=b"\n"):
    out = b""
    for i in range(n):
        q = qual(i) if qual else b"I" * 8
        out += b"@r%d" % i + eol + b"ACGTACGT" + eol + b"+" + eol + q + eol
    return out


def test_chunk_cut_keeps_whole_records():
    """The feeder cuts a buffer that ends inside a record at the last position that is KNOWN to start a record."""
    whole = _fq(5)
    rec = len(whole) // 5
    # the buffer ends inside record 4 (header + part of the sequence line): everything before record 3's start is certainly whole
    # (record 3 itself is the last one whose '+' line is visible), so the cut is at record 3
    assert api.cut_chunk(whole[: 4 * rec + 9], True) == 3 * rec
    # it ends exactly at a record boundary: the last record start found is still the cut (the tail record goes with the next read)
    assert api.cut_chunk(whole, True) == 4 * rec
    # a single, incomplete record: nothing to cut yet
    assert api.cut_chunk(whole[: rec - 3], True) == 0
    assert api.cut_chunk(b"", True) == 0


def test_chunk_cut_is_not_fooled_by_quality_lines_starting_with_at():
    """'@' is a valid quality character (Phred 31): a quality line may start with it.  Two lines after a real header comes the '+'
    line; two lines after such a quality line comes a sequence line."""
    whole = _fq(6, qual=lambda i: b"@" + b"I" * 7)
    rec = len(whole) // 6
    for cut_at in (5 * rec + 2, 5 * rec + 12, 5 * rec + rec - 1):
        off = api.cut_chunk(whole[:cut_at], True)
        assert off % rec == 0 and 0 < off <= 4 * rec + rec, (cut_at, off)
        assert whole[off:off + 2] == b"@r"
    # the same with CRLF line ends
    crlf = _fq(6, qual=lambda i: b"@" + b"I" * 7, eol=b"\r\n")
    rec = len(crlf) // 6
    off = api.cut_chunk(crlf[: 5 * rec + 7], True)
    assert off % rec == 0 and off > 0 and crlf[off:off + 2] == b"@r"


def test_chunk_cut_fasta():
    fa = b"".join(b">s%d\nACGTACGTAC\n" % i for i in range(4))
    rec = len(fa) // 4
    assert api.cut_chunk(fa[: 3 * rec + 4], False) == 3 * rec      # '>' starts a record, the rest of it follows with the next read
    assert api.cut_chunk(fa[: rec - 2], False) == 0
