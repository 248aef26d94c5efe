"""GPU parity, pass 1: .kmerFreq and the full node table (k-mer, 8 link counters, coverage, single/linear/deleted flags) in
REFERENCE ITERATION ORDER must equal the oracle's dump bit for bit.  All calls go through the C-ABI."""
import os

import pytest

from soapdenovo2_b200 import api, synth
from tests import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _build():
    util.build_oracle()


@pytest.fixture(params=["direct", "aggregated"], autouse=True)
def _insert_mode(request, monkeypatch):
    """Every case runs twice: per-instance inserts (k_chop_insert, the default for host text) and the aggregated pass 1 (super-k-mer
    records, skm.cu: the default for device-resident text and the only path across GPUs), both forced through PGB200_SKM."""
    monkeypatch.setenv("PGB200_SKM", "0" if request.param == "direct" else "1")


def _feed_cfg_files(eng, files, fastq, stride=1, base=0, **kw):
    n = 0
    for i, fn in enumerate(files):
        data = open(fn, "rb").read()
        n += eng.feed_text(data, fastq=fastq, ord_base=base + i if stride == 2 else base + n, ord_stride=stride, **kw)
    return n


@pytest.mark.parametrize("K,P,extra", [(31, 3, ("-a", "1")), (31, 8, ("-a", "1", "-d", "1")), (21, 1, ("-a", "1"))])
def test_se_table_dump(tmp_path, K, P, extra):
    cfg = synth.scenario_se_fasta(str(tmp_path))
    mod = str(tmp_path / "mod")
    dump = str(tmp_path / "mod.table")
    util.run_model(util.MODEL63, cfg, mod, K, P, ("-1", "-T", dump, *extra))
    D = int(extra[extra.index("-d") + 1]) if "-d" in extra else 0
    eng = api.PregraphEngine(K=K, P=P, initG=1, D=D, max_rd_len=100)
    _feed_cfg_files(eng, [str(tmp_path / "se.fa")], fastq=False)
    st = eng.finish_pass1()
    hist, lin, rem = eng.sweeps()
    assert api.kmerfreq_text(hist) == open(mod + ".kmerFreq", "rb").read()
    eng.build_layout()
    got, want = eng.dump_nodes(), open(dump, "rb").read()
    assert st.distinct * 26 == len(want)
    assert got == want
    eng.close()


def test_pe_fastq_k63_table_dump(tmp_path):
    cfg = synth.scenario_pe_fastq(str(tmp_path))
    mod, dump = str(tmp_path / "mod"), str(tmp_path / "mod.table")
    util.run_model(util.MODEL63, cfg, mod, 63, 8, ("-1", "-T", dump, "-a", "1"))
    eng = api.PregraphEngine(K=63, P=8, initG=1, max_rd_len=150)
    n1 = eng.feed_text(open(tmp_path / "pe_1.fq", "rb").read(), fastq=True, ord_base=0, ord_stride=2)
    n2 = eng.feed_text(open(tmp_path / "pe_2.fq", "rb").read(), fastq=True, ord_base=1, ord_stride=2)
    assert n1 == n2 == 6000
    st = eng.finish_pass1()
    assert st.instances == 12000 * (150 - 63 + 1)
    hist, _, _ = eng.sweeps()
    assert api.kmerfreq_text(hist) == open(mod + ".kmerFreq", "rb").read()
    eng.build_layout()
    assert eng.dump_nodes() == open(dump, "rb").read()
    eng.close()


def test_k127_table_dump(tmp_path):
    cfg = synth.scenario_pe_fastq(str(tmp_path))
    mod, dump = str(tmp_path / "mod"), str(tmp_path / "mod.table")
    util.run_model(util.MODEL127, cfg, mod, 127, 3, ("-1", "-T", dump, "-a", "1"))
    eng = api.PregraphEngine(K=127, P=3, initG=1, flavour127=1, max_rd_len=150)
    eng.feed_text(open(tmp_path / "pe_1.fq", "rb").read(), fastq=True, ord_base=0, ord_stride=2)
    eng.feed_text(open(tmp_path / "pe_2.fq", "rb").read(), fastq=True, ord_base=1, ord_stride=2)
    eng.finish_pass1()
    hist, _, _ = eng.sweeps()
    assert api.kmerfreq_text(hist) == open(mod + ".kmerFreq", "rb").read()
    eng.build_layout()
    assert eng.dump_nodes() == open(dump, "rb").read()
    eng.close()


def test_chunked_feed_and_growth(tmp_path):
    """Feeding the same file in many small chunks with a tiny initial table (forces growth) must not change anything."""
    cfg = synth.scenario_se_fasta(str(tmp_path))
    mod, dump = str(tmp_path / "mod"), str(tmp_path / "mod.table")
    util.run_model(util.MODEL63, cfg, mod, 31, 3, ("-1", "-T", dump, "-a", "1"))
    data = open(tmp_path / "se.fa", "rb").read()
    eng = api.PregraphEngine(K=31, P=3, initG=1, max_rd_len=100, table_slots=1024)
    lines = data.split(b"\n")[:-1]
    recs = [b"\n".join(lines[i:i + 2]) + b"\n" for i in range(0, len(lines), 2)]
    base = 0
    for i in range(0, len(recs), 500):
        base += eng.feed_text(b"".join(recs[i:i + 500]), fastq=False, ord_base=base)
    assert base == 4000
    st = eng.finish_pass1()
    assert st.table_slots > 1024
    eng.sweeps()
    eng.build_layout()
    assert eng.dump_nodes() == open(dump, "rb").read()
    eng.close()


def test_cli_pass1_kmerfreq_vs_reference(tmp_path):
    cfg = synth.scenario_multilib(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = util.golden("multilib", 0, 63, 8, ("-a", "1"), cfg=cfg)
    env = dict(os.environ, PGB200_PASS1_ONLY="1")
    import subprocess
    r = subprocess.run([api.BIN63, "pregraph", "-s", cfg, "-K", "63", "-p", "8", "-a", "1", "-o", gpu], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    util.compare_golden(gpu, rec, ["kmerFreq"])
    line = [l for l in r.stderr.splitlines() if "node(s) allocated" in l][0]
    assert line.strip() in rec["counters"]


@pytest.mark.parametrize("K,flav,buckets,arena_mb,every", [(63, 0, "1", "0", "0"), (63, 0, "3", "1", "2"), (127, 1, "2", "0", "0"), (127, 1, "4096", "1", "3"), (31, 0, "0", "1", "1")])
def test_aggregated_stress_paths(tmp_path, monkeypatch, K, flav, buckets, arena_mb, every):
    """The aggregated pass 1 under stress: 1..4 buckets (every k-mer spills past the shared-memory table and buckets are deferred
    until the tiny global table has grown), a 1 MB arena (mid-stream flushes because the arena is full), periodic flushes, many
    small chunks.  Same table dump as the oracle."""
    if os.environ.get("PGB200_SKM") == "0":
        pytest.skip("aggregated path only")
    if buckets != "0":
        monkeypatch.setenv("PGB200_SKM_BUCKETS", buckets)
    if arena_mb != "0":
        monkeypatch.setenv("PGB200_SKM_ARENA_MB", arena_mb)
    if every != "0":
        monkeypatch.setenv("PGB200_SKM_FLUSH_EVERY", every)
    cfg = synth.scenario_pe_fastq(str(tmp_path))
    mod, dump = str(tmp_path / "mod"), str(tmp_path / "mod.table")
    util.run_model(util.MODEL127 if flav else util.MODEL63, cfg, mod, K, 4, ("-1", "-T", dump, "-a", "1"))
    eng = api.PregraphEngine(K=K, P=4, initG=1, flavour127=flav, max_rd_len=150, table_slots=2048)
    for mate, fn in enumerate(("pe_1.fq", "pe_2.fq")):
        lines = open(tmp_path / fn, "rb").read().split(b"\n")[:-1]
        recs = [b"\n".join(lines[i:i + 4]) + b"\n" for i in range(0, len(lines), 4)]
        for i in range(0, len(recs), 700):
            eng.feed_text(b"".join(recs[i:i + 700]), fastq=True, ord_base=2 * i + mate, ord_stride=2)
    st = eng.finish_pass1()
    assert st.table_slots > 2048
    hist, _, _ = eng.sweeps()
    assert api.kmerfreq_text(hist) == open(mod + ".kmerFreq", "rb").read()
    eng.build_layout()
    assert eng.dump_nodes() == open(dump, "rb").read()
    eng.close()


SKM_SOFT_LIMIT = 1024 - 256 - 64   # skm.cu: claims in a bucket's shared-memory table stop at this many distinct k-mers


@pytest.mark.gpu
@pytest.mark.parametrize("K,flav,D,buckets", [(31, 0, 0, "2"), (63, 0, 1, "3"), (91, 1, 0, "2"), (31, 0, 2, "0"),
                                              *[(k, f, d, "limit") for k, f in ((31, 0), (63, 0), (127, 1)) for d in (1, 2, 3)]])
def test_fused_sweeps_with_spilled_keys(tmp_path, monkeypatch, K, flav, D, buckets):
    """One aggregation launch into a table that is large enough (no growth): the end-of-pass sweeps ride on its flush, and the keys
    whose instances went straight to the table (2-3 buckets: almost every k-mer spills past the shared-memory table) are swept from
    the launch's list afterwards.  kmerFreq, the linear / deleted flags (table dump) and the counters equal the oracle's; a second
    sweeps() call returns the same numbers.

    "limit": about two soft limits of distinct k-mers per bucket, so nearly every bucket's claim count crosses the limit while its
    warps run, and a key can be claimed in shared memory by one warp while another spills an instance of it.  With -d the flush must
    then store that partial aggregate unswept (links seen once in each part add up to 2, not 0 + 1)."""
    if os.environ.get("PGB200_SKM") == "0":
        pytest.skip("aggregated path only")
    monkeypatch.setenv("PGB200_SKM", "1")
    cfg = synth.scenario_pe_fastq(str(tmp_path))
    mod, dump = str(tmp_path / "mod"), str(tmp_path / "mod.table")
    extra = ("-1", "-T", dump, "-a", "1") + (("-d", str(D)) if D else ())
    util.run_model(util.MODEL127 if flav else util.MODEL63, cfg, mod, K, 4, extra)
    if buckets == "limit":
        distinct = os.path.getsize(dump) // ((4 if flav else 2) * 8 + 10)
        buckets = str(max(1, distinct // (2 * SKM_SOFT_LIMIT)))
    if buckets != "0":
        monkeypatch.setenv("PGB200_SKM_BUCKETS", buckets)
    eng = api.PregraphEngine(K=K, P=4, initG=1, D=D, flavour127=flav, max_rd_len=150)
    for mate, fn in enumerate(("pe_1.fq", "pe_2.fq")):
        eng.feed_text(open(tmp_path / fn, "rb").read(), fastq=True, ord_base=mate, ord_stride=2)
    eng.finish_pass1()
    hist, lin, rem = eng.sweeps()
    assert api.kmerfreq_text(hist) == open(mod + ".kmerFreq", "rb").read()
    assert (hist, lin, rem) == eng.sweeps()
    eng.build_layout()
    assert eng.dump_nodes() == open(dump, "rb").read()
    eng.close()
