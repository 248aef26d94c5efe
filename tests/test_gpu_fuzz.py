"""GPU parity on the seeded random scenarios of synth.scenario_fuzz (long, truncated and CRLF reads, unusual bytes, several
libraries, K at the key-width edges, random -p / -a / -d / -R), each run with the engine settings its seed draws: insert path,
chunk size, initial table size, bucket count, arena size, flush period, TMA off.  The `pregraph-b200-*` CLI must write every file
byte-identical to the reference's (stored digests) and print the same counters.  On a mismatch the C model, which
tests/test_oracle_fuzz.py pins to the same digests, runs on the same config and the failure names the first differing line.
The single-library seeds also compare the pass-1 node table entry by entry with the model's, over both insert paths."""
import os

import pytest

from soapdenovo2_b200 import api, synth
from tests import util
from tests.test_gpu_full import _engine, _suffixes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _build():
    util.build_oracle()


def _model(flavour127):
    return util.MODEL127 if flavour127 else util.MODEL63


@pytest.mark.parametrize("seed", util.FUZZ_SEEDS)
def test_cli_matches_reference(tmp_path, seed):
    cfg, K, flavour127, P, extra, env = synth.scenario_fuzz(str(tmp_path), seed)
    rec = util.golden(f"fuzz{seed}", flavour127, K, P, extra, cfg=cfg)
    gpu = str(tmp_path / "gpu")
    log = _engine(flavour127, cfg, gpu, K, P, extra, env=env)
    sfx = _suffixes(extra)
    missing = [s for s in sfx if not os.path.exists(f"{gpu}.{s}")]
    assert not missing, f"seed {seed}: no {missing} written"
    bad = [s for s in sfx if util.sha256(f"{gpu}.{s}") != rec["files"][s]]
    if bad:
        mod = str(tmp_path / "mod")
        util.run_model(_model(flavour127), cfg, mod, K, P, extra)
        pytest.fail(f"seed {seed} (K={K} -p {P} {' '.join(extra)} {env}): {bad} differ from the reference's; first difference in "
                    f".{bad[0]}, GPU vs model: {util.first_difference(f'{gpu}.{bad[0]}', f'{mod}.{bad[0]}')}")
    assert util.counter_lines(log) == rec["counters"]


@pytest.mark.parametrize("seed", [
    pytest.param(79, id="chop_insert_48KB_tile_max_rd_len_768"),   # k_chop_insert: tile + static shared memory over the default 48 KB
    pytest.param(5, id="pass2_48KB_tile_max_rd_len_1536"),         # k_pass2: the same at 128 reads x 48 words
])
def test_regression(tmp_path, seed):
    """Seeds that once failed: the launch was refused (invalid argument) because the kernel asked for more shared memory than the
    default limit without opting in."""
    test_cli_matches_reference(tmp_path, seed)


def _feed_file(eng, path, fastq, ord_base, ord_stride, rev, cut, chunk):
    """One read file in pieces of whole records of at most `chunk` bytes (0: in one piece); returns the number of records."""
    data = open(path, "rb").read()
    per = 4 if fastq else 2
    lines = data.split(b"\n")[:-1]
    recs = [b"\n".join(lines[i:i + per]) + b"\n" for i in range(0, len(lines), per)]
    n, piece, size = 0, [], 0
    for r in recs + [None]:
        if piece and (r is None or (chunk and size + len(r) > chunk)):
            n += eng.feed_text(b"".join(piece), fastq=fastq, ord_base=ord_base + n * ord_stride, ord_stride=ord_stride, reverse_seq=rev, maxlen=cut)
            piece, size = [], 0
        if r is not None:
            piece.append(r)
            size += len(r)
    return n


def _feed_plan(eng, cfg, chunk):
    """Feed a config's read files the way the stage does: open order, mates interleaved (ordinal = base + 2 pair + mate),
    reverse_seq, the library's length cut, pieces of at most `chunk` bytes."""
    _, plan = api.plan_files(cfg)
    ord_next, i = 0, 0
    while i < len(plan):
        mate, fastq, rev, cut, path = plan[i]
        if mate == 0:
            n1 = _feed_file(eng, path, bool(fastq), ord_next, 2, rev, cut, chunk)
            _, fq2, rev2, cut2, path2 = plan[i + 1]
            assert _feed_file(eng, path2, bool(fq2), ord_next + 1, 2, rev2, cut2, chunk) == n1
            ord_next += 2 * n1
            i += 2
        else:
            ord_next += _feed_file(eng, path, bool(fastq), ord_next, 1, rev, cut, chunk)
            i += 1


@pytest.mark.parametrize("skm", ["0", "1"], ids=["direct", "aggregated"])
@pytest.mark.parametrize("seed", util.FUZZ_TABLE_SEEDS)
def test_pass1_table_matches_model(tmp_path, monkeypatch, seed, skm):
    """Through the C-ABI: .kmerFreq and the whole node table (k-mer, links, coverage, flags, in the reference's iteration order)."""
    cfg, K, flavour127, P, extra, env = synth.scenario_fuzz(str(tmp_path), seed)
    assert util.cfg_libs(cfg) == 1
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("PGB200_SKM", skm)
    opts = tuple(x for x in extra if x != "-R")
    mod, dump = str(tmp_path / "mod"), str(tmp_path / "mod.table")
    util.run_model(_model(flavour127), cfg, mod, K, P, ("-1", "-T", dump, *opts))
    initG = int(opts[opts.index("-a") + 1]) if "-a" in opts else 0
    D = int(opts[opts.index("-d") + 1]) if "-d" in opts else 0
    max_rd_len, _ = api.plan_files(cfg)
    eng = api.PregraphEngine(K=K, P=P, initG=initG, D=D, flavour127=flavour127, max_rd_len=max_rd_len,
                             table_slots=int(env.get("PGB200_TABLE_SLOTS", 0)))
    try:
        _feed_plan(eng, cfg, int(env.get("PGB200_CHUNK_MB", 0)) << 20)
        eng.finish_pass1()
        hist, _, _ = eng.sweeps()
        assert api.kmerfreq_text(hist) == open(mod + ".kmerFreq", "rb").read()
        eng.build_layout()
        assert eng.dump_nodes() == open(dump, "rb").read()
    finally:
        eng.close()
