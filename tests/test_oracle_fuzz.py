"""Pin the C model (oracle/pregraph_model.c) against the reference on the seeded random scenarios of synth.scenario_fuzz: long,
truncated and CRLF reads, unusual bytes, several libraries, K at the key-width edges, random -p / -a / -d / -R.  These are the
seeds tests/test_gpu_fuzz.py runs on the GPU, where the model explains a mismatch.  Every pregraph file must equal the reference's
(SHA-256 digests in tests/golden/reference_outputs.json).  CPU only."""
import pytest

from soapdenovo2_b200 import synth
from tests import util


@pytest.fixture(scope="module", autouse=True)
def _build():
    util.build_oracle()


@pytest.mark.parametrize("seed", util.FUZZ_SEEDS)
def test_model_matches_reference(tmp_path, seed):
    cfg, K, flavour127, P, extra, _env = synth.scenario_fuzz(str(tmp_path), seed)
    rec = util.golden(f"fuzz{seed}", flavour127, K, P, extra, cfg=cfg)
    mod = str(tmp_path / "mod")
    util.run_model(util.MODEL127 if flavour127 else util.MODEL63, cfg, mod, K, P, extra)
    util.compare_golden(mod, rec, util.SUFFIXES_R if "-R" in extra else util.SUFFIXES)


def test_fuzz_seeds_cover_the_edges(tmp_path):
    """The stored seeds keep reaching the shapes they were chosen for (a change to the generator must not lose one)."""
    seen = set()
    for seed in util.FUZZ_SEEDS:
        d = tmp_path / str(seed)
        d.mkdir()
        cfg, K, flavour127, P, extra, env = synth.scenario_fuzz(str(d), seed)
        text = open(cfg).read()
        max_rd_len = int(text.split("max_rd_len=")[1].split()[0])
        seen.add(("max_rd_len", max_rd_len) if max_rd_len in synth.FUZZ_LONG_MAX else ("max_rd_len", max_rd_len > 1537))
        for l in text.splitlines():
            if l.split("=")[0] in ("f", "q", "f1", "f2", "q1", "q2"):
                data = open(l.split("=", 1)[1], "rb").read()
                lines = data.split(b"\n")
                seen.add(("long line", max(len(x) for x in lines) > 2048))
                if b"\r\n" in data and any(len(x.rstrip(b"\r")) >= max_rd_len for x in lines[1::2]):
                    seen.add(("crlf truncated", True))
        seen.add(("K", flavour127, K))
        seen.add(("insert path, -d", env["PGB200_SKM"], "-d" in extra))
        seen.add(("no tma", "PGB200_NO_TMA" in env))
        if seed in util.FUZZ_TABLE_SEEDS:
            assert util.cfg_libs(cfg) == 1, f"seed {seed}: not a single-library case"
    want = {("max_rd_len", m) for m in synth.FUZZ_LONG_MAX} | {("max_rd_len", True), ("long line", True), ("crlf truncated", True),
                                                              ("no tma", True)}
    want |= {("K", 0, k) for k in synth.FUZZ_K63} | {("K", 1, k) for k in synth.FUZZ_K127}
    want |= {("insert path, -d", p, d) for p in ("0", "1") for d in (False, True)}
    assert want <= seen, f"edges no seed reaches: {sorted(want - seen, key=str)}"
