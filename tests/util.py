"""Shared helpers for the parity tests: run the reference binary / the C model / the engine and compare files, directly or
against the digests of the reference's outputs stored in tests/golden/reference_outputs.json."""
import filecmp
import hashlib
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")
REF63 = os.path.join(ROOT, "oracle", "_ref", "SOAPdenovo-63mer")
REF127 = os.path.join(ROOT, "oracle", "_ref", "SOAPdenovo-127mer")
MODEL63 = os.path.join(ROOT, "oracle", "pregraph_model_63")
MODEL127 = os.path.join(ROOT, "oracle", "pregraph_model_127")
ENGINE63 = os.path.join(ROOT, "soapdenovo2_b200", "bin", "pregraph-b200-63mer")
ENGINE127 = os.path.join(ROOT, "soapdenovo2_b200", "bin", "pregraph-b200-127mer")
SUFFIXES = ["kmerFreq", "vertex", "preGraphBasic", "preArc", "edge.gz"]
SUFFIXES_R = SUFFIXES + ["markOnEdge", "path"]


def have_ref():
    return os.path.exists(REF63) and os.path.exists(REF127)


def build_oracle():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "model"], check=True)


def run(cmd, timeout=600):
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired as ex:   # show where it hung
        err = ex.stderr.decode(errors="replace") if isinstance(ex.stderr, bytes) else (ex.stderr or "")
        raise AssertionError(f"{' '.join(cmd)}\ntimed out after {timeout} s; stderr tail:\n{err[-3000:]}")
    assert r.returncode == 0, f"{' '.join(cmd)}\nrc={r.returncode}\n{r.stderr[-4000:]}"
    return r.stderr


def run_ref(binary, cfg, out, K, P, extra=()):
    return run([binary, "pregraph", "-s", cfg, "-K", str(K), "-p", str(P), "-o", out, *extra])


def run_model(binary, cfg, out, K, P, extra=()):
    return run([binary, "-s", cfg, "-K", str(K), "-p", str(P), "-o", out, *extra])


def compare(a, b, suffixes):
    bad = [s for s in suffixes if not filecmp.cmp(f"{a}.{s}", f"{b}.{s}", shallow=False)]
    assert not bad, f"files differ: {bad} ({a} vs {b})"


# ---- golden reference outputs (written by scripts/make_reference_golden.py from the unmodified reference binaries)
COUNTER_KEYS = ("node(s) allocated", "tip(s) removed", "linear node(s) marked", "edge(s) and", "vertex(es) output", "pre-arc(s) added",
                "kmer(s) removed")
CONTIG_SUFFIXES = ["contig", "Arc", "updated.edge", "ContigIndex"]


def counter_lines(log):
    """The counters a pregraph run prints on stderr (no paths, no times)."""
    return [l.strip() for l in log.splitlines() if any(k in l for k in COUNTER_KEYS)]


def open_order(log):
    """Base names of the read files in the order the run opened them during pass 1."""
    lines = log.splitlines()
    order = []
    for i, l in enumerate(lines):
        if l.startswith("Import reads from file:"):
            order.append(os.path.basename(lines[i + 1].strip()))
        if "done hashing nodes" in l:
            break
    return order


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 20), b""):
            h.update(b)
    return h.hexdigest()


def cfg_inputs(cfg):
    """{base name: sha256} of the read files a config names."""
    out = {}
    for l in open(cfg):
        k, _, v = l.strip().partition("=")
        if k in ("f", "f1", "f2", "q", "q1", "q2"):
            out[os.path.basename(v)] = sha256(v)
    return out


def adversarial_name(crlf, K_hint):
    return f"adversarial_crlf{int(crlf)}_k{K_hint}"


def scenario_midsize(d):
    """2 Mbp genome with a 4-copy 2 kbp repeat, 30x 150 bp PE FASTQ (17.6 M k-mer instances at K=63)."""
    from soapdenovo2_b200 import synth
    g = synth.genome(2_000_000, 11, repeat=(2000, 4))
    r1, r2 = synth.pe_reads(g, 200_000, 150, 300, 0.001, 12)
    synth.write_fastq(os.path.join(d, "a_1.fq"), r1, "m")
    synth.write_fastq(os.path.join(d, "a_2.fq"), r2, "m")
    cfg = os.path.join(d, "mid.cfg")
    synth.write_config(cfg, 150, [{"avg_ins": 300, "files": [("q1", os.path.join(d, "a_1.fq")), ("q2", os.path.join(d, "a_2.fq"))]}])
    return cfg


# Seeds of synth.scenario_fuzz with stored reference outputs (scenario names fuzz<seed>).  Chosen so that every edge the generator
# aims at occurs: max_rd_len 768 (79), 769 (28 29 54 76), 1536 (5), 1537 (162) and above (53 92); lines longer than a 2 KB decode
# tile (5 53 92); CRLF with truncation (1 5 10 ...); both insert paths, each with -d; PGB200_NO_TMA (10 14 23 ...); every K of both
# builds, every -p, -a and -d; single-library cases (FUZZ_TABLE_SEEDS) whose pass-1 table is compared entry by entry.
FUZZ_SEEDS = [1, 2, 5, 10, 14, 15, 20, 23, 24, 27, 28, 29, 32, 33, 36, 38, 44, 46, 48, 49, 50, 51, 52, 53, 54, 59, 60, 61, 63, 68,
              70, 71, 72, 75, 76, 78, 79, 85, 86, 90, 92, 116, 149, 153, 156, 159, 162, 169]
FUZZ_TABLE_SEEDS = [1, 2, 10, 23, 24, 27, 28, 32, 36, 38, 46, 49, 50, 53, 54, 59, 60, 63, 72, 78, 79, 85, 149, 156, 159, 169]


def cfg_libs(cfg):
    """Number of libraries of a config that the pregraph stage reads (asm_flags 1 or 3)."""
    flags = [l.strip().split("=", 1)[1] for l in open(cfg) if l.startswith("asm_flags=")]
    return sum(f in ("1", "3") for f in flags)


def first_difference(a, b):
    """'line N: <a line> != <b line>' for the first line where files a and b differ (.gz files are decompressed)."""
    import gzip
    op = gzip.open if a.endswith(".gz") else open
    with op(a, "rb") as fa, op(b, "rb") as fb:
        for n, (x, y) in enumerate(zip(fa, fb), 1):
            if x != y:
                return f"line {n}: {x[:200]!r} != {y[:200]!r}"
        rest_a, rest_b = fa.read(), fb.read()
    return f"one file is longer ({len(rest_a)} vs {len(rest_b)} trailing bytes)" if rest_a != rest_b else "no difference"


def ref_key(scenario, flavour127, K, P, extra=()):
    return " ".join([scenario, "127mer" if flavour127 else "63mer", "-K", str(K), "-p", str(P), *extra])


_golden = None


def golden(scenario, flavour127, K, P, extra=(), cfg=None):
    """The reference's record for `pregraph -s <scenario> -K K -p P <extra>`: output digests, counter lines, file open order.
    With `cfg`, the read files it names must be the ones the record was made from."""
    global _golden
    if _golden is None:
        _golden = json.load(open(GOLDEN_REF))
    key = ref_key(scenario, flavour127, K, P, extra)
    assert key in _golden["runs"], f"no golden reference record for '{key}' (add it to scripts/make_reference_golden.py)"
    if cfg is not None:
        assert cfg_inputs(cfg) == _golden["inputs"][scenario], f"the {scenario} read set differs from the one the golden record was made from"
    return _golden["runs"][key]


def compare_golden(out, rec, suffixes):
    """Byte identity with the reference's files, through their stored SHA-256 digests."""
    bad = [s for s in suffixes if sha256(f"{out}.{s}") != rec["files"][s]]
    assert not bad, f"files differ from the reference's (golden digests): {bad} ({out})"
