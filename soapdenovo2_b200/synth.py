"""Seeded synthetic read sets for the pregraph path (host-side numpy; test + bench plumbing, not the product path).

Recipe follows SURVEY.md section 8(d): uniform i.i.d. ACGT genome, uniform fragment starts, i.i.d. substitution
errors, constant quality 'I'.  Files avoid the reference reader's quirks (SURVEY.md A.9): single-line FASTA,
4-line FASTQ, trailing newline, sizes that are not a multiple of 32768 bytes.
"""
from __future__ import annotations

import os
import numpy as np

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTNacgtn", b"TGCANtgcan"):
    _COMP[_a] = _b


def genome(n: int, seed: int, repeat: tuple[int, int] | None = None) -> np.ndarray:
    rng = np.random.default_rng(seed)
    g = _ACGT[rng.integers(0, 4, size=n)]
    if repeat is not None:  # (length, copies): plant an exact repeat so the graph has real branches
        ln, copies = repeat
        unit = g[:ln].copy()
        for c in range(1, copies):
            p = (c * n) // copies
            g[p:p + ln] = unit
    return g


def _mutate(reads: np.ndarray, err: float, rng) -> np.ndarray:
    if err <= 0:
        return reads
    mask = rng.random(reads.shape) < err
    idx = np.searchsorted(_ACGT, reads[mask])  # 0..3 in "ACGT" order
    reads[mask] = _ACGT[(idx + rng.integers(1, 4, size=idx.shape)) % 4]
    return reads


def _sample(g: np.ndarray, n_reads: int, rd_len: int, rng, starts=None) -> np.ndarray:
    if starts is None:
        starts = rng.integers(0, len(g) - rd_len + 1, size=n_reads)
    return g[starts[:, None] + np.arange(rd_len)[None, :]].copy()


def _revcomp(reads: np.ndarray) -> np.ndarray:
    return _COMP[reads[:, ::-1]]


def _pad_if_32k(path: str) -> None:
    """The reference's AIO reader mis-handles files whose size is k*32768 (SURVEY.md A.9): dodge by renaming a read."""
    if os.path.getsize(path) % 32768 == 0:
        with open(path, "rb") as f:
            data = f.read()
        nl = data.index(b"\n")
        with open(path, "wb") as f:
            f.write(data[:nl] + b"x" + data[nl:])


def write_fasta(path: str, reads: np.ndarray, tag: str = "r") -> None:
    n, L = reads.shape
    with open(path, "wb") as f:
        for i in range(n):
            f.write(b">" + f"{tag}{i}".encode() + b"\n")
            f.write(reads[i].tobytes() + b"\n")
    _pad_if_32k(path)


def write_fastq(path: str, reads: np.ndarray, tag: str = "r") -> None:
    n, L = reads.shape
    q = b"I" * L
    with open(path, "wb") as f:
        for i in range(n):
            f.write(b"@" + f"{tag}{i}".encode() + b"\n" + reads[i].tobytes() + b"\n+\n" + q + b"\n")
    _pad_if_32k(path)


def se_reads(g, n_reads, rd_len, err, seed, both_strands=True):
    rng = np.random.default_rng(seed)
    r = _sample(g, n_reads, rd_len, rng)
    if both_strands:
        flip = rng.random(n_reads) < 0.5
        r[flip] = _revcomp(r[flip])
    return _mutate(r, err, rng)


def pe_reads(g, n_pairs, rd_len, insert, err, seed):
    rng = np.random.default_rng(seed)
    starts = rng.integers(0, len(g) - insert + 1, size=n_pairs)
    r1 = _sample(g, n_pairs, rd_len, rng, starts)
    r2 = _revcomp(_sample(g, n_pairs, rd_len, rng, starts + insert - rd_len))
    flip = rng.random(n_pairs) < 0.5  # fragment strand
    r1f, r2f = r1.copy(), r2.copy()
    r1f[flip], r2f[flip] = r2[flip], r1[flip]
    return _mutate(r1f, err, rng), _mutate(r2f, err, rng)


def write_config(path: str, max_rd_len: int, libs: list[dict]) -> None:
    """libs: [{'avg_ins':200, 'reverse_seq':0, 'asm_flags':3, 'rd_len_cutoff':None, 'files':[('q1',p),('q2',p),...]}]"""
    with open(path, "w") as f:
        f.write(f"max_rd_len={max_rd_len}\n")
        for lib in libs:
            f.write("[LIB]\n")
            f.write(f"avg_ins={lib.get('avg_ins', 200)}\n")
            f.write(f"reverse_seq={lib.get('reverse_seq', 0)}\n")
            f.write(f"asm_flags={lib.get('asm_flags', 3)}\n")
            if lib.get("rd_len_cutoff"):
                f.write(f"rd_len_cutoff={lib['rd_len_cutoff']}\n")
            f.write("rank=1\n")
            for k, p in lib["files"]:
                f.write(f"{k}={p}\n")


# ---------------------------------------------------------------- canned scenarios (SURVEY.md Appendix B list)
def scenario_se_fasta(d: str, genome_len=20000, n_reads=4000, rd_len=100, err=0.005, seed=1) -> str:
    g = genome(genome_len, seed)
    write_fasta(os.path.join(d, "se.fa"), se_reads(g, n_reads, rd_len, err, seed + 100))
    cfg = os.path.join(d, "se.cfg")
    write_config(cfg, rd_len, [{"avg_ins": 200, "files": [("f", os.path.join(d, "se.fa"))]}])
    return cfg


def scenario_pe_fastq(d: str, genome_len=60000, n_pairs=6000, rd_len=150, insert=300, err=0.004, seed=3,
                      repeat=(400, 3)) -> str:
    g = genome(genome_len, seed, repeat=repeat)
    r1, r2 = pe_reads(g, n_pairs, rd_len, insert, err, seed + 100)
    write_fastq(os.path.join(d, "pe_1.fq"), r1, "p")
    write_fastq(os.path.join(d, "pe_2.fq"), r2, "p")
    cfg = os.path.join(d, "pe.cfg")
    write_config(cfg, rd_len, [{"avg_ins": insert, "files": [("q1", os.path.join(d, "pe_1.fq")), ("q2", os.path.join(d, "pe_2.fq"))]}])
    return cfg


def scenario_multilib(d: str, genome_len=40000, seed=5) -> str:
    """4 libraries, mixed FASTA/FASTQ/SE/PE, rd_len_cutoff, reverse_seq, N's + lower case, an asm_flags=2 lib to ignore."""
    g = genome(genome_len, seed, repeat=(300, 2))
    rng = np.random.default_rng(seed + 7)
    a1, a2 = pe_reads(g, 1500, 100, 500, 0.004, seed + 1)
    write_fasta(os.path.join(d, "m_a1.fa"), a1, "a"); write_fasta(os.path.join(d, "m_a2.fa"), a2, "a")
    s = se_reads(g, 1500, 120, 0.004, seed + 2)
    nmask = rng.random(s.shape) < 0.002
    s[nmask] = ord("N")
    low = rng.random(s.shape[0]) < 0.3
    s[low] = np.char.lower(s[low].view("S1")).view(np.uint8) if low.any() else s[low]
    write_fasta(os.path.join(d, "m_s.fa"), s, "s")
    q1, q2 = pe_reads(g, 2000, 150, 200 + 100, 0.004, seed + 3)
    write_fastq(os.path.join(d, "m_q1.fq"), q1, "q"); write_fastq(os.path.join(d, "m_q2.fq"), q2, "q")
    rq = se_reads(g, 1200, 130, 0.004, seed + 4)
    write_fastq(os.path.join(d, "m_rq.fq"), rq, "z")
    ig = se_reads(g, 500, 100, 0.0, seed + 5)
    write_fasta(os.path.join(d, "m_ig.fa"), ig, "i")
    cfg = os.path.join(d, "multi.cfg")
    j = lambda n: os.path.join(d, n)
    write_config(cfg, 150, [
        {"avg_ins": 500, "files": [("f1", j("m_a1.fa")), ("f2", j("m_a2.fa"))]},
        {"avg_ins": 200, "rd_len_cutoff": 140, "files": [("f", j("m_s.fa")), ("q1", j("m_q1.fq")), ("q2", j("m_q2.fq"))]},
        {"avg_ins": 2000, "reverse_seq": 1, "files": [("q", j("m_rq.fq"))]},
        {"avg_ins": 300, "asm_flags": 2, "files": [("f", j("m_ig.fa"))]},
    ])
    return cfg


def scenario_adversarial(d: str, seed=9, crlf=False, K_hint=31) -> str:
    """Edge cases the reference's readers / counters / edge builder care about: ragged read lengths (incl. shorter than K+1
    and exactly K+1), N's, lower case, '.', a poly-A stretch (counter saturation: links 63, coverage 255), tandem repeats,
    a reverse-complement palindrome (bal_edge = 0 edges), optional CRLF line ends (the '\\r' is dropped, readseq1by1.c:182-200)."""
    rng = np.random.default_rng(seed)
    g = genome(12000, seed)
    unit = g[100:137].copy()
    g[3000:3000 + 37 * 6] = np.tile(unit, 6)                       # tandem repeat
    g[5000:5400] = ord("A")                                         # poly-A
    half = g[7000:7150].copy()
    g[7150:7300] = _COMP[half[::-1]]                                # palindrome: half + revcomp(half)
    nl = b"\r\n" if crlf else b"\n"
    reads = []
    for i in range(3500):
        L = int(rng.choice([K_hint - 3, K_hint, K_hint + 1, K_hint + 2, 60, 75, 100, 100, 100]))
        s = int(rng.integers(0, len(g) - L))
        r = g[s:s + L].copy()
        if rng.random() < 0.5:
            r = _COMP[r[::-1]]
        m = rng.random(L) < 0.004
        r[m] = _ACGT[rng.integers(0, 4, size=int(m.sum()))]
        if rng.random() < 0.05:
            r[int(rng.integers(0, L))] = ord("N")
        if rng.random() < 0.05:
            r[int(rng.integers(0, L))] = ord(".")
        if rng.random() < 0.2:
            r = np.frombuffer(r.tobytes().lower(), dtype=np.uint8).copy()
        reads.append(r.tobytes())
    for i in range(600):                                            # deep poly-A coverage -> saturated counters
        reads.append(b"A" * int(rng.choice([80, 100])))
    order = rng.permutation(len(reads))
    fa, fq = os.path.join(d, "adv.fa"), os.path.join(d, "adv.fq")
    with open(fa, "wb") as f:
        for j in order[: len(order) // 2]:
            f.write(b">r%d" % j + nl + reads[j] + nl)
    with open(fq, "wb") as f:
        for j in order[len(order) // 2:]:
            f.write(b"@r%d" % j + nl + reads[j] + nl + b"+" + nl + b"I" * len(reads[j]) + nl)
    for p in (fa, fq):
        _pad_if_32k(p)
    cfg = os.path.join(d, "adv.cfg")
    write_config(cfg, 100, [{"avg_ins": 200, "files": [("f", fa), ("q", fq)]}])
    return cfg


# ---------------------------------------------------------------- seeded random scenarios (fuzzing the whole stage)
FUZZ_K63 = (13, 15, 17, 21, 31, 33, 45, 61, 63)
FUZZ_K127 = (63, 65, 67, 97, 99, 125, 127)
# max_rd_len values at the edges of k_chop_insert's shared-memory modes (256 reads x ceil(L / 32) words: 48 KB / 96 KB)
FUZZ_LONG_MAX = (768, 769, 1536, 1537)
_IUPAC = b"RYKMSWBDHVrykmswbdhv"
_DROPPED = b"0123456789-* \t"   # bytes the reader drops from a sequence line (not a letter, not '.')


def _fuzz_seq(g, L, err, rng, junk):
    """One read of L bases from g (either strand), substitution errors, then the scenario's unusual bytes (`junk`: subset of
    'N', 'n', '.', 'lower', 'iupac', 'drop')."""
    s = int(rng.integers(0, len(g) - L + 1))
    r = g[s:s + L].copy()
    if rng.random() < 0.5:
        r = _COMP[r[::-1]]
    if err > 0:
        m = rng.random(L) < err
        r[m] = _ACGT[(np.searchsorted(_ACGT, r[m]) + rng.integers(1, 4, size=int(m.sum()))) % 4]
    return _fuzz_bytes(r, rng, junk)


def _fuzz_bytes(r, rng, junk):
    r = r.copy()
    L = len(r)
    if "lower" in junk and rng.random() < 0.2:
        a, b = sorted(int(x) for x in rng.integers(0, L + 1, size=2))
        r[a:b] |= 0x20
    for c, sym in (("N", b"N"), ("n", b"n"), (".", b"."), ("iupac", _IUPAC)):
        if c in junk and rng.random() < 0.08:
            for _ in range(int(rng.integers(1, 4))):
                r[int(rng.integers(0, L))] = sym[int(rng.integers(0, len(sym)))]
    out = r.tobytes()
    if "drop" in junk and rng.random() < 0.1:
        for _ in range(int(rng.integers(1, 6))):
            p = int(rng.integers(0, len(out) + 1))
            out = out[:p] + bytes([_DROPPED[int(rng.integers(0, len(_DROPPED)))]]) * int(rng.integers(1, 3)) + out[p:]
    return out


def _write_fuzz_file(path, seqs, fastq, crlf, tag):
    nl = b"\r\n" if crlf else b"\n"
    with open(path, "wb") as f:
        for i, s in enumerate(seqs):
            if fastq:
                f.write(b"@%s%d" % (tag, i) + nl + s + nl + b"+" + nl + b"I" * len(s) + nl)
            else:
                f.write(b">%s%d" % (tag, i) + nl + s + nl)
    _pad_if_32k(path)


def scenario_fuzz(d: str, seed: int):
    """A random whole-stage scenario, deterministic from `seed`.  Returns (cfg, K, flavour127, P, extra, env): the config, the run
    options (K, -p and the other flags of `pregraph`) and environment variables for the engine that select its insert path, chunk
    size, table and bucket sizes, arena size, flush policy and TMA use (none of them may change the output).

    Drawn independently: one to three libraries of f / q / f1+f2 / q1+q2 files (LF or CRLF per file), reverse_seq, rd_len_cutoff,
    an asm_flags=2 library that must be ignored; ragged read lengths with exactly K+1 and multiples of 32 +-1; about one case in
    six with 700-9000 bp reads and max_rd_len on either side of 768 and 1536 (lines longer than a 2 KB decode tile); max_rd_len
    below the longest lines (truncation); N, n, '.', lower case, IUPAC letters and dropped bytes (digits, '-', '*', space, tab)
    inside sequence lines; poly-A reads (saturated counters); K at the key-width and minimizer-length edges; -p, -a, -d, -R.

    Shapes the reference itself mishandles are never drawn: '>' / '@' inside sequence lines, reads near 64 kbp, file sizes that are
    multiples of 32 KiB, lines longer than its line buffers, and -R with long reads that could cross more than 255 edges (long-read
    cases with -R are error-free)."""
    rng = np.random.default_rng(seed)
    flavour127 = int(rng.random() < 0.35)
    K = int(rng.choice(FUZZ_K127 if flavour127 else FUZZ_K63))
    P = int(rng.choice([1, 2, 3, 5, 8, 16]))
    extra = []
    a = int(rng.choice([0, 1, 2]))
    if a:
        extra += ["-a", str(a)]
    D = int(rng.integers(0, 4))
    if D:
        extra += ["-d", str(D)]
    rflag = bool(rng.random() < 0.5)
    if rflag:
        extra += ["-R"]
    long_reads = bool(rng.random() < 1 / 6)
    if long_reads:
        max_rd_len = int(rng.choice(FUZZ_LONG_MAX)) if rng.random() < 0.6 else int(rng.integers(700, 9001))
    else:
        max_rd_len = max(K + 10, int(rng.choice([100, 128, 150, 160, int(rng.integers(K + 10, 200))])))
    # The reference reads a line into a buffer of max(5000, max_rd_len + 1) bytes and carries a partial record over in one of
    # 4 max_rd_len + 1024 bytes: longer lines overrun them.  16 bytes stay free for dropped bytes and a '\r'.
    line_cap = max_rd_len if max_rd_len > 4900 else min(4900, 2 * max_rd_len + 400)
    if long_reads:
        top = int(rng.integers(max_rd_len, line_cap - 16 + 1)) if line_cap > max_rd_len else max_rd_len - 16   # longest read
        glen = max(20000, 3 * top)
    else:
        top = max_rd_len + int(rng.choice([0, 0, 1, 20, 60]))               # > max_rd_len: truncation
        glen = int(rng.integers(4000, 30000))
    clean = long_reads and rflag   # error-free: a long read then crosses few edges
    err = 0.0 if clean else float(rng.choice([0.0, 0.002, 0.006]))
    junk = {c for c in ("N", "n", ".", "lower", "iupac", "drop") if rng.random() < 0.5}
    if clean:
        junk &= {"lower", "drop"}
    g = genome(glen, seed, repeat=None if clean else (int(rng.integers(50, 400)), int(rng.integers(1, 4))))
    lens_fixed = [K + 1, K + 1, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, max_rd_len - 1, max_rd_len, max_rd_len + 1, top]

    def length():
        if long_reads and rng.random() < 0.7:
            L = int(rng.choice([max_rd_len, max_rd_len + 1, top])) if rng.random() < 0.3 else int(rng.integers(700, top + 1))
        elif rng.random() < 0.4:
            L = int(rng.choice(lens_fixed))
        else:
            L = int(rng.integers(max(K - 3, 13), min(top, 200) + 1))
        return max(13, min(L, top, glen))

    def seqs(n):
        out = []
        for _ in range(n):
            if not clean and rng.random() < 0.03:
                out.append(b"A" * int(rng.integers(K + 1, min(top, 200) + 1)))   # poly-A: links saturate at 63, coverage at 255
            else:
                out.append(_fuzz_seq(g, length(), err, rng, junk))
        return out

    budget = int(rng.integers(150_000, 600_000))   # bases per library
    mean_len = (700 + top) / 2 * 0.7 + 100 * 0.3 if long_reads else min(top, 150)
    libs = []
    n_libs = int(rng.integers(1, 4))
    ins = [int(x) for x in rng.choice(np.arange(150, 3000, 7), size=n_libs + 1, replace=False)]   # distinct: the sort order is defined
    for li in range(n_libs):
        kinds = [k for k in ("f", "q", "f12", "q12") if rng.random() < 0.45] or [str(rng.choice(["f", "q", "f12", "q12"]))]
        files = []
        per = max(40, int(budget / mean_len / len(kinds)))
        for kind in kinds:
            fq = kind.startswith("q")
            tag = b"l%d%s" % (li, kind.encode())
            if kind in ("f", "q"):
                p = os.path.join(d, f"fz{li}_{kind}.{'fq' if fq else 'fa'}")
                _write_fuzz_file(p, seqs(per), fq, bool(rng.random() < 0.3), tag)
                files.append((kind, p))
            else:
                n = max(20, per // 2)
                for m in (1, 2):
                    p = os.path.join(d, f"fz{li}_{kind[0]}{m}.{'fq' if fq else 'fa'}")
                    _write_fuzz_file(p, seqs(n), fq, bool(rng.random() < 0.3), tag)
                    files.append((f"{kind[0]}{m}", p))
        lib = {"avg_ins": ins[li], "reverse_seq": int(rng.random() < 0.25), "asm_flags": int(rng.choice([3, 3, 1])), "files": files}
        if rng.random() < 0.25:
            lib["rd_len_cutoff"] = int(rng.integers(K + 10, max_rd_len + 30))
        libs.append(lib)
    if rng.random() < 0.3:   # a library the pregraph stage must not read (asm_flags=2: scaffolding only)
        p = os.path.join(d, "fz_ignored.fa")
        _write_fuzz_file(p, seqs(50), False, False, b"ig")
        libs.append({"avg_ins": ins[-1], "asm_flags": 2, "files": [("f", p)]})
    cfg = os.path.join(d, "fuzz.cfg")
    write_config(cfg, max_rd_len, libs)

    env = {"PGB200_SKM": str(int(rng.integers(0, 2)))}
    if rng.random() < 0.3:
        env["PGB200_CHUNK_MB"] = "1"
    if rng.random() < 0.25:
        env["PGB200_TABLE_SLOTS"] = str(int(rng.choice([1024, 4096])))
    if rng.random() < 0.3:
        env["PGB200_SKM_BUCKETS"] = str(int(rng.choice([1, 3, 37, 256, 1024])))
    if rng.random() < 0.2:   # a small arena (mid-stream aggregations) that still holds the records of one 1 MB chunk
        env["PGB200_SKM_ARENA_MB"] = "64"
        env["PGB200_CHUNK_MB"] = "1"
    if rng.random() < 0.2:
        env["PGB200_SKM_FLUSH_EVERY"] = str(int(rng.integers(1, 4)))
    if rng.random() < 0.25:
        env["PGB200_NO_TMA"] = "1"
    return cfg, K, flavour127, P, tuple(extra), env


# ---------------------------------------------------------------- vectorised writers for the config-sized cases (millions of reads)
def _names(n: int, tag: bytes, width: int = 9) -> np.ndarray:
    ids = np.arange(n, dtype=np.int64)
    out = np.empty((n, len(tag) + width), dtype=np.uint8)
    out[:, :len(tag)] = np.frombuffer(tag, dtype=np.uint8)
    for d in range(width):
        out[:, len(tag) + width - 1 - d] = (ids // 10 ** d) % 10 + 48
    return out


def write_fastq_fast(path: str, reads: np.ndarray, tag: str = "r") -> None:
    n, L = reads.shape
    nm = _names(n, b"@" + tag.encode())
    rec = np.empty((n, nm.shape[1] + 1 + L + 3 + L + 1), dtype=np.uint8)
    o = nm.shape[1]
    rec[:, :o] = nm
    rec[:, o] = 10
    rec[:, o + 1:o + 1 + L] = reads
    rec[:, o + 1 + L] = 10
    rec[:, o + 2 + L] = ord("+")
    rec[:, o + 3 + L] = 10
    rec[:, o + 4 + L:o + 4 + 2 * L] = ord("I")
    rec[:, o + 4 + 2 * L] = 10
    rec.tofile(path)
    _pad_if_32k(path)


def write_fasta_fast(path: str, reads: np.ndarray, tag: str = "r") -> None:
    n, L = reads.shape
    nm = _names(n, b">" + tag.encode())
    rec = np.empty((n, nm.shape[1] + 1 + L + 1), dtype=np.uint8)
    o = nm.shape[1]
    rec[:, :o] = nm
    rec[:, o] = 10
    rec[:, o + 1:o + 1 + L] = reads
    rec[:, o + 1 + L] = 10
    rec.tofile(path)
    _pad_if_32k(path)


def config_c1(d: str, genome_len=4_600_000, coverage=30, seed=1) -> str:
    """BASELINE.json configs[0]: E. coli-sized genome, one library, 100 bp SE single-line FASTA, err 0.5 %, K=31 (SURVEY 8d C1)."""
    g = genome(genome_len, seed)
    n = genome_len * coverage // 100
    write_fasta_fast(os.path.join(d, "c1.fa"), se_reads(g, n, 100, 0.005, seed + 100), "e")
    cfg = os.path.join(d, "c1.cfg")
    write_config(cfg, 100, [{"avg_ins": 200, "files": [("f", os.path.join(d, "c1.fa"))]}])
    return cfg


def config_c2(d: str, genome_len=10_000_000, coverage=30, seed=42) -> str:
    """BASELINE.json configs[1] shape at a size the reference finishes in about a minute: 150 bp PE FASTQ q1/q2, insert 300, err 0.1 %."""
    g = genome(genome_len, seed)
    r1, r2 = pe_reads(g, genome_len * coverage // 300, 150, 300, 0.001, seed + 1)
    write_fastq_fast(os.path.join(d, "c2_1.fq"), r1, "p")
    write_fastq_fast(os.path.join(d, "c2_2.fq"), r2, "p")
    cfg = os.path.join(d, "c2.cfg")
    write_config(cfg, 150, [{"avg_ins": 300, "files": [("q1", os.path.join(d, "c2_1.fq")), ("q2", os.path.join(d, "c2_2.fq"))]}])
    return cfg


def config_c5(d: str, genome_len=20_000_000, seed=5) -> str:
    """BASELINE.json configs[4] (SURVEY 8d C5): three libraries -- rank1 avg_ins=200 q1/q2 150 bp; rank2 avg_ins=500 f1/f2 100 bp
    FASTA; rank3 avg_ins=2000 reverse_seq=1 asm_flags=3 f= + q= SE -- about 30x in total, planted repeats so the graph branches."""
    g = genome(genome_len, seed, repeat=(3000, 6))
    j = lambda n: os.path.join(d, n)
    a1, a2 = pe_reads(g, genome_len * 15 // 300, 150, 200 + 100, 0.002, seed + 1)
    write_fastq_fast(j("c5_a1.fq"), a1, "a"); write_fastq_fast(j("c5_a2.fq"), a2, "a")
    b1, b2 = pe_reads(g, genome_len * 10 // 200, 100, 500, 0.002, seed + 2)
    write_fasta_fast(j("c5_b1.fa"), b1, "b"); write_fasta_fast(j("c5_b2.fa"), b2, "b")
    write_fasta_fast(j("c5_c.fa"), se_reads(g, genome_len * 3 // 100, 100, 0.002, seed + 3), "c")
    write_fastq_fast(j("c5_d.fq"), se_reads(g, genome_len * 2 // 120, 120, 0.002, seed + 4), "d")
    cfg = j("c5.cfg")
    write_config(cfg, 150, [
        {"avg_ins": 200, "files": [("q1", j("c5_a1.fq")), ("q2", j("c5_a2.fq"))]},
        {"avg_ins": 500, "files": [("f1", j("c5_b1.fa")), ("f2", j("c5_b2.fa"))]},
        {"avg_ins": 2000, "reverse_seq": 1, "asm_flags": 3, "files": [("f", j("c5_c.fa")), ("q", j("c5_d.fq"))]},
    ])
    return cfg
