#!/usr/bin/env python
"""bench.py -- distinct k-mers hashed / second at K=63 (pregraph pass 1) on N B200s, next to the reference's CPU path.

One "step" = one complete pass 1 (prlRead2HashTable equivalent: FASTQ text -> 2-bit reads -> canonical k-mers ->
table insert/count -> delow/mark-linear/kmerFreq sweeps) over the synthetic read set of BASELINE.json configs[1]
(100 Mbp genome, 30x, 150 bp PE FASTQ, K=63), including clearing the table from the previous step.

  value  : whole-job distinct k-mers / s with the FASTQ text already resident in HBM (device pointers through the C-ABI)
  e2e    : the same metric through the C-ABI with HOST (pinned) text buffers: H2D copies inside the timed region, plus a
           D2H read of the coverage histogram / statistics every step.  N=1: the engine inserts host text per instance (that hides
           under the copies; the aggregation cannot finish before the last chunk); N>1: the same aggregated kernels as `value`.
  roofline: the insert (k_skm_count/scatter + k_skm_apply, soapdenovo2_b200/csrc/skm.cu), HBM bound by SURVEY.md 8(d): algorithmic
           bytes = 64 B per k-mer instance (one 32 B slot sector read + written back); time = CUDA events recorded by the engine on
           its own stream around those launches.  The aggregated insert moves far fewer bytes than that (one table update per
           DISTINCT k-mer) and is issue-bound: `traffic` / `issue_slots_pct` are the measured ncu figures (profiles/), `frac` is the
           algorithmic-equivalent fraction so that rounds stay comparable.
  cpu_baseline: the UNMODIFIED reference binary (oracle/_ref/SOAPdenovo-63mer pregraph, built from /root/reference by
           oracle/Makefile) timed on this box's host cores up to its "node(s) allocated" line, on a bounded sample
  --impl reference: the same binary on the FULL workload files (written to local scratch), run once per thread count
N>1 (torchrun): strong scaling, the same read set; chunk i is decoded and partitioned by rank i % N, every super-k-mer record is
stored straight into the arena of the GPU that owns its minimizer bucket (NVLink peer stores from the partition kernel), each GPU
aggregates its buckets.  torch.distributed carries the IPC handles once and one barrier per step.  See DESIGN.md (e).
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 63
RD_LEN = 150
INSERT = 300
ERR = 0.001
NAME_W = 10   # "@" + 10 chars
REC_BYTES = 1 + NAME_W + 1 + RD_LEN + 1 + 2 + RD_LEN + 1
DIGESTS = os.path.join(ROOT, "tests", "golden", "bench_digests.json")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--genome", type=int, default=int(os.environ.get("PGB200_BENCH_GENOME", 100_000_000)))
    ap.add_argument("--coverage", type=float, default=30.0)
    ap.add_argument("--chunk-reads", type=int, default=0, help="reads per fed chunk (0: 1 M at N=1, sized so that every rank gets whole chunks at N>1)")
    ap.add_argument("--sample-genome", type=int, default=2_500_000, help="cpu_baseline sample: sub-genome size at the same coverage")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--K", type=int, default=63, help="63 (headline, 63-mer flavour) or e.g. 127 (127-mer flavour, 256-bit keys; configs[3] shape)")
    ap.add_argument("--scale", default="strong", choices=["strong", "weak"],
                    help="N>1: strong = the same read set split over the ranks (default); weak = every rank brings its own --genome/N ... see --weak-genome")
    ap.add_argument("--weak-genome", type=int, default=0, help="weak scaling / configs[2]: TOTAL genome size; every rank generates and feeds 1/N of the reads")
    ap.add_argument("--write-digest", action="store_true", help="record this run's distinct count + histogram hash as the golden digest of the workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64): coverage_hist "
                         "(256 counts of distinct k-mers by coverage, 255 = saturated) and pass1_counts (records, reads kept, k-mer "
                         "instances, distinct k-mers, linear nodes marked, k-mers removed)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ----------------------------------------------------------------------------------------------- synthetic reads (torch = plumbing)
def gen_genome(torch, dev, genome_len, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    out = torch.empty(genome_len, dtype=torch.uint8, device=dev)
    PIECE = 1 << 28
    for o in range(0, genome_len, PIECE):
        n = min(PIECE, genome_len - o)
        out[o:o + n] = acgt[torch.randint(0, 4, (n,), device=dev, generator=g)]
    return out, g


def gen_reads(torch, dev, genome, n_pairs, g, id_base=0):
    """Two uint8 device tensors holding FASTQ text (fixed 316-byte records) for mates 1 and 2, sampled from `genome`."""
    genome_len = genome.numel()
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    comp = torch.zeros(256, dtype=torch.uint8, device=dev)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    ar = torch.arange(RD_LEN, device=dev)
    BATCH = 2_000_000
    bufs = [torch.empty((n_pairs, REC_BYTES), dtype=torch.uint8, device=dev) for _ in range(2)]
    lut = torch.tensor([0, 1, 3, 2], device=dev)    # base code -> index in "ACGT"
    for b0 in range(0, n_pairs, BATCH):
        nb = min(BATCH, n_pairs - b0)
        starts = torch.randint(0, genome_len - INSERT + 1, (nb,), device=dev, generator=g)
        r1 = genome[starts[:, None] + ar[None, :]]
        r2 = comp[genome[(starts + INSERT - RD_LEN)[:, None] + ar[None, :]].long()].flip(1)
        flip = torch.rand(nb, device=dev, generator=g) < 0.5
        m1 = torch.where(flip[:, None], r2, r1)
        m2 = torch.where(flip[:, None], r1, r2)
        for mate, reads in enumerate((m1, m2)):
            errm = torch.rand(reads.shape, device=dev, generator=g) < ERR
            code = ((reads >> 1) & 3).long()               # A(0x41)->0 C(0x43)->1 T(0x54)->2 G(0x47)->3
            sub = acgt[(lut[code] + torch.randint(1, 4, reads.shape, device=dev, generator=g)) % 4]   # always a different letter
            reads = torch.where(errm, sub, reads)
            rec = bufs[mate][b0:b0 + nb]
            rec[:, 0] = ord("@")
            ids = torch.arange(id_base + b0, id_base + b0 + nb, device=dev)
            rec[:, 1] = ord("r")
            for d in range(NAME_W - 1):
                rec[:, 1 + NAME_W - 1 - d] = ((ids // (10 ** d)) % 10 + 48).to(torch.uint8)
            o = 1 + NAME_W
            rec[:, o] = 10
            rec[:, o + 1:o + 1 + RD_LEN] = reads
            rec[:, o + 1 + RD_LEN] = 10
            rec[:, o + 2 + RD_LEN] = ord("+")
            rec[:, o + 3 + RD_LEN] = 10
            rec[:, o + 4 + RD_LEN:o + 4 + 2 * RD_LEN] = ord("I")
            rec[:, o + 4 + 2 * RD_LEN] = 10
    return bufs[0].reshape(-1), bufs[1].reshape(-1)


def gen_pe_fastq_gpu(torch, dev, genome_len, n_pairs, seed):
    """The configs[1] recipe: genome and reads from one seeded generator (kept bit-compatible with round 1's workload)."""
    genome, g = gen_genome(torch, dev, genome_len, seed)
    t = gen_reads(torch, dev, genome, n_pairs, g)
    del genome
    return t


# ----------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.stop, self.index = [], False, index
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------------- reference CPU arm
def write_read_files(torch, workdir, genome_len, coverage, seed, tag):
    n_pairs = int(genome_len * coverage / (2 * RD_LEN))
    if n_pairs % 8192 == 0:
        n_pairs -= 1   # file size must not be a multiple of 32768 B (reference AIO reader quirk, SURVEY.md A.9)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    t1, t2 = gen_pe_fastq_gpu(torch, dev, genome_len, n_pairs, seed)
    p1, p2 = os.path.join(workdir, f"{tag}_1.fq"), os.path.join(workdir, f"{tag}_2.fq")
    for t, p in ((t1, p1), (t2, p2)):
        with open(p, "wb") as f:
            PIECE = 1 << 28
            for o in range(0, t.numel(), PIECE):
                f.write(t[o:o + PIECE].cpu().numpy().tobytes())
    del t1, t2
    cfg = os.path.join(workdir, f"{tag}.cfg")
    with open(cfg, "w") as f:
        f.write(f"max_rd_len={RD_LEN}\n[LIB]\navg_ins={INSERT}\nreverse_seq=0\nasm_flags=3\nrank=1\nq1={p1}\nq2={p2}\n")
    return cfg, n_pairs


def time_reference_pass1(cfg, workdir, threads, tag, init_g=2):
    """Run the unmodified reference pregraph and time it from launch to its 'node(s) allocated' stderr line (= pass 1)."""
    ref = os.path.join(ROOT, "oracle", "_ref", "SOAPdenovo-63mer" if K <= 63 else "SOAPdenovo-127mer")
    kind = "reference"
    if not os.path.exists(ref):
        ref, kind = os.path.join(ROOT, "oracle", "pregraph_model_63" if K <= 63 else "pregraph_model_127"), "port"
        if not os.path.exists(ref):
            subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "model"], check=True)
    if kind == "reference":
        cmd = [ref, "pregraph", "-s", cfg, "-K", str(K), "-p", str(threads), "-a", str(init_g), "-o", os.path.join(workdir, tag)]
    else:
        cmd, threads = [ref, "-1", "-s", cfg, "-K", str(K), "-p", "8", "-a", str(init_g), "-o", os.path.join(workdir, tag)], 1
    t0 = time.perf_counter()
    p = subprocess.Popen(cmd, stderr=subprocess.PIPE, stdout=subprocess.DEVNULL, text=True)
    distinct, t_done = None, None
    for line in p.stderr:
        if "node(s) allocated" in line:
            distinct = int(line.split()[0])
            t_done = time.perf_counter()   # printed right after the last batch was inserted (prlHashReads.c:717)
            if kind == "reference":
                p.kill()   # the exact child we started; later phases are not part of the metric
                break
    p.wait()
    if distinct is None:
        raise RuntimeError("reference run produced no 'node(s) allocated' line")
    return distinct, t_done - t0, kind, threads


def thread_choices():
    """BASELINE.md: the layout value -p 8, and best-of {cores/2, cores} (the reference degrades when -p >= cores); -p <= 255."""
    cores = os.cpu_count() or 1
    out = []
    for x in (8, min(cores // 2, 64), min(cores, 128)):
        x = max(1, min(x, 255))
        if x not in out:
            out.append(x)
    return out


def reference_arm(args, torch, workdir, workload):
    """The reference's own pthreads pass 1 on the FULL workload (same files the GPU arm's read set would make), run ONCE per thread
    count; --steps / --warmup apply to the GPU arm only (a run takes minutes)."""
    cfg, n_pairs = write_read_files(torch, workdir, args.genome, args.coverage, 42, "refarm")
    init_g = max(2, int(args.genome * 2.3 * 24 * 1.4 / (1 << 30)) + 1)   # -a: static tables large enough (prlHashReads.c:372-385)
    runs, budget, t_start = [], float(os.environ.get("PGB200_REF_BUDGET_S", "300")), time.perf_counter()
    for thr in thread_choices():
        if runs and time.perf_counter() - t_start + runs[-1]["seconds"] > budget:
            break
        d, secs, kind, used = time_reference_pass1(cfg, workdir, thr, "refarm", init_g)
        runs.append({"threads": used, "seconds": secs, "distinct": d, "value": d / secs})
    best = max(runs, key=lambda r: r["value"])
    reads = 2 * n_pairs
    sample = (f"FULL workload: {reads} reads, {reads*(RD_LEN-K+1)} k-mer instances, {best['distinct']} distinct; pass 1 only (launch -> 'node(s) allocated'); "
              f"one run per thread count {[r['threads'] for r in runs]}, best reported; --steps/--warmup apply to the GPU arm")
    for p in (os.path.join(workdir, "refarm_1.fq"), os.path.join(workdir, "refarm_2.fq")):
        try:
            os.remove(p)
        except OSError:
            pass
    print(json.dumps({"impl": "reference", "metric": f"distinct k-mers hashed/sec at K={K}", "value": best["value"], "unit": "distinct k-mers/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": best["seconds"] * 1e3, "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                      "config": {"workload": workload, "reads": reads, "kmer_instances": reads * (RD_LEN - K + 1), "distinct_kmers": best["distinct"], "runs": runs,
                                 "host_cores_available": os.cpu_count()},
                      "cpu_baseline": {"value": best["value"], "unit": "distinct k-mers/s", "cores": best["threads"], "kind": kind, "sample": sample},
                      "e2e": {"value": best["value"], "unit": "distinct k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def hist_digest(hist):
    return hashlib.sha256(",".join(str(int(x)) for x in hist).encode()).hexdigest()


def main():
    args = parse_args()
    global K
    K = args.K
    import torch
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    # scratch for the reference arm's read files: a private temporary directory unless PGB200_BENCH_DIR names one
    own_workdir = "PGB200_BENCH_DIR" not in os.environ
    workdir = tempfile.mkdtemp(prefix="pgb200_bench_") if own_workdir else os.environ["PGB200_BENCH_DIR"]
    os.makedirs(workdir, exist_ok=True)
    try:
        run(args, torch, workdir, rank, world, local_rank)
    finally:
        if own_workdir:
            shutil.rmtree(workdir, ignore_errors=True)


def run(args, torch, workdir, rank, world, local_rank):
    weak = args.scale == "weak" or args.weak_genome > 0
    total_genome = args.weak_genome if args.weak_genome > 0 else (args.genome * world if weak else args.genome)
    workload = f"synthetic {total_genome/1e6:g} Mbp genome, {args.coverage:g}x {RD_LEN} bp PE FASTQ (insert {INSERT}, {ERR*100:g}% subst.), K={K}"

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, torch, workdir, workload)
        return

    from soapdenovo2_b200 import api
    from soapdenovo2_b200 import dist as pdist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- workload
    n_pairs_total = int(total_genome * args.coverage / (2 * RD_LEN))
    if weak:
        # every rank samples its own reads (own seed) from the SAME genome and feeds all of them; ordinals are global
        n_pairs = n_pairs_total // world
        genome, _ = gen_genome(torch, dev, total_genome, 42)
        g = torch.Generator(device=dev)
        g.manual_seed(1000 + rank)
        t1, t2 = gen_reads(torch, dev, genome, n_pairs, g, id_base=rank * n_pairs)
        del genome
        pair_base = rank * n_pairs
    else:
        # every rank generates the SAME read set (same seed) and feeds chunk i iff i % N == rank
        n_pairs = n_pairs_total
        t1, t2 = gen_pe_fastq_gpu(torch, dev, total_genome, n_pairs, seed=42)
        pair_base = 0
    torch.cuda.synchronize()
    torch.cuda.empty_cache()   # hand the generator's temporaries back: the engine allocates with cudaMalloc
    chunk_reads = args.chunk_reads
    if not chunk_reads:
        if weak:
            per_mate = max(1, -(-n_pairs // 1_250_000))
            per_mate = max(1, min(per_mate, 120 // (2 * world)))   # segments per epoch: SKM_MAX_SEGS = 128 over all senders
            chunk_reads = -(-n_pairs // per_mate)
        else:
            per_rank = max(1, round(10 / world))                   # chunks per mate and rank: 10 x 1 M reads at N=1
            chunk_reads = -(-n_pairs // (world * per_rank))
    # genome + the k-mers the substitutions create: 0.001 x coverage errors per genome base, each covered by ~36 (K=63) / ~19 (K=127:
    # only 24 k-mers per 150 bp read) k-mers of its read -- measured at 30x: 2.07 x and 1.56 x the genome size; 10 % head room
    est_distinct = int(total_genome * 1.1 * (1.0 + 0.001 * args.coverage * (36 if K <= 63 else 19))) + 1_000_000
    slots = 1 << max(20, (int(est_distinct / world * 2.2 * float(os.environ.get('PGB200_BENCH_SLOTS_MULT', '1')))).bit_length())
    eng = api.PregraphEngine(K=K, P=8, initG=0, flavour127=int(K > 63), max_rd_len=RD_LEN, device=local_rank, table_slots=slots, world=world, rank=rank,
                             verbose=int(os.environ.get("PGB200_VERBOSE", "0")))
    def make_work(reads_per_chunk):
        out = []   # (mate, byte offset, nbytes, ordinal base)
        for mate, t in enumerate((t1, t2)):
            off = 0
            while off < t.numel():
                n = min(reads_per_chunk * REC_BYTES, t.numel() - off)
                out.append((mate, off, n, (pair_base + off // REC_BYTES) * 2 + mate))
                off += n
        return out

    work = make_work(chunk_reads)
    mine = list(range(len(work))) if weak else pdist.deal(len(work), world, rank)
    # One GPU, text already in HBM: nothing has to overlap with a copy, so the feed uses fewer, larger chunks (4 M reads = 0.63 GB of
    # text per feed_text call; every kernel of the front end then runs 6 times per step instead of 20: 64.8 vs 67.5 ms per step on the
    # same box).  The host-buffer pass (e2e) keeps 1 M-read chunks: there the chunk is the unit of the copy / compute overlap.
    chunk_reads_dev = 4_000_000 if (world == 1 and not weak and not args.chunk_reads) else chunk_reads
    work_dev = make_work(chunk_reads_dev) if chunk_reads_dev != chunk_reads else work
    mine_dev = list(range(len(work_dev))) if work_dev is not work else mine
    total_instances = 2 * n_pairs * (world if weak else 1) * (RD_LEN - K + 1)
    xchg = None
    if world > 1:
        # arena: this rank's share of the job's records (about one record per 15.9 k-mers at K=63, 10 at K=127; 40 % head room),
        # double-buffered inside the engine
        per_rec = 15.0 if K <= 63 else 9.0
        xchg = pdist.RecordExchange(eng, dist, cap_records=int(float(os.environ.get("PGB200_BENCH_ARENA_FACTOR", "1.4")) * total_instances / per_rec / world) + (1 << 20))

    timeline = [0.0] * 5 if os.environ.get("PGB200_BENCH_TIMELINE") else None   # host seconds: reset, feeds, epoch end, finish, sweeps

    def one_step(bufs, on_device):
        """bufs: per mate a device tensor, or {work index: (host pointer, nbytes)} for this rank's chunks."""
        tl = [time.perf_counter()]
        eng.reset_pass1()
        tl.append(time.perf_counter())
        for i in (mine_dev if on_device else mine):
            mate, off, n, ob = (work_dev if on_device else work)[i]
            if on_device:
                eng.feed_text(bufs[mate].data_ptr() + off, n, on_device=True, fastq=True, ord_base=ob, ord_stride=2)
            else:
                eng.feed_text(bufs[i][0], bufs[i][1], on_device=False, fastq=True, ord_base=ob, ord_stride=2)
        tl.append(time.perf_counter())
        if xchg:
            xchg.end_epoch()
        tl.append(time.perf_counter())
        st = eng.finish_pass1()
        tl.append(time.perf_counter())
        hist, lin, rem = eng.sweeps()   # D2H of the histogram + counters: the step's result
        tl.append(time.perf_counter())
        if timeline is not None:
            for j in range(5):
                timeline[j] += tl[j + 1] - tl[j]
        return st, hist, lin, rem

    def timed(bufs, on_device, steps, warmup):
        for _ in range(warmup):
            one_step(bufs, on_device)
        if timeline is not None:
            for j in range(5):
                timeline[j] = 0.0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ins_ms = app_ms = dec_ms = 0.0
        launches = 0
        e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            st, hist, lin, rem = one_step(bufs, on_device)
            ins_ms += st.ms_insert
            app_ms += st.ms_apply
            dec_ms += st.ms_decode
            launches += st.launches + 3
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        if timeline is not None and rank == 0:
            sys.stderr.write("[bench] host timeline, ms per timed step: reset %.2f, feeds %.2f, epoch end %.2f, finish_pass1 %.2f, sweeps %.2f\n"
                             % tuple(1e3 * v / steps for v in timeline))
            for j in range(5):
                timeline[j] = 0.0
        dev_ms = e0.elapsed_time(e1)
        ms = max(dev_ms, 0.0) if dev_ms > 0 else wall * 1e3
        if world > 1:
            tt = torch.tensor([ms, float(st.distinct), float(st.instances), ins_ms, app_ms, dec_ms], device=dev, dtype=torch.float64)
            mx = tt.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = tt.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            ms, distinct, instances, ins_ms, app_ms, dec_ms = mx[0].item(), sm[1].item(), sm[2].item(), mx[3].item(), mx[4].item(), mx[5].item()
            hh = torch.tensor(hist, device=dev, dtype=torch.int64); dist.all_reduce(hh); hist = hh.tolist()
            cc = torch.tensor([st.records, st.reads_kept, lin, rem], device=dev, dtype=torch.int64); dist.all_reduce(cc)
            records, reads_kept, lin, rem = cc.tolist()
        else:
            distinct, instances, records, reads_kept = st.distinct, st.instances, st.records, st.reads_kept
        counts = [records, reads_kept, int(instances), int(distinct), lin, rem]   # the job's, as --dump-outputs writes them
        return {"ms": ms / steps, "distinct": int(distinct), "instances": int(instances), "ins_ms": ins_ms / steps, "app_ms": app_ms / steps,
                "dec_ms": dec_ms / steps, "launches": launches // steps, "hist": hist, "counts": counts, "st": st}

    with ClockSampler(local_rank) as cs:
        r = timed((t1, t2), True, args.steps, args.warmup)
    clocks = cs.summary()
    value = r["distinct"] / (r["ms"] / 1e3)

    # ---- parity guard inside the bench: the all-reduced result must equal the recorded single-GPU digest of this workload
    key = f"G{total_genome}_c{args.coverage:g}_K{K}_{'weak%d' % world if weak else 'strong'}"
    digest = {"distinct": r["distinct"], "instances": r["instances"], "hist_sha256": hist_digest(r["hist"])}
    known = {}
    try:
        known = json.load(open(DIGESTS))
    except Exception:
        pass
    parity = "no golden digest for this workload"
    if key in known:
        if {k: known[key][k] for k in digest} != digest:
            raise SystemExit(f"bench.py: PARITY FAILURE at N={world}: {digest} != golden {known[key]} ({DIGESTS})")
        parity = f"distinct count, instance count and coverage histogram equal the golden single-GPU digest ({os.path.relpath(DIGESTS, ROOT)}:{key})"
    if args.write_digest and rank == 0:
        known[key] = dict(digest, n_gpus=world)
        json.dump(known, open(DIGESTS, "w"), indent=1, sort_keys=True)
    assert r["instances"] == total_instances, (r["instances"], total_instances)
    assert sum(r["hist"]) == r["distinct"]
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "coverage_hist.npy"), np.asarray(r["hist"], dtype=np.float64))
        np.save(os.path.join(args.dump_outputs, "pass1_counts.npy"), np.asarray(r["counts"], dtype=np.float64))

    e2e = None
    if not args.no_e2e:
        # the same step from HOST pinned buffers through the C-ABI (H2D inside), result read back every step
        import ctypes
        lib = api.load()
        hb, h2d = {}, 0
        for i in mine:
            mate, off, n, ob = work[i]
            p = lib.pgb200_host_alloc(n)
            arr = (ctypes.c_ubyte * n).from_address(p)
            torch.frombuffer(arr, dtype=torch.uint8).copy_((t1, t2)[mate][off:off + n].cpu())
            hb[i] = (p, n)
            h2d += n
        re_ = timed(hb, False, max(1, args.steps), 1)
        assert re_["distinct"] == r["distinct"] and re_["hist"] == r["hist"], "e2e result differs from the device-resident result"
        if world > 1:
            tt = torch.tensor([float(h2d)], device=dev, dtype=torch.float64); dist.all_reduce(tt); h2d = int(tt.item())
        e2e = {"value": re_["distinct"] / (re_["ms"] / 1e3), "unit": "distinct k-mers/s", "ms_per_step": re_["ms"], "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": 256 * 8 + 18 * 8 * (len(work) + 4)}
        for p, _ in hb.values():
            lib.pgb200_host_free(p)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    inst_per_rank = r["instances"] / world
    slot_bytes = 64 if K <= 63 else 128   # one slot sector read + written back (SURVEY 8d)
    ins_ms = r["ins_ms"]
    achieved = inst_per_rank * slot_bytes / (ins_ms / 1e3) / 1e9 if ins_ms > 0 else None
    prof = {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_skm_apply_traffic.json")))
    except Exception:
        pass
    nw = 2 if K <= 63 else 4
    traffic = prof.get("dram_bytes_per_step") if K == 63 and world == 1 and total_genome == 100_000_000 else None
    roof = {"kernel": f"k_skm_apply<{nw}> (+ k_skm_count / k_skm_scatter<{nw}>: the aggregated insert)", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak if achieved else None, "traffic": traffic,
            "frac_kind": "algorithmic-equivalent: SURVEY 8(d)'s 64 B per k-mer instance / the insert launches' time; the aggregated kernel moves fewer bytes and is issue-bound",
            "issue_slots_pct": prof.get("issue_slots_pct") if traffic else None,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
            "algorithmic_bytes_per_instance": slot_bytes, "instances_per_step_per_gpu": inst_per_rank, "insert_kernel_ms_per_step": ins_ms,
            "apply_kernel_ms_per_step": r["app_ms"], "apply_only_frac": (inst_per_rank * slot_bytes / (r["app_ms"] / 1e3) / 1e9 / peak) if r["app_ms"] > 0 else None,
            "decode_stream_ms_per_step": r["dec_ms"], "decode_note": "elapsed on the decode stream, which runs concurrently with the insert stream (not a sum of kernel times; see profiles/ for those)"}

    cpu_b = None
    if not args.no_cpu_baseline:
        try:
            cfg, sp = write_read_files(torch, workdir, args.sample_genome, args.coverage, 4242, "cpub")
            runs = []
            for thr in thread_choices()[:2]:
                d, secs, kind, used = time_reference_pass1(cfg, workdir, thr, "cpub")
                runs.append({"threads": used, "seconds": secs, "value": d / secs})
            best = max(runs, key=lambda x: x["value"])
            cpu_b = {"value": best["value"], "unit": "distinct k-mers/s", "cores": best["threads"], "kind": kind, "host_cores_available": os.cpu_count(), "runs": runs,
                     "sample": f"{args.sample_genome/1e6:g} Mbp sub-genome at {args.coverage:g}x ({2*sp} reads, {2*sp*(RD_LEN-K+1)} instances, {d} distinct), pass 1 only, best of the listed thread counts; the full-size run is `--impl reference`"}
        except Exception as ex:   # keep the GPU line even if the CPU leg fails
            cpu_b = {"value": None, "error": str(ex)[:200]}

    st = r["st"]
    print(json.dumps({
        "metric": f"distinct k-mers hashed/sec at K={K}", "value": value, "unit": "distinct k-mers/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": workload, "reads": 2 * n_pairs_total, "kmer_instances": r["instances"], "distinct_kmers": r["distinct"],
                   "instances_per_s": r["instances"] / (r["ms"] / 1e3), "table_slots_per_gpu": int(st.table_slots), "chunk_reads": chunk_reads_dev, "chunks": len(work_dev), "e2e_chunk_reads": chunk_reads,
                   "parallelism": (f"minimizer buckets owned in {world} contiguous ranges; chunk i decoded + partitioned by rank i % {world}; super-k-mer records stored straight into the "
                                   f"owner GPU's arena by the partition kernel (NVLink peer stores over CUDA IPC mappings, no library collective on the data path); one barrier per step"
                                   if world > 1 else "1 GPU"),
                   "insert_mode": ("aggregated pass 1 (super-k-mer records, one table update per distinct k-mer) for value AND e2e" if world > 1 or os.environ.get("PGB200_SKM") == "1"
                                   else ("PGB200_SKM=0: per-instance inserts" if os.environ.get("PGB200_SKM") == "0"
                                         else "value (text resident in HBM): aggregated pass 1, one table update per distinct k-mer; e2e (text over PCIe): per-instance inserts, hidden under the H2D copies -- see DESIGN.md section 5")),
                   "parity": parity, "digest": digest,
                   "l2_policy": f"inputs ({(t1.numel()+t2.numel())/1e9:.1f} GB text per rank, {st.table_slots*32*(2 if K>63 else 1)/1e9:.1f} GB table) are far larger than the 126 MB L2; the table is cleared every step"},
        "e2e": e2e, "gpu_launches": int(r["launches"]), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu_b}))


if __name__ == "__main__":
    main()
