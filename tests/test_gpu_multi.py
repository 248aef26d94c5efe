"""2-GPU parity (run with gpurun --gpus 2): pass 1 with the minimizer buckets owned by two GPUs and every super-k-mer record
stored straight into its owner's arena (NVLink peer stores over CUDA IPC, no collective on the data path) must give the same
coverage histogram, distinct count and per-k-mer entries as the single-GPU oracle -- across processes (the bench's layout) and
inside one process (the CLI's layout: one engine per GPU, peer access)."""
import os

import pytest
import torch

from soapdenovo2_b200 import api, synth
from tests import util

pytestmark = pytest.mark.gpu


def _work_items(d):
    """every file split into 3 record-aligned chunks: (text, ordinal base)"""
    work = []
    for fn, mate in ((os.path.join(d, "pe_1.fq"), 0), (os.path.join(d, "pe_2.fq"), 1)):
        lines = open(fn, "rb").read().split(b"\n")[:-1]
        recs = [b"\n".join(lines[i:i + 4]) + b"\n" for i in range(0, len(lines), 4)]
        per = (len(recs) + 2) // 3
        for c in range(3):
            work.append((b"".join(recs[c * per:(c + 1) * per]), (c * per) * 2 + mate))
    return work


def _worker(rank, world, port, d, out, epochs):
    import torch.distributed as dist
    from soapdenovo2_b200 import dist as pdist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    eng = api.PregraphEngine(K=63, P=8, initG=1, max_rd_len=150, device=rank, world=world, rank=rank)
    xchg = pdist.RecordExchange(eng, dist, cap_records=1 << 20)
    work = _work_items(d)
    rounds = [work[i:i + world] for i in range(0, len(work), world)]
    for ri, rnd in enumerate(rounds):
        if rank < len(rnd):
            eng.feed_text(rnd[rank][0], fastq=True, ord_base=rnd[rank][1], ord_stride=2)
        if epochs == "many" or ri == len(rounds) - 1:
            xchg.end_epoch()          # "many": one exchange epoch per round (alternating arena halves)
    st = eng.finish_pass1()
    hist, lin, rem = eng.sweeps()
    h = torch.tensor(hist, device=dev, dtype=torch.int64)
    dist.all_reduce(h)
    cnt = torch.tensor([st.distinct, st.instances], device=dev, dtype=torch.int64)
    dist.all_reduce(cnt)
    eng.build_layout()      # per-shard layout: records are only compared as a SET below
    out[rank] = (h.tolist(), cnt.tolist(), eng.dump_nodes())
    dist.barrier()
    eng.close()
    dist.destroy_process_group()


def _oracle(d):
    util.build_oracle()
    cfg = synth.scenario_pe_fastq(d)
    mod, dump = os.path.join(d, "mod"), os.path.join(d, "mod.table")
    util.run_model(util.MODEL63, cfg, mod, 63, 8, ("-1", "-T", dump, "-a", "1"))
    return open(mod + ".kmerFreq", "rb").read(), open(dump, "rb").read()


def _check(out, kmerfreq, want):
    hist, cnt, _ = out[0]
    assert api.kmerfreq_text(hist) == kmerfreq
    assert cnt[0] * 26 == len(want) and cnt[1] == 12000 * 88
    recs = lambda b: {b[i:i + 26] for i in range(0, len(b), 26)}
    # every k-mer lives on exactly one GPU with exactly the oracle's counters (linear/deleted flags included)
    assert recs(out[0][2]) | recs(out[1][2]) == recs(want)
    assert not (recs(out[0][2]) & recs(out[1][2]))
    assert len(out[0][2]) > 0 and len(out[1][2]) > 0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (gpurun --gpus 2)")
@pytest.mark.parametrize("epochs", ["one", "many"])
def test_two_gpu_two_processes(tmp_path, epochs):
    import torch.multiprocessing as mp
    d = str(tmp_path)
    kmerfreq, want = _oracle(d)
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(2, 29541 if epochs == "one" else 29543, d, out, epochs), nprocs=2, join=True)
    _check(out, kmerfreq, want)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (gpurun --gpus 2)")
def test_two_gpu_one_process(tmp_path):
    """Both engines in this process (what the multi-GPU CLI does): arenas exchanged as plain pointers, peer access enabled."""
    d = str(tmp_path)
    kmerfreq, want = _oracle(d)
    engs = [api.PregraphEngine(K=63, P=8, initG=1, max_rd_len=150, device=r, world=2, rank=r) for r in range(2)]
    for e in engs:
        e.xchg_setup(1 << 20)
    for r, e in enumerate(engs):
        e.xchg_import_ptr(1 - r, 1 - r, engs[1 - r].xchg_base())
    for i, (text, ob) in enumerate(_work_items(d)):
        engs[i % 2].feed_text(text, fastq=True, ord_base=ob, ord_stride=2)
    for e in engs:
        e.xchg_fence()
    out = {}
    for r, e in enumerate(engs):
        e.flush()
        st = e.finish_pass1()
        hist, _, _ = e.sweeps()
        e.build_layout()
        out[r] = (hist, [st.distinct, st.instances], e.dump_nodes())
    hist = [a + b for a, b in zip(out[0][0], out[1][0])]
    cnt = [out[0][1][0] + out[1][1][0], out[0][1][1] + out[1][1][1]]
    out[0] = (hist, cnt, out[0][2])
    _check(out, kmerfreq, want)
    for e in engs:
        e.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (gpurun --gpus 2)")
@pytest.mark.parametrize("gpus", [2, "all"])
def test_cli_multi_gpu_byte_identical(tmp_path, gpus):
    """configs[4] shape through the unchanged CLI with pass 1 sharded over the GPUs (PGB200_GPUS): all seven files and the
    reference's own `contig` outputs must equal the unmodified reference binary's (golden digests); tiny chunks so that every GPU gets many."""
    import subprocess
    cfg = synth.scenario_multilib(str(tmp_path))
    gpu = str(tmp_path / "gpu")
    rec = util.golden("multilib", 0, 63, 8, ("-a", "1", "-R"), cfg=cfg)
    env = dict(os.environ, PGB200_GPUS=str(gpus), PGB200_CHUNK_MB="1", PGB200_VERBOSE="1")
    r = subprocess.run([api.BIN63, "pregraph", "-s", cfg, "-K", "63", "-p", "8", "-a", "1", "-R", "-o", gpu], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert "pass 1 sharded over" in r.stderr
    util.compare_golden(gpu, rec, util.SUFFIXES_R)
    if util.have_ref():   # the contigs follow from the pregraph files; run the reference's own contig stage where it is built
        util.run([util.REF63, "contig", "-g", gpu, "-R"])
        util.compare_golden(gpu, rec, util.CONTIG_SUFFIXES)
