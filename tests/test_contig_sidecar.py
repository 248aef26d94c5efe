"""CPU: f2 -- the binary edge sidecar and its `contig` loader (SURVEY 8f, loadPreGraph.c:448-544).

The reference's `contig` stage, linked with csrc/contig_sidecar.c (scripts/link_dropin.sh: loadEdge renamed inside the reference's
own object with objcopy), must produce the same .contig / .Arc / .updated.edge / .ContigIndex whether it parses <prefix>.edge.gz or
reads <prefix>.edge.b200, and the same as the unmodified reference binary.  The sidecar here is made by the library's host-side
converter from the reference's own .edge.gz (no GPU involved); tests/test_gpu_dropin.py checks that the GPU stage writes the same
sidecar bytes itself."""
import os
import shutil
import subprocess

import pytest

from soapdenovo2_b200 import api, synth
from tests import util

B63 = os.path.join(util.ROOT, "oracle", "_ref", "SOAPdenovo-63mer-b200")
B127 = os.path.join(util.ROOT, "oracle", "_ref", "SOAPdenovo-127mer-b200")
OUT = ["contig", "Arc", "updated.edge", "ContigIndex"]


@pytest.fixture(scope="module", autouse=True)
def _build():
    subprocess.run(["make", "-s", "-j8", "-C", os.path.join(util.ROOT, "soapdenovo2_b200", "csrc")], check=True)


@pytest.fixture(scope="module")
def _dropin():
    """The drop-in binaries are linked from the reference's own objects: only where oracle/Makefile could build those."""
    if not (util.have_ref() and os.path.isdir(os.path.join(util.ROOT, "oracle", "_ref", "o63"))):
        pytest.skip("oracle/_ref absent (the reference's objects are built by `make -C oracle ref` where its sources are)")
    subprocess.run(["bash", os.path.join(util.ROOT, "scripts", "link_dropin.sh")], check=True, capture_output=True)


def _copy_pregraph(src, dst):
    for s in util.SUFFIXES_R:
        if os.path.exists(f"{src}.{s}"):
            shutil.copy(f"{src}.{s}", f"{dst}.{s}")


@pytest.mark.parametrize("flav,K,extra", [(0, 63, ("-R",)), (0, 31, ()), (1, 91, ("-R",))])
def test_contig_reads_the_sidecar(_dropin, tmp_path, flav, K, extra):
    cfg = synth.scenario_multilib(str(tmp_path)) if K != 31 else synth.scenario_se_fasta(str(tmp_path))
    ref_bin, b200_bin = (util.REF127, B127) if flav else (util.REF63, B63)
    ref = str(tmp_path / "ref")
    util.run([ref_bin, "pregraph", "-s", cfg, "-K", str(K), "-p", "4", "-a", "1", "-o", ref, *extra])
    text_run, side_run = str(tmp_path / "text"), str(tmp_path / "side")
    _copy_pregraph(ref, text_run)
    _copy_pregraph(ref, side_run)
    api.edge_gz_to_sidecar(side_run, K, flav)
    assert os.path.getsize(side_run + ".edge.b200") > 48
    log = {}
    for exe, pre in ((ref_bin, ref), (b200_bin, text_run), (b200_bin, side_run)):
        log[pre] = util.run([exe, "contig", "-g", pre, *extra])
    util.compare(ref, text_run, OUT)      # the renamed original loader still works through the wrapper
    util.compare(ref, side_run, OUT)      # and the sidecar gives the same graph
    pick = lambda l: [x for x in l.splitlines() if "edge(s) input" in x or "pre-arcs loaded" in x]
    assert pick(log[ref]) == pick(log[side_run]) != []
    # the sidecar really was the source: without the .edge.gz the stage still runs
    os.remove(side_run + ".edge.gz")
    util.run([b200_bin, "contig", "-g", side_run, *extra])
    util.compare(ref, side_run, OUT)
    # and the way back: the sidecar regenerates the reference's .edge.gz byte for byte (text AND deflate stream)
    api.sidecar_to_edge_gz(side_run)
    util.compare(ref, side_run, ["edge.gz"])
    os.remove(side_run + ".edge.gz")
    util.run([api.BIN127 if flav else api.BIN63, "edgegz", "-g", side_run])   # the same through the CLI
    util.compare(ref, side_run, ["edge.gz"])


def test_sidecar_converter_rejects_garbage(tmp_path):
    lib = api.load()
    bad = b">length 5,1 2,3 4,cvg x, 1\nACGTA\n"
    assert lib.pgb200_edge_text_to_sidecar(bad, len(bad), 31, 0, 2, str(tmp_path / "x.b200").encode()) != 0
    open(str(tmp_path / "y.edge.b200"), "wb").write(b"PGB2EDGE" + bytes(20))
    assert lib.pgb200_sidecar_to_edge_gz(str(tmp_path / "y").encode()) != 0
    assert lib.pgb200_sidecar_to_edge_gz(str(tmp_path / "absent").encode()) != 0
