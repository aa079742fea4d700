"""End to end: BAM + GTF + FASTA in, fusions.tsv / fusions.discarded.tsv out, byte-identical to the reference's files."""
import os
import pytest
import worldutil
from arriba_b200 import lib as L


def check_e2e(world, lib_path, tmp_path, threads=4):
    out = os.path.join(str(tmp_path), "fusions.tsv"); disc = os.path.join(str(tmp_path), "fusions.discarded.tsv")
    p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=lib_path, output=out, discarded=disc)
    p.run_all()
    p.close()
    assert world.output_lines("fusions.tsv") > 5
    assert world.same_output("fusions.tsv", out), "fusions.tsv differs from the reference's"
    assert world.same_output("fusions.discarded.tsv", disc), "discarded file differs"


def test_e2e_hostsim(worlds, hostsim_lib, tmp_path):
    check_e2e(worlds.get("small"), hostsim_lib, tmp_path)


def test_e2e_hostsim_row_blocks(worlds, hostsim_lib, tmp_path, monkeypatch):
    """the discarded rows are formatted on the device in blocks of rows (32-bit offsets inside a block): many small blocks"""
    monkeypatch.setenv("ARB_ROW_BLOCK", "1000")
    check_e2e(worlds.get("small"), hostsim_lib, tmp_path)


@pytest.mark.gpu
def test_e2e_cuda_row_blocks(worlds, cuda_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("ARB_ROW_BLOCK", "1000")
    check_e2e(worlds.get("small"), cuda_lib, tmp_path, threads=8)


def test_e2e_hostsim_consensus_overflow(worlds, hostsim_lib, tmp_path, monkeypatch):
    """pileups and consensus of the fusions rows (csrc/consensus_hd.h) with tiny tables: most jobs go through the second launch, some are left to the host code"""
    monkeypatch.setenv("ARB_CONSENSUS_TILES", "4")
    check_e2e(worlds.get("small"), hostsim_lib, tmp_path)


def test_e2e_hostsim_consensus_on_host(worlds, hostsim_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("ARB_DEVICE_CONSENSUS", "0")
    check_e2e(worlds.get("small"), hostsim_lib, tmp_path)


@pytest.mark.gpu
def test_e2e_cuda_consensus_overflow(worlds, cuda_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("ARB_CONSENSUS_TILES", "4")
    check_e2e(worlds.get("small"), cuda_lib, tmp_path, threads=8)


@pytest.mark.gpu
def test_e2e_cuda_consensus_on_host(worlds, cuda_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("ARB_DEVICE_CONSENSUS", "0")
    check_e2e(worlds.get("small"), cuda_lib, tmp_path, threads=8)


def test_e2e_hostsim_l151(worlds, hostsim_lib, tmp_path):
    check_e2e(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), hostsim_lib, tmp_path)


def test_e2e_hostsim_mismapper_heavy(worlds, hostsim_lib, tmp_path):
    from test_events import CFG5
    check_e2e(worlds.get("cfg5", **CFG5), hostsim_lib, tmp_path)


@pytest.mark.gpu
def test_e2e_cuda_mismapper_heavy(worlds, cuda_lib, tmp_path):
    from test_events import CFG5
    check_e2e(worlds.get("cfg5", **CFG5), cuda_lib, tmp_path, threads=8)


@pytest.mark.gpu
def test_e2e_cuda(worlds, cuda_lib, tmp_path):
    check_e2e(worlds.get("small"), cuda_lib, tmp_path, threads=8)


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [(), ("-v", "19,20,21,22,X,Y", "-T", "2")], ids=["default", "viral_contigs"])
def test_cli_cuda(worlds, tmp_path, extra):
    """The drop-in executable: same command line as the reference (run_arriba.sh:38-48), byte-identical files; with contigs declared viral the two
    per-contig heuristics and their device rules (filter_top_expressed_viral_contigs, filter_low_coverage_viral_contigs) take part."""
    import subprocess
    from arriba_b200 import _build
    args = ("-f", "blacklist") + tuple(extra)
    w = worlds.get("small", oracle_args=args)
    out = str(tmp_path / "fusions.tsv"); disc = str(tmp_path / "fusions.discarded.tsv")
    r = subprocess.run([_build.build_cli(), "-x", w.prefix + ".bam", "-g", w.prefix + ".gtf", "-a", w.prefix + ".fa", "-o", out, "-O", disc, "-@", "4"] + list(args),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert w.same_output("fusions.tsv", out)
    assert w.same_output("fusions.discarded.tsv", disc)


def test_e2e_hostsim_compressed_chr_names_normal_pairs(worlds, hostsim_lib, tmp_path):
    """Deflate-compressed BGZF blocks (zlib path instead of the stored-block copy), `chr`-prefixed contig names in the BAM header (remove_chr, arriba.cpp:52-58),
    and as many proper pairs as chimeric fragments (mate pairing, coverage, read-through extraction on normal reads)."""
    check_e2e(worlds.get("zchr", seed=11, extra=("--compress", "6", "--chr", "--normal-frac", "0.5")), hostsim_lib, tmp_path, threads=3)


def test_e2e_hostsim_deep_breakpoints(worlds, hostsim_lib, tmp_path):
    """A few breakpoints far beyond the subsampling threshold of 300 supporting reads (-U; fusions.cpp:423-441)."""
    check_e2e(worlds.get("deep", seed=12, breakpoints=300, extra=("--deep-frac", "0.02", "--deep-depth", "1500")), hostsim_lib, tmp_path, threads=5)


@pytest.mark.gpu
def test_e2e_cuda_compressed_chr_names_normal_pairs(worlds, cuda_lib, tmp_path):
    check_e2e(worlds.get("zchr", seed=11, extra=("--compress", "6", "--chr", "--normal-frac", "0.5")), cuda_lib, tmp_path, threads=8)


@pytest.mark.gpu
def test_e2e_cuda_deep_breakpoints(worlds, cuda_lib, tmp_path):
    check_e2e(worlds.get("deep", seed=12, breakpoints=300, extra=("--deep-frac", "0.02", "--deep-depth", "1500")), cuda_lib, tmp_path, threads=8)
