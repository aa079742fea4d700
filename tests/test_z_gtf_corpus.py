"""Damaged annotation files (tests/gtftools.py: 18 kinds the reference's GTF reader has defined behaviour for, annotation.cpp:113-377) through the oracle and
through the product (one of the two worlds also with a re-written assembly file: descriptions, ragged and empty lines, mixed case, IUPAC codes,
unplaced contigs): gene and exon tables, annotated fragment table, labels and both output files must be the reference's."""
import os
import pytest
import gtftools, worldutil
from test_ingest import check_front_end
from test_e2e import check_e2e


@pytest.fixture(scope="module")
def damaged(worlds, tmp_path_factory):
    out = {}
    for seed, rate, base in ((31, 0.08, worlds.get("small")), (32, 0.3, worlds.get("wide", scale=0.02, fragments=8000, breakpoints=100))):   # contigs beyond 3 Mb: room for a gene id that reappears too far away
        names, seqs = base.fasta
        lengths = {n: len(s) for n, s in zip(names, seqs)}
        d = os.path.join(str(tmp_path_factory.mktemp("gtf_corpus")), "w%d" % seed); os.makedirs(d)
        prefix = os.path.join(d, "w")
        os.symlink(base.prefix + ".bam", prefix + ".bam")
        if seed == 31:   # and the assembly as another tool might have written it
            gtftools.rewrite_fasta(names, seqs, prefix + ".fa", seed)
        else:
            os.symlink(base.prefix + ".fa", prefix + ".fa")
        tally = gtftools.damage_gtf(base.prefix + ".gtf", prefix + ".gtf", seed, rate, lengths)
        assert set(tally) == set(gtftools.KINDS), tally
        w = out[seed] = worldutil.reference_world(prefix, os.path.join(d, "oracle"))
        assert w.stderr_has("extends beyond end of contig") and w.stderr_has("failed to parse line in GTF file") and w.stderr_has("CDS record has unknown transcript ID")
        assert seed != 32 or w.stderr_has("appears to be non-unique")
    return out


@pytest.mark.parametrize("seed,threads", [(31, 1), (32, 4)])
def test_front_end_hostsim_damaged_gtf(damaged, hostsim_lib, seed, threads):
    check_front_end(damaged[seed], hostsim_lib, threads=threads)


@pytest.mark.parametrize("seed", [31, 32])
def test_e2e_hostsim_damaged_gtf(damaged, hostsim_lib, tmp_path, seed):
    check_e2e(damaged[seed], hostsim_lib, tmp_path)


@pytest.mark.gpu
def test_e2e_cuda_damaged_gtf(damaged, cuda_lib, tmp_path):
    check_front_end(damaged[31], cuda_lib, threads=8)
    check_e2e(damaged[32], cuda_lib, tmp_path, threads=8)
