"""Degenerate samples: one to a few hundred fragments, no split reads at all, only split reads, nearly everything a duplicate or a multimapper -- stages that see
no fragment, no candidate or no surviving row (both files then hold the header line only). Fragment table, coverage, labels and both files are the reference's."""
import os
import pytest
from test_ingest import check_front_end
from arriba_b200 import lib as L

WORLDS = [(1, 1, ()), (3, 2, ()), (10, 1, ()), (40, 3, ("--normal-frac", "0.9")), (300, 2, ("--split-frac", "0.0")), (300, 2, ("--split-frac", "1.0")),
          (200, 5, ("--dup-frac", "0.9")), (500, 3, ("--multimap-frac", "0.9"))]


def world_of(worlds, fragments, breakpoints, extra):
    return worlds.get("degenerate", fragments=fragments, breakpoints=breakpoints, genes=50, scale=0.0005, extra=extra)


def check(world, lib_path, tmp_path, threads):
    check_front_end(world, lib_path, threads)
    out = os.path.join(str(tmp_path), "fusions.tsv"); disc = os.path.join(str(tmp_path), "fusions.discarded.tsv")
    p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=lib_path, output=out, discarded=disc)
    p.run_all(); p.close()
    assert world.same_output("fusions.tsv", out)
    assert world.same_output("fusions.discarded.tsv", disc)
    return len(open(out).read().splitlines()) - 1


@pytest.mark.parametrize("fragments,breakpoints,extra", WORLDS)
def test_degenerate_hostsim(worlds, hostsim_lib, tmp_path, fragments, breakpoints, extra):
    rows = check(world_of(worlds, fragments, breakpoints, extra), hostsim_lib, tmp_path, threads=2)
    assert fragments > 10 or rows == 0     # the smallest ones leave no row at all


@pytest.mark.gpu
def test_degenerate_cuda(worlds, cuda_lib, tmp_path):
    for fragments, breakpoints, extra in WORLDS:
        check(world_of(worlds, fragments, breakpoints, extra), cuda_lib, tmp_path, threads=3)
