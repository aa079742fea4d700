"""Committed golden fixtures (tests/golden/, produced by make_golden.py from the unmodified reference):
 * the reference's recorded run on the world the generator makes must have written them (pins the generator; while recording, the oracle),
 * the product must reproduce them: output files byte for byte, labels and per-stage candidate state exactly."""
import json, os
import numpy as np
import pytest
import worldutil
from arriba_b200 import lib as L

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
WORLDS = sorted(d for d in os.listdir(GOLDEN) if os.path.isdir(os.path.join(GOLDEN, d)))


def synth_world(name, tmp):
    params = json.load(open(os.path.join(GOLDEN, name, "params.json")))["synth"]
    extra = tuple(params.pop("extra", ()))
    prefix = os.path.join(str(tmp), "w")
    worldutil.run_synth(prefix, extra=extra, **params)
    return prefix


@pytest.mark.parametrize("name", WORLDS)
def test_oracle_reproduces_golden(name, tmp_path):
    prefix = synth_world(name, tmp_path)
    w = worldutil.reference_world(prefix, os.path.join(str(tmp_path), "oracle"))
    for f in ("fusions.tsv", "fusions.discarded.tsv"):
        assert w.same_output(f, os.path.join(GOLDEN, name, f)), f


def check_product_against_golden(name, tmp_path, lib_path):
    prefix = synth_world(name, tmp_path)
    g = np.load(os.path.join(GOLDEN, name, "stages.npz"))
    out = os.path.join(str(tmp_path), "fusions.tsv"); disc = os.path.join(str(tmp_path), "fusions.discarded.tsv")
    p = L.Pipeline(prefix + ".bam", prefix + ".gtf", prefix + ".fa", threads=3, lib_path=lib_path, output=out, discarded=disc)
    p.run(L.STEP_FIND_FUSIONS)
    labels, _ = p.context().fragment_filters()
    assert np.array_equal(labels, g["labels_after_read_filters"])
    st = p.stats()
    assert st.max_mate_gap == int(g["max_mate_gap"][0])
    p.events(0)
    index = {tuple(int(x) for x in row): i for i, row in enumerate(g["candidate_keys"])}
    stages = [n for n in L.EV_NAMES[1:] if n != "kmer_index"]
    seen = {}
    for s, name_ in enumerate(L.EV_NAMES[1:], start=1):
        p.events(s)
        if name_ == "kmer_index":
            continue
        base = {"internal_tandem_duplication": "internal_tandem_duplication", "select_best2": "select_best"}.get(name_, name_)
        occ = seen.get(base, 0); seen[base] = occ + 1
        tag = "ev_" + base if occ == 0 else "ev_%s_%d" % (base, occ + 1)
        c = p.candidates()
        perm = np.array([index[(int(c["gene1"][i]), int(c["gene2"][i]), int(c["contig1"][i]), int(c["contig2"][i]), int(c["breakpoint1"][i]), int(c["breakpoint2"][i]),
                                int(c["direction1"][i]), int(c["direction2"][i]))] for i in range(c["n"])])
        for col in ("filter", "split_reads1", "split_reads2", "discordant_mates"):
            assert np.array_equal(c[col], g[tag + "." + col][perm]), (tag, col)
        if s >= 3:
            assert np.array_equal(c["evalue"].view(np.uint32), g[tag + ".evalue"][perm].view(np.uint32)), (tag, "evalue")
    assert np.array_equal(p.candidates()["labels"], g["labels_final"])
    p.write_output(); p.close()
    assert open(out).read() == open(os.path.join(GOLDEN, name, "fusions.tsv")).read()
    assert open(disc).read() == open(os.path.join(GOLDEN, name, "fusions.discarded.tsv")).read()


@pytest.mark.parametrize("name", WORLDS)
def test_hostsim_reproduces_golden(name, tmp_path, hostsim_lib):
    check_product_against_golden(name, tmp_path, hostsim_lib)


@pytest.mark.gpu
@pytest.mark.parametrize("name", WORLDS)
def test_cuda_reproduces_golden(name, tmp_path, cuda_lib):
    check_product_against_golden(name, tmp_path, cuda_lib)
