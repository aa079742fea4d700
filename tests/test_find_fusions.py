"""Parity of candidate generation (find_fusions): candidate table, supporting lists and mate canonicalisation vs. the oracle."""
import numpy as np
import pytest
import worldutil
from worldutil import digest


def key_of(t, i):
    return (int(t["gene1"][i]), int(t["gene2"][i]), int(t["contig1"][i]), int(t["contig2"][i]), int(t["breakpoint1"][i]), int(t["breakpoint2"][i]),
            int(t["direction1"][i]), int(t["direction2"][i]))


KEY = ("gene1", "gene2", "contig1", "contig2", "breakpoint1", "breakpoint2", "direction1", "direction2")


def by_key(t):
    """permutation that sorts a candidate table by its 8-tuple key"""
    return np.lexsort([np.asarray(t[k]).astype(np.int64) for k in reversed(KEY)])


def candidate_digests(t, bits, bits2):
    """digests of a candidate table in key order: keys, read counts, filter, anchors, exonic / spliced / strand bits and the supporting lists"""
    o = by_key(t)
    out = {k: digest(np.asarray(t[k])[o]) for k in KEY + ("split_reads1", "split_reads2", "discordant_mates", "filter", "anchor_start1", "anchor_start2")}
    out["bits"] = digest(np.asarray(bits)[o]); out["bits2"] = digest(np.asarray(bits2)[o])
    for lname, oname in (("list1", "list1_off"), ("list2", "list2_off"), ("listd", "listd_off")):
        off = np.asarray(t[oname]).astype(np.int64)
        out[lname] = digest(worldutil._segments(t[lname], off[:-1][o], np.diff(off)[o]))
        out[lname + "_sizes"] = digest(np.diff(off)[o])
    out["n"] = len(o); out["n_unique"] = len(set(zip(*[np.asarray(t[k]).tolist() for k in KEY])))
    return out


def reference_candidates(w):
    ff = w.stage("find_fusions")
    bits = (ff["exonic1"].astype(np.int64) | ff["exonic2"].astype(np.int64) << 1 | ff["spliced1"].astype(np.int64) << 2 | ff["spliced2"].astype(np.int64) << 3 |
            ff["predicted_strand1"].astype(np.int64) << 4 | ff["predicted_strand2"].astype(np.int64) << 5 | ff["predicted_strands_ambiguous"].astype(np.int64) << 6 |
            ff["transcript_start"].astype(np.int64) << 7)
    return candidate_digests(ff, bits, ff["transcript_start_ambiguous"])


def reference_swaps(w):
    """mate canonicalisation in the reference (fusions.cpp:416-421): the fragments whose first alignment changed"""
    ff, ann = w.stage("find_fusions"), w.stage("annotated")
    first = ann["aln_off"][:-1]
    swapped = (ff["slot0_start"] != ann["start"][first]) | (ff["slot0_contig"] != ann["contig"][first])
    return {"swapped": digest(np.nonzero(swapped)[0]), "n": int(swapped.sum())}


def check_find_fusions(world, lib_path):
    p = worldutil.front_end(world, lib_path)
    fr = p.fragments(); n = fr["n_fragments"]
    # a swap of two mates with identical start and contig is not observable in the reference's dump
    twins = (fr["start"][:n] == fr["start"][n:2 * n]) & (fr["contig"][:n] == fr["contig"][n:2 * n]) & (fr["n_aln"] > 1)
    ctx = p.context()
    # start from the reference's labels so that this test isolates find_fusions
    ctx.run_read_filters()
    labels, _ = ctx.fragment_filters()
    assert digest(labels) == world.stage_digest("rf_low_entropy", "frag_filter")
    ctx.set_fragment_filters(labels)
    ctx.find_fusions(world.stage_scalar("find_fusions", "max_mate_gap"))
    got = ctx.candidates()
    want = world.fact("find_fusions/candidates", reference_candidates)
    assert want["n_unique"] == want["n"] and got["n"] == want["n"]
    mine = candidate_digests(got, got["bits"], got["bits2"])
    bad = [k for k in want if mine[k] != want[k]]
    assert not bad, ("candidate columns differ from the reference's", bad)
    assert want["n"] > 0
    # candidates are numbered in the reference's first-insertion order: first supporting fragment ascending
    # mate canonicalisation (fusions.cpp:416-421)
    ref = world.fact("find_fusions/swaps", reference_swaps)
    swapped_got = ctx.slot_swaps().astype(bool)
    assert digest(np.nonzero(swapped_got & ~twins)[0]) == ref["swapped"], "canonicalisation differs from the reference's"
    assert int((got["filter"] == 0).sum()) == world.stage_scalar("find_fusions", "remaining")
    p.close()


def test_find_fusions_hostsim(worlds, hostsim_lib):
    check_find_fusions(worlds.get("small"), hostsim_lib)


def test_find_fusions_hostsim_l151_shuffled(worlds, hostsim_lib):
    check_find_fusions(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), hostsim_lib)


@pytest.mark.gpu
def test_find_fusions_cuda(worlds, cuda_lib):
    check_find_fusions(worlds.get("small"), cuda_lib)


@pytest.mark.gpu
def test_find_fusions_cuda_l151(worlds, cuda_lib):
    check_find_fusions(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), cuda_lib)
