"""Event-level chain: after every stage the candidate table (filter, read counts, e-value) must equal the oracle's."""
import numpy as np
import pytest
from arriba_b200 import lib as L
from test_find_fusions import KEY, by_key
from worldutil import digest

COLUMNS = ("filter", "split_reads1", "split_reads2", "discordant_mates")


def stage_digests(t, with_evalue, with_confidence):
    """a candidate table in key order: keys, filter, read counts, supporting list sizes (and e-values, confidence)"""
    o = by_key(t)
    out = {c: digest(np.asarray(t[c])[o]) for c in KEY + COLUMNS + (("evalue",) if with_evalue else ()) + (("confidence",) if with_confidence else ())}
    for oname in ("list1_off", "list2_off"):
        out[oname + " sizes"] = digest(np.diff(np.asarray(t[oname]).astype(np.int64))[o])
    return out


def reference_stage(name, occ, with_evalue):
    def compute(w):
        t = w.stage("ev_" + name, occ)
        return {"candidates": stage_digests(t, with_evalue, name == "confidence"), "remaining": int(t["remaining"][0]),
                "frag_filter": digest(t["frag_filter"]) if "frag_filter" in t else None}
    return compute


def compare_stage(got, want, stage, check_evalue):
    mine = stage_digests(got, check_evalue, stage == "confidence")
    bad = [k for k in want if mine[k] != want[k]]
    assert not bad, (stage, "candidate columns differ from the reference's", bad)


def check_events(world, lib_path, threads=4, keep=False):
    p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=lib_path)
    p.run(L.STEP_FIND_FUSIONS)
    p.events(0)
    got = p.candidates()
    # the replayed unordered_map iteration order must be the reference's
    want_keys = world.fact("find_fusions/order", lambda w: {k: digest(w.stage("find_fusions")[k]) for k in KEY})
    got_keys = {k: digest(got[k][got["order"]]) for k in KEY}
    assert got_keys == want_keys, "iteration order of the candidate table differs from the reference's unordered_map"
    stages = ["merge_adjacent", "multimappers", "evalue", "non_coding_neighbors", "intragenic_exonic", "min_support", "relative_support", "internal_tandem_duplication",
              "intronic", "in_vitro", "spliced", "select_best", "marginal_read_through", "many_spliced", "short_anchor", "end_to_end", "no_coverage",
              "kmer_index", "homologs", "mismappers", "select_best", "isoforms", "confidence"]
    occurrence = {}
    seen_evalue = False
    for s, name in enumerate(stages, start=1):
        p.events(s)
        got = p.candidates()
        if name == "kmer_index":
            continue
        occ = occurrence.get(name, 0); occurrence[name] = occ + 1
        seen_evalue = seen_evalue or name == "evalue"
        want = world.fact("ev_%s/%d/candidates" % (name, occ), reference_stage(name, occ, seen_evalue))
        compare_stage(got, want["candidates"], name, seen_evalue)
        if want["frag_filter"] is not None:
            assert digest(got["labels"]) == want["frag_filter"], (name, "fragment labels")
        assert int((got["filter"] == 0).sum()) == want["remaining"] or name in ("evalue", "confidence"), name
    if keep:
        return p
    p.close()


def test_events_hostsim(worlds, hostsim_lib):
    check_events(worlds.get("small"), hostsim_lib)


def test_events_hostsim_l151(worlds, hostsim_lib):
    check_events(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), hostsim_lib)


CFG5 = dict(scale=0.002, genes=800, breakpoints=400, fragments=40000, extra=("--mismapper-frac", "0.3", "--paralog-frac", "0.15"))


def test_events_hostsim_mismapper_heavy(worlds, hostsim_lib):
    """BASELINE.json configs[4] in miniature: homologous partners, clipped segments alignable in the donor, adjacent breakpoints, ITD merges."""
    w = worlds.get("cfg5", **CFG5)
    n = w.fact("ev/mismapper_heavy_counts", lambda w: [int((w.stage("ev_mismappers")["frag_filter"] == 11).sum()), int((w.stage("ev_mismappers")["filter"] == 11).sum()),
                                                       int((w.stage("ev_homologs")["filter"] == 37).sum()), int((w.stage("ev_merge_adjacent")["filter"] == 23).sum())])
    assert n[0] > 1000 and n[1] > 20 and n[2] > 5
    assert n[3] > 20
    check_events(w, hostsim_lib)


def test_events_hostsim_cooperative_realignment(worlds, hostsim_lib, monkeypatch):
    """A tiny step budget pushes almost every (candidate, read) pair through the cooperative second pass; labels must not change."""
    monkeypatch.setenv("ARB_MISMAP_BUDGET", "24"); monkeypatch.setenv("ARB_MISMAP_LANES", "7")
    monkeypatch.setenv("ARB_MISMAP_SPAWN", "6"); monkeypatch.setenv("ARB_MISMAP_TASK_LANES", "3")
    p = check_events(worlds.get("cfg5", **CFG5), hostsim_lib, keep=True)
    tm = p.context().timings(); p.close()
    assert tm.mismapper_heavy_items > 0.2 * tm.mismapper_items
    assert tm.mismapper_tasks > 1000 and tm.mismapper_rounds >= 2   # continuations of continuations were registered as well


@pytest.mark.parametrize("spawn,table", [("0", "1048576"), ("0", "64"), ("5", "1")])
def test_events_hostsim_continuation_registry(worlds, hostsim_lib, monkeypatch, spawn, table):
    """No bounded attempts (every continuation is registered), and registries so small that most registrations fail over to the in-line search."""
    monkeypatch.setenv("ARB_MISMAP_BUDGET", "24"); monkeypatch.setenv("ARB_MISMAP_LANES", "5")
    monkeypatch.setenv("ARB_MISMAP_SPAWN", spawn); monkeypatch.setenv("ARB_MISMAP_TASK_LANES", "4"); monkeypatch.setenv("ARB_MISMAP_TABLE_TOTAL", table)
    check_events(worlds.get("cfg5", **CFG5), hostsim_lib)


@pytest.mark.parametrize("lanes", ["1", "7"])
def test_events_hostsim_homolog_lanes(worlds, hostsim_lib, monkeypatch, lanes):
    """filter_homologs' identity test with one thread per gene pair and with lanes that split the positions: same verdicts."""
    monkeypatch.setenv("ARB_HOMOLOG_LANES", lanes)
    check_events(worlds.get("cfg5", **CFG5), hostsim_lib)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", ["1", "32"])
def test_events_cuda_homolog_lanes(worlds, cuda_lib, monkeypatch, lanes):
    monkeypatch.setenv("ARB_HOMOLOG_LANES", lanes)
    check_events(worlds.get("cfg5", **CFG5), cuda_lib)


@pytest.mark.gpu
def test_events_cuda_mismapper_heavy(worlds, cuda_lib):
    check_events(worlds.get("cfg5", **CFG5), cuda_lib)


@pytest.mark.gpu
@pytest.mark.parametrize("budget,lanes,spawn,task_lanes", [("16", "32", "4", "32"), ("200", "256", "0", "32"), ("0", "1", "0", "1"), ("64", "8", "16", "5")])
def test_events_cuda_cooperative_realignment(worlds, cuda_lib, monkeypatch, budget, lanes, spawn, task_lanes):
    monkeypatch.setenv("ARB_MISMAP_BUDGET", budget); monkeypatch.setenv("ARB_MISMAP_LANES", lanes)
    monkeypatch.setenv("ARB_MISMAP_SPAWN", spawn); monkeypatch.setenv("ARB_MISMAP_TASK_LANES", task_lanes)
    check_events(worlds.get("cfg5", **CFG5), cuda_lib)


@pytest.mark.gpu
def test_events_cuda(worlds, cuda_lib):
    check_events(worlds.get("small"), cuda_lib)
