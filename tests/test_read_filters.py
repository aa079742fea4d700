"""Parity of the read-level filter cascade: device labels vs. the oracle's per-stage labels (bit-exact)."""
import numpy as np
import pytest
import worldutil
from worldutil import digest


def check_read_filters(world, lib_path):
    p = worldutil.front_end(world, lib_path)
    ctx = p.context()
    ctx.run_read_filters()
    got, early = ctx.fragment_filters()
    assert digest(got) == world.stage_digest("rf_low_entropy", "frag_filter"), "labels differ from the reference's"
    assert digest(early) == world.stage_digest("rf_low_coverage_viral_contigs", "frag_filter")
    counts = ctx.filter_counts()
    want = world.fact("rf_low_entropy/0/frag_filter/bincount", lambda w: np.bincount(w.stage("rf_low_entropy")["frag_filter"], minlength=38)[:38].tolist())
    assert counts.tolist() == want
    assert int(counts[0]) == world.stage_scalar("rf_low_entropy", "remaining")
    # the world must actually exercise the rules
    assert want[1] > 0 and want[10] > 0 and want[36] > 0
    p.close()


def test_read_filters_hostsim(worlds, hostsim_lib):
    check_read_filters(worlds.get("small"), hostsim_lib)


def test_read_filters_hostsim_l151_shuffled(worlds, hostsim_lib):
    check_read_filters(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), hostsim_lib)


@pytest.mark.gpu
def test_read_filters_cuda(worlds, cuda_lib):
    check_read_filters(worlds.get("small"), cuda_lib)


@pytest.mark.gpu
def test_read_filters_cuda_l151(worlds, cuda_lib):
    check_read_filters(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), cuda_lib)


def check_packed_mismatch_counts(world, lib_path):
    """The eight-bases-per-step comparison on the 4-bit reference must count exactly like the base-by-base walk, also with ambiguity
    codes in reads and reference, reverse-complemented split reads, N bases and blocks running over the contig end."""
    from arriba_b200 import lib
    rng = np.random.default_rng(5)
    names, flags, seqs = worldutil.contigs_from_world(world)
    iupac = np.frombuffer(b"=ACMGRSVTWYHKDBN", np.uint8)
    seqs2 = []
    for s in seqs:
        a = np.frombuffer(s, np.uint8).copy()
        hit = rng.random(len(a)) < 0.02
        a[hit] = iupac[rng.integers(0, 16, int(hit.sum()))]
        seqs2.append(a.tobytes())
    p = worldutil.front_end(world, lib_path)   # the reference's annotated fragments and gene / exon tables
    ch = {k: np.array(v, copy=True) for k, v in p.fragments().items() if isinstance(v, np.ndarray)}
    n = ch["n_fragments"] = int(p.stats().n_fragments)
    g = p.genes(); p.close()
    ann = {k: v for k, v in g.items()}
    ann["exon_next_start"] = np.full(g["n_exons"], -1, np.int32)   # the exon and gene indexes are not read by the counts under test
    for k in ("exon", "gene"):
        ann[k + "_region_begin"] = np.zeros(g["n_contigs"] + 1, np.uint32); ann[k + "_region_end"] = np.zeros(1, np.int32)
        ann[k + "_region_off"] = np.zeros(1, np.uint32); ann[k + "_region_items"] = np.zeros(1, np.uint32)
    seq = ch["seq"]
    hit = rng.random(len(seq)) < 0.05                       # random nibbles: all 16 codes
    seq[hit] = rng.integers(0, 256, int(hit.sum()), dtype=np.uint8)
    flip = rng.random(n) < 0.5                              # supplementary on the other strand -> reverse-complemented comparison
    ch["aflags"][2 * n:][flip] ^= 8
    shift = rng.random(n) < 0.01                            # a few alignments hanging over the contig start
    ch["start"][:n][shift] = -3
    ctx = lib.Context(0, lib_path)
    ctx.set_contigs(flags, seqs2)
    ctx.set_annotation(ann)
    ctx.push_chunk(ch)
    out = np.zeros((n, 8), np.uint32)
    assert ctx.lib.arb_selftest_mismatch_counts(ctx.h, lib.ptr(out)) == 0
    assert np.array_equal(out[:, :4], out[:, 4:])
    assert out[:, 1].sum() > 50 * n and (out[:, 0] > 0).mean() > 0.5
    ctx.close()


def test_packed_mismatch_counts_hostsim(worlds, hostsim_lib):
    check_packed_mismatch_counts(worlds.get("small"), hostsim_lib)


@pytest.mark.gpu
def test_packed_mismatch_counts_cuda(worlds, cuda_lib):
    check_packed_mismatch_counts(worlds.get("small"), cuda_lib)
