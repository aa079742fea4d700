"""Parity of the host front end (BAM ingest, annotation, dummy genes, strandedness, fragment length) with the oracle,
and of the whole file-to-candidates path."""
import numpy as np
import pytest
import worldutil
from worldutil import digest
from arriba_b200 import lib as L


frag_tables_equal = worldutil.frag_tables_equal


def check_front_end(world, lib_path, threads):
    p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=lib_path)
    p.step(L.STEP_LOAD_REFERENCE)
    p.step(L.STEP_INGEST)
    st = p.stats()
    assert st.mapped_reads == world.stage_scalar("read_chimeric_alignments", "mapped_reads")
    assert st.n_fragments == world.stage_scalar("read_chimeric_alignments", "total")
    frag_tables_equal(p.fragments(), world, "ingest", check_genes=False, check_pred=False)
    # coverage windows, contig by contig
    def coverage_ref(w):
        rca = w.stage("read_chimeric_alignments")
        return {"sizes": digest(np.diff(rca["coverage_off"].astype(np.int64))), "coverage": digest(rca["coverage"]),
                "starts": digest(rca["fragment_starts"]), "ends": digest(rca["fragment_ends"]), "n_contigs": len(rca["coverage_off"]) - 1}
    want = world.fact("coverage", coverage_ref)
    windows = [p.coverage(c) for c in range(want["n_contigs"])]
    got = {"sizes": digest([len(w[0]) for w in windows]), "n_contigs": want["n_contigs"]}
    for i, k in enumerate(("coverage", "starts", "ends")):
        got[k] = digest(np.concatenate([w[i] for w in windows]) if windows else [])
    assert got == want, [k for k in want if got[k] != want[k]]
    p.step(L.STEP_ANNOTATE)
    assert p.stats().strandedness == world.stage_scalar("strandedness", "strandedness")
    frag_tables_equal(p.fragments(), world, "annotated", check_genes=True, check_pred=True)
    g = p.genes()
    assert g["n_genes"] == world.fact("fragment_length/n_genes", lambda w: len(w.stage("fragment_length")["gene_id"]))
    for k in ("gene_contig", "gene_start", "gene_end", "gene_strand", "gene_exonic_length"):
        assert digest(g[k]) == world.stage_digest("fragment_length", k), k
    assert digest(g["gene_flags"]) == world.fact("fragment_length/gene_flags", lambda w: digest(w.stage("fragment_length")["gene_is_dummy"] | w.stage("fragment_length")["gene_is_protein_coding"] << 1))
    exon_columns = ("exon_gene", "exon_start", "exon_end", "exon_cds_start", "exon_cds_end", "exon_flags")
    want_ann = world.fact("fragment_length/exons", lambda w: {k: digest(v) for k, v in worldutil.annotation_from_dump(w.stage("fragment_length"), g["n_contigs"]).items() if k in exon_columns})
    for k in exon_columns:
        assert digest(g[k]) == want_ann[k], k
    # device stages fed by the product's own front end
    p.step(L.STEP_UPLOAD); p.step(L.STEP_READ_FILTERS); p.step(L.STEP_FRAGMENT_LENGTH)
    ctx = p.context()
    labels, early = ctx.fragment_filters()
    assert digest(labels) == world.stage_digest("rf_low_entropy", "frag_filter")
    st = p.stats()
    assert st.fragment_length_ok == world.stage_scalar("fragment_length", "ok")
    if st.fragment_length_ok:
        gap = world.fact("fragment_length/gap_mean_stddev_readlen", lambda w: [float(x) for x in w.stage("fragment_length")["gap_mean_stddev_readlen"]])
        assert st.mate_gap_mean == gap[0] and st.mate_gap_stddev == gap[1]
        assert st.read_length_mean == gap[2]
    assert st.max_mate_gap == world.stage_scalar("find_fusions", "max_mate_gap")
    p.step(L.STEP_FIND_FUSIONS)
    cand = ctx.candidates()
    assert cand["n"] == world.fact("find_fusions/n", lambda w: len(w.stage("find_fusions")["gene1"]))
    assert int((cand["filter"] == 0).sum()) == world.stage_scalar("find_fusions", "remaining")
    p.close()


def test_front_end_hostsim(worlds, hostsim_lib):
    check_front_end(worlds.get("small"), hostsim_lib, threads=1)


def test_front_end_hostsim_threads_shuffled(worlds, hostsim_lib):
    check_front_end(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), hostsim_lib, threads=5)


@pytest.mark.gpu
def test_front_end_cuda(worlds, cuda_lib):
    check_front_end(worlds.get("small"), cuda_lib, threads=8)


@pytest.mark.parametrize("threads,min_bytes", [(7, "20000"), (16, "1000"), (3, "300")])
def test_front_end_hostsim_parallel_record_scan(worlds, hostsim_lib, monkeypatch, threads, min_bytes):
    """Record boundaries found piecewise from guessed starts (verified against the true chain; csrc/bamscan.cu), down to pieces smaller than a record."""
    monkeypatch.setenv("ARB_SCAN_MIN_BYTES", min_bytes)
    monkeypatch.setenv("ARB_BAM_SCAN_PIECE", str(max(50, int(min_bytes) // 4)))
    check_front_end(worlds.get("l151", read_length=151, seed=7, extra=("--shuffle", "--varnames")), hostsim_lib, threads=threads)


@pytest.mark.parametrize("threads,min_bytes", [(6, "5000"), (13, "100")])
def test_front_end_hostsim_parallel_block_table_compressed(worlds, hostsim_lib, monkeypatch, threads, min_bytes):
    """The BGZF block table is found piecewise too (guessed block starts, verified against the true chain): deflate-compressed blocks, whose payload is
    arbitrary bytes, and pieces smaller than one block."""
    monkeypatch.setenv("ARB_SCAN_MIN_BYTES", min_bytes)
    check_front_end(worlds.get("zsmall", seed=5, extra=("--compress", "6")), hostsim_lib, threads=threads)


def test_block_table_errors_are_the_serial_ones(worlds, hostsim_lib, monkeypatch, tmp_path):
    """A file cut inside a block, or with a damaged block header in the middle, fails with the message of the one-thread walk."""
    from arriba_b200 import lib as L
    world = worlds.get("small")
    raw = open(world.prefix + ".bam", "rb").read()
    damaged = bytearray(raw); mid = raw.find(b"\x1f\x8b\x08\x04", len(raw) // 2); damaged[mid + 1] = 0
    cases = {"cut": raw[:len(raw) * 2 // 3], "damaged": bytes(damaged)}
    for name, data in cases.items():
        path = str(tmp_path / (name + ".bam")); open(path, "wb").write(data)
        messages = []
        for min_bytes, threads in (("1000000000", 1), ("1000", 9)):
            monkeypatch.setenv("ARB_SCAN_MIN_BYTES", min_bytes)
            p = L.Pipeline(path, world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=hostsim_lib)
            p.step(L.STEP_LOAD_REFERENCE)
            with pytest.raises(L.ArbError) as err:
                p.step(L.STEP_INGEST)
            messages.append(str(err.value)); p.close()
        assert messages[0] == messages[1] and "failed to load alignments" in messages[0], (name, messages)


@pytest.mark.parametrize("threads,chunk_bytes,extra", [(4, "70000", ()), (3, "300000", ("--compress", "6")), (9, "1", ("--shuffle", "--varnames"))])
def test_front_end_hostsim_many_chunks(worlds, hostsim_lib, monkeypatch, threads, chunk_bytes, extra):
    """The file is read in chunks (128 MiB in production): records that straddle a chunk boundary are carried over, mates that wait for their partner
    survive the recycling of the buffer, and the workers' pools are reserved ahead after the first chunk. Here: chunks of one to a few BGZF blocks."""
    monkeypatch.setenv("ARB_CHUNK_BYTES", chunk_bytes)
    name = "chunks_" + "_".join(x.strip("-") for x in extra) if extra else "small"
    kw = dict(seed=5, extra=extra) if extra else {}
    check_front_end(worlds.get(name, **kw), hostsim_lib, threads=threads)


def test_pools_are_kept_between_samples_and_can_be_released(worlds, hostsim_lib, tmp_path):
    """the ingest keeps the workers' pools of a finished sample (csrc/host/ingest.cpp, take_workers / put_workers): a second sample in the same process, a third
    after arb_release_host_memory, and one with another number of workers must all read the same table"""
    import numpy as np
    from arriba_b200 import lib as L
    world = worlds.get("small")
    def table(threads):
        p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=hostsim_lib,
                       output=str(tmp_path / "f.tsv"), discarded=str(tmp_path / "d.tsv"))
        p.step(L.STEP_LOAD_REFERENCE); p.step(L.STEP_INGEST)
        f = p.fragments()
        mine = ("n_aln", "fflags", "contig", "start", "end", "cigar_off", "cigar_cnt", "seq_off", "seq_len", "cigar", "seq", "name_off")   # what the ingest itself fills (the gene columns belong to the annotation)
        out = {k: np.array(f[k], copy=True) for k in mine}
        out["names"] = np.frombuffer(f["names_blob"], dtype=np.uint8).copy()
        p.close()
        return out
    first = table(4)
    again = table(4)
    L.load(hostsim_lib).arb_release_host_memory()
    after_release = table(4)
    other_width = table(3)
    for other in (again, after_release, other_width):
        assert sorted(other) == sorted(first)
        for k in first:
            assert np.array_equal(first[k], other[k]), k
