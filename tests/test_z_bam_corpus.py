"""(File names with z: the input corpora run after the established tests.)
BAM files from a second, independent writer (tests/bamtools.py: plain-Python reading of SAMv1 4.1 / 4.2) through the oracle and through the product's
ingest. The file means the same to the reference as the synth-written one it was made from (same core fields, CIGARs, sequences, HI and SA), so
 (1) the oracle must write the same two output files for both -- a check of the oracle's htslib shim against a writer that shares no code with it --
 (2) the product's front end must reproduce the oracle's fragment table, coverage and labels field by field from the transcoded file, and
 (3) both output files must come out byte-identical,
while every auxiliary type, tag order and integer width, missing qualities, and BGZF members of 1 byte .. 64 KiB (stored / deflated, empty ones in the
middle, records and their length words split over members, no EOF marker) pass through the readers."""
import os, shutil
import pytest
import bamtools, worldutil
from test_ingest import check_front_end
from test_e2e import check_e2e


def transcoded_world(worlds, tmp_root, seed, eof=True, **kw):
    base = worlds.get(**kw) if kw else worlds.get("small")
    d = os.path.join(str(tmp_root), "transcoded_%d_%d" % (seed, eof)); os.makedirs(d, exist_ok=True)
    prefix = os.path.join(d, "w")
    for ext in (".fa", ".gtf"):
        if not os.path.exists(prefix + ext):
            os.symlink(base.prefix + ext, prefix + ext)
    if not os.path.exists(prefix + ".bam"):
        n = bamtools.transcode(base.prefix + ".bam", prefix + ".bam", seed, eof)
        assert n > 1000
    return base, worldutil.reference_world(prefix, os.path.join(d, "oracle"))


@pytest.fixture(scope="module")
def corpus(worlds, tmp_path_factory):
    root = tmp_path_factory.mktemp("bam_corpus")
    return {(seed, eof): transcoded_world(worlds, root, seed, eof) for seed, eof in ((1, True), (2, False))}


def test_python_reader_round_trip(worlds, tmp_path):
    """the reader/writer pair itself: records survive split -> join unchanged, and a re-framed file reads back the same"""
    base = worlds.get("small")
    text, refs, bodies = bamtools.read_bam(base.prefix + ".bam")
    assert all(bamtools.join_record(bamtools.split_record(b)) == b for b in bodies[:5000])
    import random
    out = os.path.join(str(tmp_path), "again.bam")
    bamtools.write_bam(out, text, refs, bodies[:20000], random.Random(5))
    assert bamtools.read_bam(out) == (text, refs, bodies[:20000])


@pytest.mark.parametrize("which", [(1, True), (2, False)])
def test_oracle_reads_the_transcoded_file_the_same(corpus, which):
    base, tr = corpus[which]
    for name in ("fusions.tsv", "fusions.discarded.tsv"):
        assert tr.output_digest(name) == base.output_digest(name), name
    assert tr.output_lines("fusions.tsv") > 5


@pytest.mark.parametrize("which,threads", [((1, True), 3), ((2, False), 1)])
def test_front_end_hostsim_transcoded(corpus, hostsim_lib, which, threads):
    check_front_end(corpus[which][1], hostsim_lib, threads=threads)


def test_front_end_hostsim_transcoded_small_chunks(corpus, hostsim_lib, monkeypatch):
    """with the file read in chunks of a few members and the record boundaries found piecewise"""
    monkeypatch.setenv("ARB_CHUNK_BYTES", "50000"); monkeypatch.setenv("ARB_SCAN_MIN_BYTES", "700")
    check_front_end(corpus[(1, True)][1], hostsim_lib, threads=6)


def test_e2e_hostsim_transcoded(corpus, hostsim_lib, tmp_path):
    check_e2e(corpus[(2, False)][1], hostsim_lib, tmp_path)


@pytest.mark.gpu
def test_front_end_cuda_transcoded(corpus, cuda_lib):
    check_front_end(corpus[(1, True)][1], cuda_lib, threads=8)


@pytest.mark.gpu
def test_e2e_cuda_transcoded(corpus, cuda_lib, tmp_path):
    check_e2e(corpus[(2, False)][1], cuda_lib, tmp_path, threads=8)


# ---- files an aligner would not write: flag combinations, malformed fragments, orphans, wrong-end clips, missing / odd HI (bamtools.MUTATIONS) ----
def mutated_world(worlds, root, mutation_seed, rate, **kw):
    base = worlds.get(**kw) if kw else worlds.get("small")
    d = os.path.join(str(root), "mutated_%d" % mutation_seed); os.makedirs(d, exist_ok=True)
    prefix = os.path.join(d, "w")
    for ext in (".fa", ".gtf"):
        os.symlink(base.prefix + ext, prefix + ext)
    tally = bamtools.mutate(base.prefix + ".bam", prefix + ".bam", mutation_seed, rate)
    assert set(tally) == set(bamtools.MUTATIONS) and min(tally.values()) > 50, tally
    w = worldutil.reference_world(prefix, os.path.join(d, "oracle"))
    assert w.stderr_has("SAM records were malformed")   # the repair / rejection rules did fire in the reference
    return w


@pytest.fixture(scope="module")
def mutated(worlds, tmp_path_factory):
    root = tmp_path_factory.mktemp("bam_mutated")
    return {"collated": mutated_world(worlds, root, 21, 0.3),
            "shuffled": mutated_world(worlds, root, 22, 0.3, name="l151", read_length=151, seed=7, extra=("--shuffle", "--varnames"))}


@pytest.mark.parametrize("which,threads", [("collated", 1), ("collated", 5), ("shuffled", 4)])
def test_front_end_hostsim_mutated_records(mutated, hostsim_lib, which, threads):
    """a third of the read names carry one of 19 kinds of damage; the fragment table, the malformed count's consequences, coverage and labels equal the reference's"""
    check_front_end(mutated[which], hostsim_lib, threads=threads)


@pytest.mark.parametrize("which", ["collated", "shuffled"])
def test_e2e_hostsim_mutated_records(mutated, hostsim_lib, tmp_path, which):
    check_e2e(mutated[which], hostsim_lib, tmp_path)


@pytest.mark.gpu
def test_e2e_cuda_mutated_records(mutated, cuda_lib, tmp_path):
    check_front_end(mutated["collated"], cuda_lib, threads=8)
    check_e2e(mutated["shuffled"], cuda_lib, tmp_path, threads=8)



def test_alignment_beyond_the_contig_end_stops_the_run(worlds, hostsim_lib, tmp_path):
    """Alignments off the ends of their contig; mapped records without CIGAR, or whose CIGAR consumes more bases than the record holds (the reference dies on those:
    segmentation fault or std::out_of_range). Not valid records, and undefined in the reference (it indexes its coverage vectors and the contig string past their ends; on such files it aborts in free()
    or prints garbage): the product stops with an error instead of touching memory past the coverage windows (host) or the genome (device)."""
    import random, subprocess
    from arriba_b200 import _build
    base = worlds.get("small")
    text, refs, bodies = bamtools.read_bam(base.prefix + ".bam")
    def past(r): r["pos"] = refs[r["tid"]][1] + 5000
    def straddling(r): r["pos"] = refs[r["tid"]][1] - 30
    def before(r): r["pos"] = -5
    def cigar_longer(r): bamtools._set_cigar(r, [((o >> 4) + 50) << 4 | (o & 15) if (o & 15) == 0 else o for o in bamtools._cigar_ops(r)])
    def no_cigar(r): bamtools._set_cigar(r, [])
    def no_sequence(r): r["l_seq"] = 0; r["seq"] = b""; r["qual"] = b""
    for damage, message in ((past, "extends beyond the end of contig"), (straddling, "extends beyond the end of contig"), (before, "extends beyond the end of contig"),
                            (cigar_longer, "does not fit its sequence"), (no_cigar, "does not fit its sequence"), (no_sequence, "does not fit its sequence")):
        case = damage.__name__
        out = []; done = False
        for b in bodies:
            r = bamtools.split_record(b)
            if not done and r["tid"] >= 0 and not r["flag"] & 0x904 and (r["flag"] & 0x3) == 0x3:
                damage(r); b = bamtools.join_record(r); done = True
            out.append(b)
        prefix = os.path.join(str(tmp_path), case)
        bamtools.write_bam(prefix + ".bam", text, refs, out, random.Random(1))
        r = subprocess.run([_build.build_cli_hostsim(), "-x", prefix + ".bam", "-g", base.prefix + ".gtf", "-a", base.prefix + ".fa", "-o", prefix + ".tsv", "-O", prefix + ".d.tsv", "-f", "blacklist", "-@", "3"], capture_output=True, text=True, timeout=300)
        errors = [l for l in r.stderr.splitlines() if l.startswith("ERROR")]
        assert r.returncode == 1 and len(errors) == 1 and message in errors[0], (case, r.returncode, errors)


if __name__ == "__main__":   # python tests/test_z_bam_corpus.py SEED N : N random worlds (test_random_worlds.py), damaged and re-framed, through oracle and product
    import sys, random, tempfile
    from arriba_b200 import _build
    from test_random_worlds import random_world_arguments
    rng = random.Random(int(sys.argv[1]) if len(sys.argv) > 1 else 1)
    with tempfile.TemporaryDirectory() as d:
        cache = worldutil.WorldCache(d); bad = 0
        for k in range(int(sys.argv[2]) if len(sys.argv) > 2 else 10):
            kw = random_world_arguments(rng)
            base = cache.get("w%d" % k, **kw)
            wd = os.path.join(d, "damaged%d" % k); os.makedirs(wd)
            prefix = os.path.join(wd, "w")
            for ext in (".fa", ".gtf"):
                os.symlink(base.prefix + ext, prefix + ext)
            rate = rng.choice([0.02, 0.2, 0.6])
            bamtools.mutate(base.prefix + ".bam", prefix + ".tmp.bam", rng.randint(1, 10 ** 6), rate)
            bamtools.transcode(prefix + ".tmp.bam", prefix + ".bam", rng.randint(1, 10 ** 6)); os.remove(prefix + ".tmp.bam")
            try:
                worldutil.run_oracle(prefix, os.path.join(wd, "oracle"), dump=False)
            except RuntimeError as e:   # e.g. every chimeric fragment damaged: the reference stops with an error; the product must stop with the same one
                print(k, "reference stops:", str(e).strip().splitlines()[-1][:200], flush=True)
                continue
            w = worldutil.World(prefix, os.path.join(wd, "oracle"))
            try:
                check_e2e(w, _build.build_hostsim(), wd, threads=rng.choice([1, 3, 6])); ok = True
            except AssertionError as e:
                ok = False; print(str(e)[:1000])
            print(k, "identical" if ok else "DIFFERENT", rate, kw, flush=True); bad += not ok
            shutil.rmtree(wd)
        sys.exit(1 if bad else 0)
