"""The command line of the reference, option by option: the drop-in executable (here linked against the CPU stand-in) must write the same two files as
the reference run with the same arguments (options.cpp:270-485; defaults options.cpp:71-107)."""
import os
import subprocess
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pytest
import worldutil
from arriba_b200 import _build

OPTION_SETS = [
    ("-X",),                                        # extra columns for discarded fusions
    ("-s", "yes"), ("-s", "reverse"), ("-s", "no"),
    ("-u",),                                        # duplicates marked by the aligner
    ("-f", "blacklist,duplicates,mismatches"), ("-f", "blacklist,homologs,mismappers,merge_adjacent"), ("-f", "blacklist,low_entropy,homopolymer,read_through,select_best"),
    ("-E", "0.05", "-S", "3"), ("-m", "0.5", "-L", "0.1"), ("-H", "4", "-R", "5000"), ("-A", "30", "-M", "2"),
    ("-K", "0.3", "-V", "0.05"), ("-F", "300", "-U", "50"), ("-Q", "0.9", "-e", "0.5"), ("-l", "50", "-z", "0.2", "-Z", "5"),
    ("-i", "1,2,3,4,5,X"),
    # viral contigs: the two per-contig heuristics (top expressed, focal coverage) and the "only viral" rule; the synthetic worlds have no viral
    # genomes, so ordinary chromosomes are declared viral
    ("-v", "21,22"), ("-v", "19,20,21,22,X,Y", "-T", "2"), ("-v", "1,2,3,21,22", "-C", "0.5", "-T", "1"), ("-v", "20,21,22", "-f", "blacklist,top_expressed_viral_contigs"),
    ("-v", "20,21,22", "-f", "blacklist,low_coverage_viral_contigs"),
]


@pytest.fixture(scope="module")
def cli():
    return _build.build_cli_hostsim()


@pytest.mark.parametrize("extra", OPTION_SETS, ids=lambda o: " ".join(o))
def test_cli_option_parity(worlds, cli, tmp_path, extra):
    base = ("-f", "blacklist")
    args = tuple(extra) if "-f" in extra else base + tuple(extra)
    w = worlds.get("small", oracle_args=args)
    out = str(tmp_path / "fusions.tsv"); disc = str(tmp_path / "fusions.discarded.tsv")
    r = subprocess.run([cli, "-x", w.prefix + ".bam", "-g", w.prefix + ".gtf", "-a", w.prefix + ".fa", "-o", out, "-O", disc, "-@", "3"] + list(args), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert w.same_output("fusions.tsv", out), "fusions.tsv differs with options %s" % (args,)
    assert w.same_output("fusions.discarded.tsv", disc), "fusions.discarded.tsv differs with options %s" % (args,)


def test_cli_error_parity(worlds, cli, tmp_path):
    """Unusable inputs: same ERROR line and exit code as the reference (common.hpp:330, read_chimeric_alignments.cpp:566-609, annotation.cpp, assembly.cpp)."""
    w = worlds.get("small")
    d = str(tmp_path)
    bam = open(w.prefix + ".bam", "rb").read()
    gtf = open(w.prefix + ".gtf").read().split("\n")
    fa = open(w.prefix + ".fa").read().split(">")
    open(d + "/truncated.bam", "wb").write(bam[:len(bam) // 2 + 777])
    open(d + "/empty.bam", "wb").write(b"")
    open(d + "/garbage.bam", "wb").write(b"not a bam file at all" * 100)
    open(d + "/empty.gtf", "w").write("")
    open(d + "/no_exons.gtf", "w").write("\n".join(l for l in gtf if "\texon\t" not in l))
    open(d + "/two_contigs.fa", "w").write(">" + ">".join(fa[1:3]))
    # files that hold no chimeric fragment, no normal read, or no record at all (tests/bamtools.py re-writes the world's BAM)
    import bamtools, random
    text, refs, bodies = bamtools.read_bam(w.prefix + ".bam")
    recs = [(b, bamtools.split_record(b)) for b in bodies[:30000]]
    normal = [b for b, r in recs if (r["flag"] & 0x3) == 0x3 and not (r["flag"] & 0x900) and not any(t == b"SA" for t, _, _ in r["aux"])]
    chimeric = [b for b, r in recs if (r["flag"] & 0x1) and not (r["flag"] & 0x2)]
    assert len(normal) > 10 and len(chimeric) > 10
    bamtools.write_bam(d + "/only_normal.bam", text, refs, normal, random.Random(1)); bamtools.write_bam(d + "/only_chimeric.bam", text, refs, chimeric, random.Random(2))
    bamtools.write_bam(d + "/header_only.bam", text, refs, [], random.Random(3))
    cases = [(d + "/only_normal.bam", w.prefix + ".gtf", w.prefix + ".fa"), (d + "/only_chimeric.bam", w.prefix + ".gtf", w.prefix + ".fa"), (d + "/header_only.bam", w.prefix + ".gtf", w.prefix + ".fa"),
             (d + "/truncated.bam", w.prefix + ".gtf", w.prefix + ".fa"), (d + "/empty.bam", w.prefix + ".gtf", w.prefix + ".fa"), (d + "/garbage.bam", w.prefix + ".gtf", w.prefix + ".fa"),
             (w.prefix + ".bam", d + "/empty.gtf", w.prefix + ".fa"), (w.prefix + ".bam", d + "/no_exons.gtf", w.prefix + ".fa"), (w.prefix + ".bam", w.prefix + ".gtf", d + "/two_contigs.fa")]
    for b, g, a in cases:
        rc, errors, _ = worldutil.reference_cli(b, g, a, ["-f", "blacklist"])
        seen = [(rc, errors)]
        r = subprocess.run([cli, "-x", b, "-g", g, "-a", a, "-o", d + "/o.tsv", "-O", d + "/d.tsv", "-f", "blacklist", "-@", "2"], capture_output=True, text=True, timeout=300)
        seen.append((r.returncode, [l for l in r.stderr.split("\n") if l.startswith("ERROR")]))
        assert seen[0] == seen[1], (b, g, a, seen)
        assert seen[0][0] == 1 or b.endswith("only_chimeric.bam"), (b, g, a, seen)   # chimeric mates count as mapped reads: the reference runs through (and so must the product)


# ---- random option combinations on random worlds (python tests/test_cli_options.py SEED N runs N more) ----
FILTERS="duplicates inconsistently_clipped homopolymer read_through same_gene small_insert_size long_gap hairpin multimappers mismatches mismappers relative_support intronic non_coding_neighbors intragenic_exonic internal_tandem_duplication min_support known_fusions spliced end_to_end in_vitro merge_adjacent select_best marginal_read_through short_anchor no_coverage many_spliced no_genomic_support uninteresting_contigs viral_contigs top_expressed_viral_contigs low_coverage_viral_contigs genomic_support isoforms low_entropy homologs".split()


def random_options(rng):
    pool=[("-E",lambda: "%g"%rng.choice([0.001,0.05,0.3,1,10,1000])),("-S",lambda:str(rng.choice([0,1,2,3,5,20]))),("-m",lambda:"%g"%rng.choice([0,0.2,0.8,1])),("-L",lambda:"%g"%rng.choice([0,0.1,0.3,0.9,1])),
          ("-H",lambda:str(rng.choice([2,3,6,10,40]))),("-R",lambda:str(rng.choice([0,100,10000,1000000]))),("-A",lambda:str(rng.choice([0,10,23,40,90]))),("-M",lambda:str(rng.choice([0,1,4,10]))),
          ("-K",lambda:"%g"%rng.choice([0,0.3,0.6,1])),("-V",lambda:"%g"%rng.choice([0,0.001,0.01,0.5,1])),("-F",lambda:str(rng.choice([1,100,200,1000]))),("-U",lambda:str(rng.choice([1,2,10,300,32767]))),
          ("-Q",lambda:"%g"%rng.choice([0,0.5,0.998,1])),("-e",lambda:"%g"%rng.choice([0,0.33,1])),("-l",lambda:str(rng.choice([1,50,100,5000]))),("-z",lambda:"%g"%rng.choice([0,0.07,0.5,1])),("-Z",lambda:str(rng.choice([1,10,100]))),
          ("-s",lambda:rng.choice(["auto","yes","no","reverse"])),("-u",None),("-X",None),("-i",lambda:rng.choice(["1,2,3,4,5,X","1 2 3 4 5 6 7 8 9 10 11 12","*"])),("-v",lambda:rng.choice(["21,22","Y","AC_* NC_*"])),
          ("-T",lambda:str(rng.choice([1,2,5]))),("-C",lambda:"%g"%rng.choice([0,0.05,0.5,1]))]
    rng.shuffle(pool); out=[]
    for name,val in pool[:rng.randint(1,6)]:
        out.append(name)
        if val: out.append(val())
    fl=["blacklist"]+rng.sample(FILTERS, rng.choice([0,0,1,3,8]))
    return out+["-f",",".join(fl)]

def run_random_combination(rng, cli, d, k):
    """one random world, one random option set, reference and product side by side; True when both stop with the same error or both write the same two files"""
    from test_random_worlds import random_world_arguments
    kw = random_world_arguments(rng); pre = os.path.join(d, "w%d" % k)
    worldutil.run_synth(pre, **{kk: v for kk, v in kw.items() if kk != "extra"}, extra=kw["extra"])
    opts = random_options(rng)
    rc, errors, sha = worldutil.reference_cli(pre + ".bam", pre + ".gtf", pre + ".fa", opts, det_alloc=True)
    res = [(rc, errors)]
    r = subprocess.run([cli, "-x", pre + ".bam", "-g", pre + ".gtf", "-a", pre + ".fa", "-o", pre + ".p.tsv", "-O", pre + ".p.d.tsv"] + opts + ["-@", str(rng.choice([1, 3, 6]))],
                       capture_output=True, text=True, env=dict(os.environ, ARB_DET_ALLOC="1"), timeout=900)
    res.append((r.returncode, [l for l in r.stderr.splitlines() if l.startswith("ERROR")]))
    if res[0][0] != 0 or res[1][0] != 0:
        return res[0] == res[1], opts, kw
    same = sha == {"fusions.tsv": worldutil.file_digest(pre + ".p.tsv"), "fusions.discarded.tsv": worldutil.file_digest(pre + ".p.d.tsv")}
    return same, opts, kw


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5])
def test_cli_random_option_combination(cli, tmp_path, seed):
    import random
    ok, opts, kw = run_random_combination(random.Random(seed), cli, str(tmp_path), seed)
    assert ok, (opts, kw)


if __name__ == "__main__":
    import random, sys, tempfile
    rng = random.Random(int(sys.argv[1]) if len(sys.argv) > 1 else 1); bad = 0
    with tempfile.TemporaryDirectory() as d:
        for k in range(int(sys.argv[2]) if len(sys.argv) > 2 else 10):
            ok, opts, kw = run_random_combination(rng, _build.build_cli_hostsim(), d, k)
            print(k, "identical" if ok else "DIFFERENT", opts, "" if ok else kw, flush=True); bad += not ok
            for f in os.listdir(d):
                os.remove(os.path.join(d, f))
    sys.exit(1 if bad else 0)
