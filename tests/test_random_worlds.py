"""Differential runs on randomly parameterised worlds (read length, depth, name style, BGZF compression, contig naming, mixtures of normal pairs / split reads /
duplicates / multimappers / mismappers / paralogs / very deep breakpoints): both TSV files must equal the reference's byte for byte. `python tests/test_random_worlds.py
SEED N` runs N more of them."""
import os
import random
import sys
import pytest
import worldutil
from arriba_b200 import lib as L, _build


def random_world_arguments(rng):
    kw = dict(seed=rng.randint(1, 10 ** 6), read_length=rng.choice([76, 101, 125, 151]), fragments=rng.choice([8000, 20000, 30000]), breakpoints=rng.choice([60, 150, 300]), genes=rng.choice([200, 400, 800]))
    extra = []
    if rng.random() < 0.5: extra += ["--shuffle"]
    if rng.random() < 0.5: extra += ["--varnames"]
    if rng.random() < 0.4: extra += ["--compress", str(rng.choice([1, 6]))]
    if rng.random() < 0.4: extra += ["--chr"]
    for option, choices in (("--normal-frac", [0.1, 0.5]), ("--split-frac", [0.3, 0.9]), ("--dup-frac", [0.2]), ("--multimap-frac", [0.1, 0.3]), ("--mismapper-frac", [0.3]), ("--paralog-frac", [0.2]), ("--deep-frac", [0.03])):
        if rng.random() < 0.35: extra += [option, str(rng.choice(choices))]
    if "--deep-frac" in extra: extra += ["--deep-depth", "900"]
    kw["extra"] = tuple(extra)
    return kw


def run_one(cache, name, kw, lib_path, threads, outdir):
    w = cache.get(name, **kw)
    out = os.path.join(outdir, "fusions.tsv"); disc = os.path.join(outdir, "fusions.discarded.tsv")
    p = L.Pipeline(w.prefix + ".bam", w.prefix + ".gtf", w.prefix + ".fa", threads=threads, lib_path=lib_path, output=out, discarded=disc)
    p.run_all(); p.close()
    return w.same_output("fusions.tsv", out) and w.same_output("fusions.discarded.tsv", disc)


@pytest.mark.parametrize("seed", [11, 12, 13, 14])
def test_random_world_hostsim(worlds, hostsim_lib, tmp_path, seed):
    rng = random.Random(seed)
    kw = random_world_arguments(rng)
    assert run_one(worlds, "random%d" % seed, kw, hostsim_lib, rng.choice([1, 3, 6]), str(tmp_path)), kw


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [11, 12])
def test_random_world_cuda(worlds, cuda_lib, tmp_path, seed):
    rng = random.Random(seed)
    kw = random_world_arguments(rng)
    assert run_one(worlds, "random%d" % seed, kw, cuda_lib, 6, str(tmp_path)), kw


if __name__ == "__main__":
    import tempfile
    rng = random.Random(int(sys.argv[1]) if len(sys.argv) > 1 else 1)
    with tempfile.TemporaryDirectory() as d:
        cache = worldutil.WorldCache(d); bad = 0
        for k in range(int(sys.argv[2]) if len(sys.argv) > 2 else 10):
            kw = random_world_arguments(rng)
            ok = run_one(cache, "w%d" % k, kw, _build.build_hostsim(), rng.choice([1, 3, 6]), d)
            print(k, "identical" if ok else "DIFFERENT", kw, flush=True); bad += not ok
        sys.exit(1 if bad else 0)
