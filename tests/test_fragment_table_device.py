"""The fragment table that ingest builds on the device from its workers' pools (csrc/fragtable.cu): slot normalisation, name order, pool offsets and
multimapper flags. The name sort compares the first 16 name bytes in one radix sort and settles ties 8 bytes at a time, so the worlds here rename the
reads of a synthetic world: Illumina-style names that share their first 18 or 29 bytes (ties past 16 and past 24 bytes), and names that are prefixes of
one another ("r1" / "r10" / "r100": "r1,1" sorts before "r10,1"). The fragment table and both output files must be the reference's."""
import ctypes as C
import json, os, random
import pytest
import bamtools, worldutil
from test_ingest import check_front_end
from test_e2e import check_e2e
from arriba_b200 import lib as L

# the reference's runs on these worlds, kept apart from tests/golden/reference_runs.json
RUNS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs_fragment_table.json")
STYLES = {"illumina18": b"NB551234:99:HX2:1:", "illumina29": b"A00123:456:HGFKJDSXY:1:1101:", "nested": b"r"}


def renamed_world(worlds, root, style):
    base = worlds.get("small")
    d = os.path.join(str(root), "renamed_" + style); os.makedirs(d, exist_ok=True)
    prefix = os.path.join(d, "w")
    for ext in (".fa", ".gtf"):
        if not os.path.exists(prefix + ext):
            os.symlink(base.prefix + ext, prefix + ext)
    if not os.path.exists(prefix + ".bam"):
        text, refs, bodies = bamtools.read_bam(base.prefix + ".bam")
        names, out = {}, []
        for b in bodies:
            r = bamtools.split_record(b)
            q = r["qname"]
            if q not in names:
                k = len(names) + 1
                names[q] = STYLES[style] + (b"%d" % k if style == "nested" else b"%d:%d" % (1000 + k % 977, 2000 + k))
            r["qname"] = names[q] + b"\0"
            out.append(bamtools.join_record(r))
        assert len(names) > 1000
        bamtools.write_bam(prefix + ".bam", text, refs, out, random.Random(11))
    return worldutil.reference_world(prefix, os.path.join(d, "oracle"))


@pytest.fixture(scope="module")
def renamed(worlds, tmp_path_factory):
    rec = worldutil.RECORD
    if not worldutil.RECORDING:
        if rec.runs is None:
            rec.runs = json.load(open(worldutil.RECORD_PATH)) if os.path.exists(worldutil.RECORD_PATH) else {}
        rec.runs.update(json.load(open(RUNS)))
    root = tmp_path_factory.mktemp("renamed")
    out = {style: renamed_world(worlds, root, style) for style in STYLES}
    yield out
    if worldutil.RECORDING:   # what this module recorded goes to its own file, not to the shared record
        mine = {w.key: rec.fresh.pop(w.key) for w in out.values() if w.key in rec.fresh}
        with open(RUNS, "w") as f:
            json.dump(mine, f, indent=0, sort_keys=True, separators=(",", ":"))
            f.write("\n")


def tie_rounds(world, lib_path, threads):
    """rounds of the name sort past the first 16 bytes when this world is ingested"""
    p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, lib_path=lib_path)
    p.step(L.STEP_LOAD_REFERENCE); p.step(L.STEP_INGEST)
    lib = L.load(lib_path)
    lib.arb_fragment_table_tie_rounds.restype = C.c_uint32; lib.arb_fragment_table_tie_rounds.argtypes = [C.c_void_p]
    rounds = lib.arb_fragment_table_tie_rounds(p.context().h)
    p.close()
    return rounds


@pytest.mark.parametrize("style,threads", [("illumina18", 3), ("illumina29", 1), ("nested", 4)])
def test_front_end_hostsim_renamed(renamed, hostsim_lib, style, threads):
    check_front_end(renamed[style], hostsim_lib, threads=threads)


def test_tie_rounds_hostsim(renamed, hostsim_lib):
    """names tied past 16 bytes go through the tie loop; tied over 29 bytes, for more than one round"""
    assert tie_rounds(renamed["illumina29"], hostsim_lib, 3) >= 2
    assert tie_rounds(renamed["illumina18"], hostsim_lib, 3) >= 1


def test_front_end_hostsim_renamed_many_workers_small_chunks(renamed, hostsim_lib, monkeypatch):
    monkeypatch.setenv("ARB_CHUNK_BYTES", "60000")
    check_front_end(renamed["illumina29"], hostsim_lib, threads=11)


@pytest.mark.parametrize("style", sorted(STYLES))
def test_e2e_hostsim_renamed(renamed, hostsim_lib, tmp_path, style):
    check_e2e(renamed[style], hostsim_lib, tmp_path, threads=3)


@pytest.mark.gpu
@pytest.mark.parametrize("style", sorted(STYLES))
def test_front_end_cuda_renamed(renamed, cuda_lib, style):
    check_front_end(renamed[style], cuda_lib, threads=8)


@pytest.mark.gpu
def test_tie_rounds_cuda(renamed, cuda_lib):
    assert tie_rounds(renamed["illumina29"], cuda_lib, 8) >= 2


@pytest.mark.gpu
def test_front_end_cuda_renamed_many_workers_small_chunks(renamed, cuda_lib, monkeypatch):
    monkeypatch.setenv("ARB_CHUNK_BYTES", "60000")
    check_front_end(renamed["illumina29"], cuda_lib, threads=16)


@pytest.mark.gpu
@pytest.mark.parametrize("style", sorted(STYLES))
def test_e2e_cuda_renamed(renamed, cuda_lib, tmp_path, style):
    check_e2e(renamed[style], cuda_lib, tmp_path, threads=8)
