"""Test infrastructure: synthetic worlds, the reference's results on them, and conversion of oracle dumps into C-ABI inputs.

The tests compare the product with the unmodified reference. What they compare against is committed in tests/golden/reference_runs.json:
for every reference run the suite makes, keyed by the bytes of its input files and its arguments, the exit code, the ERROR lines, SHA-256
digests of both output files and the digests / values of the stage dumps the tests look at. The suite reads that record and never needs the
reference. Where the reference is built (oracle/_ref/arriba, see oracle/Makefile), `ARB_RECORD_REFERENCE=1 pytest -m "not gpu" tests` runs it
instead and writes the record again; the CPU tests then check the product against the fresh runs while they record them."""
import atexit, os, subprocess, hashlib, json, shutil, tempfile
import numpy as np
import arbdump
from arriba_b200 import _build

NT16 = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}
INTERESTING = set([str(i) for i in range(1, 23)] + ["X", "Y"])

# small, feature-dense default world (seconds for the oracle)
SMALL = dict(scale=0.001, genes=400, breakpoints=200, fragments=20000, read_length=101)

RECORD_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.json")
RECORDING = os.environ.get("ARB_RECORD_REFERENCE") == "1"


def digest(a):
    """SHA-256 (80 bits) of an array's values, independent of its integer width; floats by their bit patterns."""
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = a.view(np.uint32 if a.itemsize == 4 else np.uint64)
    return hashlib.sha256(np.ascontiguousarray(a.astype(np.int64)).ravel().tobytes()).hexdigest()[:20]


def file_digest(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 22), b""):
            h.update(block)
    return h.hexdigest()


class _Record:
    """tests/golden/reference_runs.json: run key -> {fact name: value}. Recording rewrites it with the runs this session made."""
    def __init__(self):
        self.runs = None; self.fresh = {}

    def get(self, key):
        if RECORDING:
            if not self.fresh:
                atexit.register(self.save)
            return self.fresh.setdefault(key, {})
        if self.runs is None:
            self.runs = json.load(open(RECORD_PATH)) if os.path.exists(RECORD_PATH) else {}
        if key not in self.runs:
            raise KeyError("no recorded reference run for these inputs (%s); record one with ARB_RECORD_REFERENCE=1 where oracle/_ref/arriba is built" % key)
        return self.runs[key]

    def save(self):
        old = json.load(open(RECORD_PATH)) if os.path.exists(RECORD_PATH) else {}
        old.update(self.fresh)
        with open(RECORD_PATH, "w") as f:
            json.dump(old, f, indent=0, sort_keys=True, separators=(",", ":"))
            f.write("\n")


RECORD = _Record()


def run_key(files, args, kind="run"):
    h = hashlib.sha256(json.dumps([kind, list(args)]).encode())
    for path in files:
        h.update(file_digest(path).encode())
    return h.hexdigest()[:24]


def reference_cli(bam, gtf, fa, args, det_alloc=False):
    """The reference's command line on these files: (exit code, its ERROR lines, {output file: sha256} when it succeeded)."""
    rec = RECORD.get(run_key((bam, gtf, fa), args, "cli"))
    if "rc" not in rec:
        if not RECORDING:
            raise KeyError("incomplete reference record")
        with tempfile.TemporaryDirectory() as d:
            env = dict(os.environ, ARB_DET_ALLOC="1") if det_alloc else None
            r = subprocess.run([_build.build_oracle(), "-x", bam, "-g", gtf, "-a", fa, "-o", d + "/o.tsv", "-O", d + "/d.tsv"] + list(args),
                               capture_output=True, text=True, env=env, timeout=900)
            rec["rc"] = r.returncode; rec["errors"] = [l for l in r.stderr.split("\n") if l.startswith("ERROR")]
            rec["sha"] = {"fusions.tsv": file_digest(d + "/o.tsv"), "fusions.discarded.tsv": file_digest(d + "/d.tsv")} if r.returncode == 0 else None
    return rec["rc"], rec["errors"], rec["sha"]


def run_synth(prefix, seed=0xA881BA, scale=0.001, genes=400, breakpoints=200, fragments=20000, read_length=101, extra=()):
    synth = _build.build_tools()
    cmd = [synth, "--prefix", prefix, "--seed", str(seed), "--scale", str(scale), "--genes", str(genes), "--breakpoints", str(breakpoints),
           "--fragments", str(fragments), "--read-length", str(read_length)] + list(extra)
    subprocess.run(cmd, check=True, stderr=subprocess.DEVNULL)


def run_oracle(prefix, outdir, dump=True, det_alloc=True, args=("-f", "blacklist"), level=2):
    oracle = _build.build_oracle()
    os.makedirs(outdir, exist_ok=True)
    env = dict(os.environ)
    if dump:
        d = os.path.join(outdir, "dump"); os.makedirs(d, exist_ok=True)
        env["ARB_DUMP_DIR"] = d; env["ARB_DUMP_LEVEL"] = str(level)
    if det_alloc:
        env["ARB_DET_ALLOC"] = "1"
    cmd = [oracle, "-x", prefix + ".bam", "-g", prefix + ".gtf", "-a", prefix + ".fa", "-o", os.path.join(outdir, "fusions.tsv"),
           "-O", os.path.join(outdir, "fusions.discarded.tsv")] + list(args)
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    with open(os.path.join(outdir, "stdout.txt"), "w") as f:
        f.write(r.stdout)
    with open(os.path.join(outdir, "stderr.txt"), "w") as f:
        f.write(r.stderr)
    if r.returncode != 0:
        raise RuntimeError("oracle failed: " + r.stderr[-2000:])
    return outdir


class World:
    """The input files at `prefix` and the reference's run on them (with stage dumps). `fact(name, compute)` is what the tests compare
    against: recorded, or, while recording, compute(self) over the oracle's dumps and output files in `outdir`."""
    def __init__(self, prefix, outdir=None, args=("-f", "blacklist")):
        self.prefix = prefix; self.outdir = outdir
        self.key = run_key((prefix + ".bam", prefix + ".gtf", prefix + ".fa"), args)
        self._dumps = None; self._fasta = None

    def fact(self, name, compute):
        rec = RECORD.get(self.key)
        if name not in rec:
            if not RECORDING:
                raise KeyError("the reference record of %s has no %r; record it with ARB_RECORD_REFERENCE=1 where oracle/_ref/arriba is built" % (self.key, name))
            rec[name] = compute(self)
        return rec[name]

    def stage_digest(self, name, column, occurrence=0):
        return self.fact("%s/%d/%s" % (name, occurrence, column), lambda w: digest(w.stage(name, occurrence)[column]))

    def stage_scalar(self, name, column, occurrence=0):
        return self.fact("%s/%d/%s[0]" % (name, occurrence, column), lambda w: w.stage(name, occurrence)[column][0].item())

    def output_digest(self, filename):
        return self.fact("sha256/" + filename, lambda w: file_digest(os.path.join(w.outdir, filename)))

    def output_lines(self, filename):
        return self.fact("lines/" + filename, lambda w: len(open(os.path.join(w.outdir, filename)).read().split("\n")))

    def stderr_has(self, phrase):
        return self.fact("stderr/" + phrase, lambda w: phrase in open(os.path.join(w.outdir, "stderr.txt")).read())

    def same_output(self, filename, path):
        """the file at `path` is byte for byte the reference's `filename`"""
        return file_digest(path) == self.output_digest(filename)

    @property
    def dumps(self):
        if self._dumps is None:
            self._dumps = arbdump.read_dir(os.path.join(self.outdir, "dump"))
        return self._dumps

    def stage(self, name, occurrence=0):
        return arbdump.stage(self.dumps, name, occurrence)

    @property
    def fasta(self):
        if self._fasta is None:
            self._fasta = read_fasta(self.prefix + ".fa")
        return self._fasta


def reference_world(prefix, outdir, args=("-f", "blacklist")):
    """The reference's run on the files at `prefix` (run only while recording)."""
    if RECORDING:
        run_oracle(prefix, outdir, args=args)
    return World(prefix, outdir, args)


class WorldCache:
    def __init__(self, root):
        self.root = root; self.cache = {}

    def get(self, name="small", oracle_args=("-f", "blacklist"), **kw):
        params = dict(SMALL); params.update(kw)
        key = name + "_" + hashlib.md5(json.dumps([params, list(oracle_args)], sort_keys=True, default=str).encode()).hexdigest()[:10]
        if key not in self.cache:
            d = os.path.join(self.root, key); os.makedirs(d, exist_ok=True)
            prefix = os.path.join(d, "w")
            extra = params.pop("extra", ())
            run_synth(prefix, extra=extra, **params)
            self.cache[key] = reference_world(prefix, os.path.join(d, "oracle"), oracle_args)
        return self.cache[key]


def read_fasta(path):
    names, seqs = [], []
    cur = []
    with open(path, "rb") as f:
        for line in f:
            if line.startswith(b">"):
                if names:
                    seqs.append(b"".join(cur).upper())
                names.append(line[1:].split()[0].decode()); cur = []
            else:
                cur.append(line.strip())
    seqs.append(b"".join(cur).upper())
    return names, seqs


def strip_chr(name):
    if name.startswith("chr"):
        name = name[3:]
    return "MT" if name == "M" else name


def contigs_from_world(world):
    """contig id = order of first appearance (assembly first), as in the reference (assembly.cpp:42-44)."""
    names, seqs = world.fasta
    flags = np.array([1 if strip_chr(n) in INTERESTING else 0 for n in names], np.uint8)
    return names, flags, seqs


def chunk_from_dump(d):
    """oracle fragment dump (stage `annotated`) -> arb_soa_chunk arrays."""
    n = len(d["n_aln"])
    aln_off = d["aln_off"].astype(np.int64)
    A = int(aln_off[-1])
    frag_of = np.repeat(np.arange(n), np.diff(aln_off))
    slot_of = np.arange(A) - aln_off[frag_of]
    dst = slot_of * n + frag_of
    ch = {"n_fragments": n, "n_aln": d["n_aln"].copy(), "filter": np.zeros(n, np.uint8),
          "fflags": (d["single_end"] | d["multimapper"] << 1 | d["duplicate"] << 2).astype(np.uint8)}
    if "names" in d and "name_off" in d:   # bit 3: same read name (up to the last comma) as the fragment before it
        blob = bytes(d["names"]); off = d["name_off"].astype(np.int64)
        stems = [blob[off[i]:off[i + 1]].rpartition(b",")[0] or blob[off[i]:off[i + 1]] for i in range(n)]
        same = np.array([i > 0 and stems[i] == stems[i - 1] for i in range(n)], bool)
        ch["fflags"] |= (same.astype(np.uint8) << 3)
    def slot_array(src, dtype):
        out = np.zeros(3 * n, dtype); out[dst] = src; return out
    ch["contig"] = slot_array(d["contig"], np.uint16); ch["start"] = slot_array(d["start"], np.int32); ch["end"] = slot_array(d["end"], np.int32)
    af = (d["supplementary"] | d["first_in_pair"] << 1 | d["exonic"] << 2 | d["strand"] << 3 | d["predicted_strand"] << 4 | d["predicted_strand_ambiguous"] << 5)
    ch["aflags"] = slot_array(af, np.uint8)
    ch["cigar_off"] = slot_array(d["cigar_off"][:-1], np.uint32); ch["cigar_cnt"] = slot_array(np.diff(d["cigar_off"].astype(np.int64)), np.uint16)
    ch["cigar"] = d["cigar"].copy()
    ch["genes_off"] = slot_array(d["genes_off"][:-1], np.uint32); ch["genes_cnt"] = slot_array(np.diff(d["genes_off"].astype(np.int64)), np.uint16)
    ch["genes"] = d["genes"].copy() if len(d["genes"]) else np.zeros(1, np.uint32)
    # sequences: ASCII -> nt16 nibbles, each sequence 16-byte aligned; slots 0 and 1 only
    seq_off_src = d["seq_off"].astype(np.int64)
    lens = np.diff(seq_off_src)
    seq_len = slot_array(lens, np.uint32)
    assert np.all(seq_len[2 * n:] == 0), "supplementary alignments carry no sequence"
    lut = np.full(256, 15, np.uint8)
    for c, v in NT16.items():
        lut[ord(c)] = v
    codes = lut[d["seq"]]
    nbytes16 = ((lens + 1) // 2 + 15) // 16
    start16 = np.concatenate([[0], np.cumsum(nbytes16)])
    total = int(start16[-1]) * 16
    packed = np.zeros(total + 16, np.uint8)
    # position of every base
    base_aln = np.repeat(np.arange(A), lens)
    base_pos = np.arange(len(codes)) - seq_off_src[base_aln]
    byte_idx = start16[base_aln] * 16 + base_pos // 2
    hi = (base_pos % 2) == 0
    np.add.at(packed, byte_idx[hi], codes[hi] << 4)
    np.add.at(packed, byte_idx[~hi], codes[~hi])
    so = np.zeros(3 * n, np.uint32); so[dst] = start16[:-1]
    ch["seq_off"] = so[:2 * n].copy(); ch["seq_len"] = seq_len[:2 * n].astype(np.uint16); ch["seq"] = packed
    return ch


def annotation_from_dump(fl, n_contigs):
    """oracle gene/exon dump (stage `fragment_length`, level 2) -> arb_annotation arrays."""
    a = {"n_genes": len(fl["gene_id"]), "n_contigs": n_contigs}
    assert np.all(fl["gene_id"] == np.arange(a["n_genes"]))
    a["gene_contig"] = fl["gene_contig"]; a["gene_start"] = fl["gene_start"]; a["gene_end"] = fl["gene_end"]; a["gene_strand"] = fl["gene_strand"]
    a["gene_exonic_length"] = fl["gene_exonic_length"]; a["gene_flags"] = (fl["gene_is_dummy"] | fl["gene_is_protein_coding"] << 1).astype(np.uint8)
    ne = len(fl["exon_gene"]); a["n_exons"] = ne
    a["exon_gene"] = fl["exon_gene"]; a["exon_start"] = fl["exon_start"]; a["exon_end"] = fl["exon_end"]
    a["exon_cds_start"] = fl["exon_cds_start"]; a["exon_cds_end"] = fl["exon_cds_end"]
    nxt = fl["exon_next"]; a["exon_next_start"] = np.where(nxt >= 0, fl["exon_start"][np.maximum(nxt, 0)], -1).astype(np.int32)
    a["exon_flags"] = ((fl["exon_prev"] >= 0).astype(np.uint8) | (nxt >= 0).astype(np.uint8) << 1)
    rc = fl["region_contig"].astype(np.int64)
    a["exon_region_begin"] = np.searchsorted(rc, np.arange(n_contigs + 1)).astype(np.uint32)
    a["exon_region_end"] = fl["region_end"]; a["exon_region_off"] = fl["region_off"]
    a["exon_region_items"] = fl["region_exons"] if len(fl["region_exons"]) else np.zeros(1, np.uint32)
    # the gene index is not needed by the device stages under test
    a["gene_region_begin"] = np.zeros(n_contigs + 1, np.uint32); a["gene_region_end"] = np.zeros(1, np.int32)
    a["gene_region_off"] = np.zeros(1, np.uint32); a["gene_region_items"] = np.zeros(1, np.uint32)
    return a


def _segments(data, starts, counts):
    """concatenation of data[starts[i]:starts[i] + counts[i]] over i"""
    starts = np.asarray(starts, np.int64); counts = np.asarray(counts, np.int64)
    total = int(counts.sum())
    if total == 0:
        return np.zeros(0, np.int64)
    return np.asarray(data)[np.arange(total) + np.repeat(starts - (np.cumsum(counts) - counts), counts)]


def fragment_digests(t, names, name_off, check_genes, check_pred):
    """Digests of a fragment table in arb_soa_chunk layout (Pipeline.fragments() or chunk_from_dump()): the fields of the alignments that exist,
    CIGARs, sequences and gene sets alignment by alignment, whatever offsets the variable-length parts sit at."""
    n = int(t["n_fragments"])
    valid = (t["n_aln"][None, :] > np.arange(3)[:, None]).ravel()
    mask = 0b001011 | (0b000100 if check_genes else 0) | (0b100000 if check_pred else 0)
    out = {"n": n, "names": digest(np.frombuffer(names, np.uint8)), "name_off": digest(name_off), "n_aln": digest(t["n_aln"]), "fflags": digest(t["fflags"])}
    for k in ("contig", "start", "end", "cigar_cnt"):
        out[k] = digest(t[k][valid])
    out["aflags"] = digest(t["aflags"][valid] & mask)
    if check_pred:   # the predicted strand only where it is not ambiguous
        out["predicted_strand"] = digest(t["aflags"][valid & ((t["aflags"] & 32) == 0)] & 16)
    out["cigar"] = digest(_segments(t["cigar"], t["cigar_off"][valid], t["cigar_cnt"][valid]))
    v2 = valid[:2 * n]
    lens = t["seq_len"][v2].astype(np.int64)
    out["seq_len"] = digest(lens)
    out["seq"] = digest(_segments(t["seq"], t["seq_off"][v2].astype(np.int64) * 16, (lens + 1) // 2))
    if check_genes:
        out["genes_cnt"] = digest(t["genes_cnt"][valid])
        out["genes"] = digest(_segments(t["genes"], t["genes_off"][valid], t["genes_cnt"][valid]))
    return out


def frag_tables_equal(got, world, stage, check_genes, check_pred):
    """got: Pipeline.fragments(); the reference's fragment table of dump stage `stage` (ingest / annotated)."""
    def ref(w):
        d = w.stage(stage)
        return fragment_digests(chunk_from_dump(d), bytes(d["names"]), d["name_off"], check_genes, check_pred)
    want = world.fact("fragments/%s/%d%d" % (stage, check_genes, check_pred), ref)
    mine = fragment_digests(got, got["names_blob"], got["name_off"], check_genes, check_pred)
    bad = [k for k in want if mine[k] != want[k]]
    assert not bad, "fragment table differs from the reference's (%s) in %s" % (stage, bad)


def front_end(world, lib_path, threads=4, device=0):
    """Pipeline on the world's files up to the upload of the fragment table, whose annotated fragments are checked to be the reference's:
    the device stages after it start from the reference's input."""
    from arriba_b200 import lib as L
    p = L.Pipeline(world.prefix + ".bam", world.prefix + ".gtf", world.prefix + ".fa", threads=threads, device=device, lib_path=lib_path)
    for s in (L.STEP_LOAD_REFERENCE, L.STEP_INGEST, L.STEP_ANNOTATE):
        p.step(s)
    frag_tables_equal(p.fragments(), world, "annotated", check_genes=True, check_pred=True)
    p.step(L.STEP_UPLOAD)
    return p
