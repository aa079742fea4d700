#!/usr/bin/env python
"""bench.py -- chimeric fragments per second of the hot path, end to end (BAM ingest -> fusions.tsv + fusions.discarded.tsv).

One "step" = one pass of the whole path over one synthetic chimeric BAM (default: BASELINE.json configs[1], 10 M fragments, 2x101 bp,
50 k breakpoints; the genome is a synthetic stand-in for hg38 at 1:10 scale because no reference genome exists offline).
  value / e2e   : fragments/s through the public Pipeline API, BAM file on disk -> both TSV files on disk (host decode, pinned H2D, kernels,
                  D2H of the results, host event logic, writer) -- what the metric names
  device_stages : fragments/s of the device-resident stages alone (CUDA events), as an explanation of the above, never the headline
  roofline      : the time-dominant kernel of the step (and the others, under "kernels")
  --impl reference : the unmodified reference (oracle/_ref/arriba) on the host cores, bounded sample of the same world
N > 1 (torchrun): --mode sharded (default) = ONE sample divided over the ranks (strong scaling); --mode samples = one sample per GPU (weak).
The last line of stdout is the JSON line. See DESIGN.md section "Measurement"."""
import argparse, json, os, subprocess, sys, time, threading, hashlib, re

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: synth parameters (tools/synth.cpp)
    "cfg2_10M_2x101_50k": dict(scale=0.1, genes=20000, breakpoints=50000, fragments=10000000, read_length=101),
    "cfg3_15M_2x151_75k": dict(scale=0.1, genes=20000, breakpoints=75000, fragments=15000000, read_length=151),
    "cfg5_10M_mismapper": dict(scale=0.1, genes=20000, breakpoints=50000, fragments=10000000, read_length=101, extra=["--mismapper-frac", "0.3", "--paralog-frac", "0.15"]),
    "mid_1M_2x101_5k": dict(scale=0.02, genes=4000, breakpoints=5000, fragments=1000000, read_length=101),
    "mid5_1M_mismapper": dict(scale=0.02, genes=4000, breakpoints=5000, fragments=1000000, read_length=101, extra=["--mismapper-frac", "0.3", "--paralog-frac", "0.15"]),
    "tiny_20k": dict(scale=0.001, genes=400, breakpoints=200, fragments=20000, read_length=101),
}
UNIT = "reads/s"   # chimeric fragments per second
SCOPE = "ingest..fusions.tsv"  # one step = BAM ingest -> read filters -> candidates -> event filters -> fusions.tsv + discarded.tsv (reference loading excluded)
GOLDEN_MD5 = os.path.join(ROOT, "tests", "golden", "full_size_md5.json")   # md5 of the reference's two output files per workload (tests/golden/make_full_size_md5.py)


def world_dir(name):
    base = os.environ.get("ARB_BENCH_DIR", "/tmp/arb_bench")
    return os.path.join(base, name)


def ensure_world(name, sample_breakpoints=None):
    """Generates (once) the synthetic world; returns the file prefix. A sample shares genome/GTF and keeps the per-breakpoint depth."""
    from arriba_b200 import _build
    synth = _build.build_tools()
    p = WORKLOADS[name]
    d = world_dir(name); os.makedirs(d, exist_ok=True)
    prefix = os.path.join(d, "w")
    common = [synth, "--seed", str(0xA881BA), "--scale", str(p["scale"]), "--genes", str(p["genes"]), "--breakpoints", str(p["breakpoints"]),
              "--fragments", str(p["fragments"]), "--read-length", str(p["read_length"])] + p.get("extra", [])
    if not os.path.exists(prefix + ".done"):
        subprocess.run(common + ["--prefix", prefix], check=True, stderr=subprocess.DEVNULL)
        open(prefix + ".done", "w").write("ok")
    if sample_breakpoints is None:
        return prefix
    sp = os.path.join(d, "sample%d" % sample_breakpoints)
    if not os.path.exists(sp + ".done"):
        subprocess.run(common + ["--prefix", sp, "--reads-only", "--emit-breakpoints", str(sample_breakpoints)], check=True, stderr=subprocess.DEVNULL)
        for ext in (".fa", ".gtf"):
            if not os.path.exists(sp + ext):
                os.symlink(prefix + ext, sp + ext)
        open(sp + ".done", "w").write("ok")
    return sp


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    def __init__(self, device):
        super().__init__(daemon=True); self.device = device; self.samples = []; self.stop_flag = False
    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q, "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)
    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None, "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def md5_of(path):
    h = hashlib.md5()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 24), b""):
            h.update(block)
    return h.hexdigest()


def reference_run(prefix, threads):
    """Runs the unmodified reference CLI; returns (fragments, seconds over SCOPE, total seconds). The reference flushes every progress line (arriba.cpp:124-612):
    SCOPE runs from the arrival of "Reading chimeric alignments" to the arrival of "Freeing resources" on its stdout, taken with this process's clock (the
    reference's own time stamps have 1 s resolution)."""
    from arriba_b200 import _build
    oracle = _build.build_oracle()
    out = prefix + ".ref_out"
    os.makedirs(out, exist_ok=True)
    cmd = [oracle, "-x", prefix + ".bam", "-g", prefix + ".gtf", "-a", prefix + ".fa", "-o", os.path.join(out, "fusions.tsv"), "-O", os.path.join(out, "discarded.tsv"), "-f", "blacklist", "-@", str(threads)]
    with open(os.path.join(out, "stderr.txt"), "wb") as err:   # thousands of per-row warnings: to a file, a pipe nobody drains would stall the run
        t0 = time.perf_counter()
        proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=err)
        fd = proc.stdout.fileno(); text = b""; t_start = t_end = None
        while True:
            piece = os.read(fd, 1 << 16)
            now = time.perf_counter()
            if not piece:
                break
            text += piece
            if t_start is None and b"Reading chimeric alignments" in text:
                t_start = now
            if t_end is None and b"Freeing resources" in text:
                t_end = now
        rc = proc.wait()
        total = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError("reference run failed: " + open(os.path.join(out, "stderr.txt"), errors="replace").read()[-500:])
    n = int(re.search(r"\(total=(\d+)\)", text.decode(errors="replace")).group(1))
    if t_start is None:
        raise RuntimeError("reference run printed no progress lines")
    scope_s = (t_end if t_end is not None else t0 + total) - t_start
    return n, scope_s, total


# full-size run of the unmodified reference on the default workload, measured once on the development container (profiles/cfg2_full_size_parity.txt):
# the sample above flatters the reference (its std::map / unordered_map walks get slower per fragment as the containers grow)
REFERENCE_FULL_SIZE = {"cfg2_10M_2x101_50k": {"fragments": 11810114, "seconds": 1535.0, "value": 11810114 / 1535.0, "cores": 1, "where": "development container, profiles/cfg2_full_size_parity.txt (25 min 35 s)"},
                       "cfg5_10M_mismapper": {"fragments": 11732540, "seconds": 968.0, "value": 11732540 / 968.0, "cores": 1, "where": "development container, tests/golden/full_size_md5.json (16 min 8 s)"},
                       "cfg3_15M_2x151_75k": {"fragments": 17587876, "seconds": None, "value": None, "cores": 1, "where": "development container: stopped after 3 h 1 min of CPU time inside filter_mismappers, not finished (profiles/r02z/full_size_host_parity.txt)"}}


CANDIDATE_COLUMNS = ("gene1", "gene2", "contig1", "contig2", "breakpoint1", "breakpoint2", "direction1", "direction2", "split_reads1", "split_reads2", "discordant_mates",
                     "filter", "evalue", "confidence", "order")
DUMP_ROWS = 1 << 18   # 18 arrays (columns and row indexes) of at most 2^18 float64 values: 36 MB, under 64 MB


def step_outputs(p):
    """What a caller of the Pipeline receives after a step: the candidate table (one array per column) and the final label of every fragment."""
    c = p.candidates()
    out = {"candidates." + k: c[k] for k in CANDIDATE_COLUMNS}
    out["fragments.label"] = c["labels"]
    return out


def write_outputs(d, outputs):
    """DIR/<table>.<column>.npy in float64; a table longer than DUMP_ROWS is sampled at rows chosen by a fixed seed (DIR/<table>.rows.npy)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    rows = {}
    for name, a in sorted(outputs.items()):
        table = name.split(".")[0]
        a = np.asarray(a)
        if len(a) > DUMP_ROWS:
            if table not in rows:
                rows[table] = np.sort(np.random.default_rng(0).choice(len(a), DUMP_ROWS, replace=False))
                np.save(os.path.join(d, table + ".rows.npy"), rows[table].astype(np.float64))
            a = a[rows[table]]
        np.save(os.path.join(d, name + ".npy"), a.astype(np.float64))


class QuietStderr:
    """The library prints the reference's per-row warnings on stderr (thousands per step on the synthetic GTF). They go to a log file; the few progress
    lines of this script go to the real stderr."""
    def __init__(self, path):
        self.path = path; self.saved = None
    def __enter__(self):
        sys.stderr.flush()
        self.saved = os.dup(2)
        fd = os.open(self.path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
        os.dup2(fd, 2); os.close(fd)
        self.real = os.fdopen(os.dup(self.saved), "w")
        return self
    def say(self, text):
        self.real.write(text + "\n"); self.real.flush()
    def __exit__(self, *a):
        sys.stderr.flush()
        os.dup2(self.saved, 2); os.close(self.saved); self.real.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2_10M_2x101_50k", choices=sorted(WORKLOADS))
    ap.add_argument("--threads", type=int, default=0, help="host threads per rank (0 = 2 per usable CPU / ranks)")
    ap.add_argument("--sample-breakpoints", type=int, default=0, help="cpu baseline sample size in breakpoints (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="N>1: skip the additional line of the other multi-GPU mode")
    ap.add_argument("--mode", choices=["samples", "sharded"], default="sharded",
                    help="N>1: 'sharded' = ONE sample divided over the ranks (strong scaling, NCCL exchanges); 'samples' = one independent sample per GPU (weak scaling, no collective)")
    ap.add_argument("--no-parity", action="store_true", help="skip the md5 comparison of the output files with the reference's")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (candidate table, fragment labels) as DIR/<name>.npy, float64, "
                                                            "a fixed sample of rows where the table exceeds 64 MB; the inputs are the same from run to run")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1
    usable = cores   # CPUs the container may actually burn: the cgroup quota, where one is set (the 1-GPU boxes show 128 CPUs and grant 16)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            usable = min(cores, max(1.0, float(quota) / float(period)))
    except Exception:
        pass
    threads_all = args.threads or max(2, min(64, int(round(2 * usable))))                 # 2 threads per usable CPU measured best (profiles/r01i)
    threads = args.threads or max(2, min(64, int(round(2 * usable / max(1, world)))))   # one sample per rank: the ranks share the host
    wl = WORKLOADS[args.workload]
    sample_bp = args.sample_breakpoints or max(50, int(wl["breakpoints"] * 400000 / wl["fragments"]))  # ~400 k fragments: 10-30 s of reference CPU time
    metric = "chimeric reads/sec end-to-end (ingest→fusions.tsv)"   # BASELINE.json; a "read" is one chimeric fragment (read pair + supplementary), the unit the reference counts
    config = {"workload": "synthetic %s: %d fragments 2x%d bp, %d breakpoints, genome %.0f%% of hg38 size (synthetic), %d genes" %
              (args.workload, wl["fragments"], wl["read_length"], wl["breakpoints"], wl["scale"] * 100, wl["genes"]),
              "scope": SCOPE, "value_is": "end to end: BAM on disk -> both TSV files on disk through the public Pipeline API, host<->device copies inside the timed region",
              "l2": "inputs (>2 GB of SoA columns per step) exceed the 126 MB L2", "host_threads_per_rank": threads, "host_threads_rank0_sharded": threads_all, "host_cpus_usable": usable}

    if args.impl == "reference":
        if rank != 0:
            return
        prefix = ensure_world(args.workload, sample_bp)
        vals = []
        for _ in range(max(1, min(args.steps, 2))):  # one reference pass takes tens of seconds
            n, scope_s, total = reference_run(prefix, cores)
            vals.append((n / scope_s, n, scope_s, total))
        v, n, scope_s, total = max(vals)
        line = {"impl": "reference", "metric": metric, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals), "warmup": 0, "ms_per_step": scope_s * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "reference",
                                 "sample": "first %d breakpoints of the workload at full depth = %d fragments; arrival times of the reference's own progress lines over %s; decode threads -@ %d have no effect in the shim build" % (sample_bp, n, SCOPE, cores),
                                 "full_size": REFERENCE_FULL_SIZE.get(args.workload)},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    import torch
    from arriba_b200 import lib as L, _build
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU reference")
    if not os.path.exists(_build.PRODUCT_LIB):
        _build.build_product()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if rank == 0:
        prefix = ensure_world(args.workload)
    if dist:
        dist.barrier()
    prefix = ensure_world(args.workload)
    outdir = os.path.join(world_dir(args.workload), "out_rank%d" % rank); os.makedirs(outdir, exist_ok=True)
    out_tsv, out_disc = os.path.join(outdir, "fusions.tsv"), os.path.join(outdir, "fusions.discarded.tsv")
    quiet = QuietStderr(os.path.join(outdir, "library_stderr.log")); quiet.__enter__()
    say = (lambda s: quiet.say(s)) if rank == 0 else (lambda s: None)

    def one_step(sharded, capture=False):
        """ingest .. fusions.tsv through the public Pipeline API; returns a dict of what the step measured (and, with capture, of what it computed)"""
        # one sample divided over the ranks: rank 0 does the host work with all host threads, the others only hold a device context
        p = L.Pipeline(prefix + ".bam", prefix + ".gtf", prefix + ".fa", threads=(threads_all if rank == 0 else 2) if sharded else threads, device=local_rank, output=out_tsv, discarded=out_disc)
        if not sharded or rank == 0:
            p.step(L.STEP_LOAD_REFERENCE)      # genome + annotation: loaded once per run in a real deployment, outside the timed region
        if rank == 0 or not sharded:   # a run writes NEW files: the previous step's outputs go before the clock starts (truncating 900 MB of cached pages is not part of a run)
            for f in (out_tsv, out_disc):
                try:
                    os.remove(f)
                except OSError:
                    pass
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if sharded:
            from arriba_b200 import sharded as S
            S.run_sharded(p, rank, world, reference_loaded=True)   # NCCL exchanges inside; rank 0 writes the files
        else:
            for s in range(L.STEP_INGEST, L.STEP_COUNT):
                p.step(s)
            p.events(len(L.EV_NAMES) - 1)          # event-level chain incl. the device stages and the D2H of the candidate table
            p.write_output()
        e2e_s = time.perf_counter() - t0
        ctx = p.context()
        st = p.stats(); tm = ctx.timings() if ctx.h else L.Timings()
        n_cand = int(st.n_candidates)
        # bytes that cross PCIe in a step, from the sizes of what is copied: up = the inflated BAM chunks (the device finds the record boundaries and deals the records to the
        # parsing threads) + the fragment table; down = the record lists, the annotation columns, candidate columns + list offsets + labels, and the text of the
        # discarded-fusions file, which the device formats (the strings of the fusions rows add a few MB)
        nf = int(st.n_fragments)
        try:
            bam_bytes = os.path.getsize(prefix + ".bam"); disc_bytes = os.path.getsize(out_disc) if (rank == 0 or not sharded) else 0
        except OSError:
            bam_bytes = disc_bytes = 0
        d2h_parts = {"record_lists": 4 * int(st.n_records), "annotation_columns": (3 + 12 + 6 + 4 * 4) * nf,   # flags, offsets, counts, ~4 gene ids per fragment
                     "candidates_lists_labels": n_cand * 46 + 3 * 4 * (n_cand + 1) + 2 * nf, "discarded_rows_text": disc_bytes}
        h2d_parts = {"bam_chunks": bam_bytes, "fragment_table": int(tm.h2d_bytes)}
        d2h = sum(d2h_parts.values())
        dev_ms = tm.annotate_ms + tm.read_filters_ms + tm.find_fusions_ms + tm.order_ms + tm.merge_adjacent_ms + tm.multimappers_ms + tm.evalue_ms + tm.in_vitro_ms + tm.kmer_index_ms + tm.homologs_ms + tm.mismappers_ms + tm.partners_ms + tm.rows_ms + tm.consensus_ms + tm.bam_scan_ms
        ev = {n: round(st.event_seconds[i], 2) for i, n in enumerate(L.EV_NAMES) if st.event_seconds[i] >= 0.2}
        say("[bench] step: e2e %.2f s, device %.1f ms, ingest %.2f, annotate %.2f, upload %.2f, output %.2f, events >= 0.2 s: %s" %
            (e2e_s, dev_ms, st.seconds[L.STEP_INGEST], st.seconds[L.STEP_ANNOTATE], st.seconds[L.STEP_UPLOAD], st.output_seconds, ev))
        outputs = step_outputs(p) if capture and rank == 0 else None   # after the clock stopped
        p.close()
        return {"n": int(st.n_fragments), "e2e_s": e2e_s, "dev_ms": dev_ms, "st": st, "tm": tm, "d2h": d2h, "n_cand": n_cand, "d2h_parts": d2h_parts, "h2d_parts": h2d_parts,
                "outputs": outputs}

    def timed(sharded, warmup, steps, capture=False):
        for _ in range(warmup):
            one_step(sharded)
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        t_begin = time.perf_counter()
        results = [one_step(sharded, capture and i == steps - 1) for i in range(steps)]
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        wall = time.perf_counter() - t_begin
        e2e_s = sum(r["e2e_s"] for r in results) / len(results)
        dev_ms = sum(r["dev_ms"] for r in results) / len(results)
        if dist:   # a step ends when its slowest rank ends
            t = torch.tensor([e2e_s, dev_ms, wall], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s, dev_ms, wall = [float(x) for x in t.tolist()]
        return results, e2e_s, dev_ms, wall

    sharded = args.mode == "sharded" and world > 1
    config["sharding"] = ("ONE sample over the ranks (strong scaling): rank 0 ingests and broadcasts its resident table over NVLink; find_fusions divided by contig pair, one NCCL all-gather of the candidate tables, filter_mismappers divided by work item (DESIGN.md section 7)" if sharded else
                          "one independent BAM per rank (weak scaling, no collective on the data path)" if world > 1 else "single GPU")
    sampler = ClockSampler(local_rank); sampler.start()
    launches1 = None
    lib = L.load()
    try:
        for _ in range(args.warmup):
            one_step(sharded)
        launches1 = lib.arb_kernel_launches()
        results, e2e_s, dev_ms, wall = timed(sharded, 0, args.steps, capture=bool(args.dump_outputs))
    except BaseException:
        import traceback
        quiet.say("bench.py (rank %d): a step failed\n%s" % (rank, traceback.format_exc()))   # on the real stderr, not in the library's log
        quiet.__exit__()
        raise
    launches = lib.arb_kernel_launches() - launches1
    sampler.stop_flag = True; sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, results[-1]["outputs"])

    # parity of the very files the timed steps wrote: md5 against the unmodified reference's output for this workload (committed; made on the CPU box)
    parity = {"checked": False}
    if rank == 0 and not args.no_parity:
        try:
            golden = json.load(open(GOLDEN_MD5)).get(args.workload)
        except Exception:
            golden = None
        if golden:
            got = {"fusions.tsv": md5_of(out_tsv), "fusions.discarded.tsv": md5_of(out_disc)}
            parity = {"checked": True, "ok": got == {k: golden[k] for k in got}, "md5": got, "reference_md5": {k: golden[k] for k in got}, "source": golden.get("source")}
        else:   # the sums of what the steps wrote are recorded all the same: the reference's run of a large workload takes hours on one core and may be compared afterwards
            parity = {"checked": False, "reason": "no committed reference md5 for this workload", "md5": {"fusions.tsv": md5_of(out_tsv), "fusions.discarded.tsv": md5_of(out_disc)}}

    secondary = None
    if dist and not args.no_secondary and e2e_s < 40.0:   # the other multi-GPU mode, a few steps
        other = not sharded
        r2, e2, d2, _ = timed(other, 1, 2)
        jobs2 = 1 if other else world
        secondary = {"mode": "sharded" if other else "samples", "scaling": "strong" if other else "weak", "value": r2[0]["n"] * jobs2 / e2, "unit": UNIT, "seconds_per_step": e2, "steps": 2, "warmup": 1,
                     "note": "ONE sample divided over all ranks" if other else "one independent sample per GPU, no collective on the data path"}
    quiet.__exit__()
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    n_frag = results[0]["n"]
    st, tm = results[-1]["st"], results[-1]["tm"]
    peak, peak_src = measured_peak()
    jobs = 1 if (sharded or world == 1) else world

    def kernel_entry(name, ms, alg_bytes, unit_note, traffic_key, l2_key=None):
        traffic = None; t = {}
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            traffic = t.get(args.workload, {}).get(traffic_key)
        except Exception:
            pass
        ach = alg_bytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        entry = {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                 "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms": ms, "algorithmic_bytes_are": unit_note}
        if l2_key:   # explanation for a gather-bound kernel: bytes its loads request from L1/L2 per launch (32-byte sectors, from the same ncu capture) over the live kernel time
            try:
                l2 = t.get(args.workload, {}).get(l2_key)
                if l2 and ms > 0:
                    entry["l1_l2_request_gbs"] = l2 / (ms * 1e-3) / 1e9
                    entry["bound_note"] = "gather bound: dependent 4-byte lookups, each a 32-byte sector; DRAM traffic ~ algorithmic bytes, the limiter is the sector rate through L1/L2"
            except Exception:
                pass
        return entry

    mean = lambda f: sum(f(r["tm"]) for r in results) / len(results)
    kernels = [
        kernel_entry("cascade_head (all coordinate / CIGAR / gene-set rules, one launch)", mean(lambda t: t.cascade_head_ms), int(tm.cascade_algorithmic_bytes[0]),
                     "SURVEY 8(d) column budget of the fragments the launch saw", "cascade_head_dram_bytes"),
        kernel_entry("cascade_sequences (mismatches + low entropy, one launch)", mean(lambda t: t.cascade_sequences_ms), int(tm.cascade_algorithmic_bytes[1]),
                     "SURVEY 8(d): sequences 3 bit/base + gathered reference 2 bit/base + CIGARs + 11 B/alignment of the queued fragments", "cascade_sequences_dram_bytes"),
        kernel_entry("mismappers pass 1 (re-alignment, one launch)", mean(lambda t: t.mismappers_pass1_ms), int(getattr(tm, "mismapper_algorithmic_bytes", 0)),
                     "SURVEY 8(d): per re-aligned sequence 3l/8 + 8(l-8) + 4*hits + l/2", "mismappers_pass1_dram_bytes", "mismappers_pass1_l2_bytes"),
    ]
    dominant = max(kernels, key=lambda k: k["kernel_ms"])
    device_ms = {"annotate": tm.annotate_ms, "order": tm.order_ms, "multimappers": tm.multimappers_ms, "in_vitro": tm.in_vitro_ms, "duplicates": tm.duplicates_ms, "classify": tm.classify_ms, "read_filters_total": tm.read_filters_ms, "find_fusions_total": tm.find_fusions_ms, "h2d": tm.h2d_ms,
                 "merge_adjacent": tm.merge_adjacent_ms, "evalue": tm.evalue_ms, "kmer_index": tm.kmer_index_ms, "homologs": tm.homologs_ms, "mismappers": tm.mismappers_ms,
                 "mismappers_pass1": tm.mismappers_pass1_ms, "mismappers_pass2": tm.mismappers_pass2_ms,
                 "partners": tm.partners_ms, "discarded_rows": tm.rows_ms, "consensus": tm.consensus_ms, "bam_scan": tm.bam_scan_ms}
    roofline = dict(dominant)
    roofline.update({"kernels": kernels, "device_ms": device_ms,
                     "mismapper_sequences": int(tm.mismapper_sequences), "mismapper_hits": int(tm.mismapper_hits),
                     "mismapper_items": int(tm.mismapper_items), "mismapper_heavy_items": int(tm.mismapper_heavy_items), "mismapper_tasks": int(tm.mismapper_tasks), "mismapper_rounds": int(tm.mismapper_rounds),
                     "mismapper_registry": {"slots": int(tm.mismapper_table_slots), "overflow": int(tm.mismapper_overflow)}, "kmer_positions": int(tm.kmer_positions), "cascade_queued": int(tm.cascade_queued)})
    line = {"metric": metric, "value": n_frag * jobs / e2e_s, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": e2e_s * 1e3, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
            "clocks": sampler.summary(),
            "e2e": {"value": n_frag * jobs / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(sum(results[-1]["h2d_parts"].values())), "d2h_bytes_per_step": int(results[-1]["d2h"]),
                    "h2d_bytes_are": results[-1]["h2d_parts"], "d2h_bytes_are": results[-1]["d2h_parts"],
                    "seconds_per_step": e2e_s, "host_seconds": {n: round(st.seconds[i], 3) for i, n in enumerate(L.STEP_NAMES) if i > 0},
                    "event_seconds": {n: round(st.event_seconds[i], 3) for i, n in enumerate(L.EV_NAMES) if st.event_seconds[i] >= 0.001}, "output_seconds": round(st.output_seconds, 3),
                    "ingest_split": {"inflate": round(st.t_inflate, 3), "parse": round(st.t_parse, 3), "finalize": round(st.t_finalize, 3)}},
            "device_stages": {"value": n_frag * jobs / (dev_ms * 1e-3), "unit": UNIT, "ms_per_step": dev_ms, "is": "sum of the CUDA-event times of the device stages, fragment table resident in HBM (not the headline)"},
            "gpu_launches": int(launches), "roofline": roofline, "parity": parity, "parity_md5_ok": parity.get("ok"),
            "candidates": int(results[-1]["n_cand"]), "unfiltered_candidates": int(st.n_unfiltered_candidates), "fragments_per_step": n_frag, "wall_seconds_timed_region": wall}
    if secondary:
        line["secondary_mode"] = secondary
    if not args.no_cpu_baseline and world == 1 and not _build.oracle_available():
        line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": None,
                                "not_measured": "the reference binary oracle/_ref/arriba is not built here (oracle/Makefile needs the reference sources)", "full_size": REFERENCE_FULL_SIZE.get(args.workload)}
    elif not args.no_cpu_baseline and world == 1:   # the CPU reference beside the GPU number: rank 0 at N=1 only
        sp = ensure_world(args.workload, sample_bp)
        n, scope_s, total = reference_run(sp, cores)
        line["cpu_baseline"] = {"value": n / scope_s, "unit": UNIT, "cores": 1, "kind": "reference",
                                "sample": "first %d breakpoints of the workload at full depth = %d fragments; unmodified reference (oracle/_ref/arriba), arrival times of its own progress lines over %s" % (sample_bp, n, SCOPE),
                                "whole_run_seconds": total, "host_cores_available": cores, "full_size": REFERENCE_FULL_SIZE.get(args.workload)}
    if dist:
        dist.destroy_process_group()
    sys.stderr.flush()
    print(json.dumps(line), flush=True)
    if parity.get("checked") and not parity.get("ok"):
        sys.stderr.write("bench.py: output files differ from the reference's (md5), see \"parity\" in the line above\n")
        sys.exit(1)


if __name__ == "__main__":
    main()
