"""Build logic for arriba-b200 (used by __graft_entry__.build(), the tests and bench.py).

product : nvcc -gencode arch=compute_100a,code=sm_100a  -> arriba_b200/libarriba_b200.so   (CUDA, the only library the package loads)
hostsim : g++ -DARB_HOSTSIM over the same sources       -> tests/hostsim/libarriba_b200_hostsim.so (CPU test-suite only)
oracle  : oracle/Makefile (unmodified reference + shim) -> oracle/_ref/arriba               (only when /root/reference exists)
tools   : tools/synth.cpp                                -> build/synth
"""
import os, subprocess, sys, shutil
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "arriba_b200", "csrc")
PRODUCT_LIB = os.path.join(ROOT, "arriba_b200", "libarriba_b200.so")
HOSTSIM_LIB = os.path.join(ROOT, "tests", "hostsim", "libarriba_b200_hostsim.so")
CLI_BIN = os.path.join(ROOT, "arriba_b200", "bin", "arriba")
SYNTH_BIN = os.path.join(ROOT, "build", "synth")
ORACLE_BIN = os.path.join(ROOT, "oracle", "_ref", "arriba")
REFERENCE = "/root/reference/source"

CU_SOURCES = ["prims.cu", "engine.cu", "bamscan.cu", "fragtable.cu", "annotate.cu", "fusions.cu", "events.cu", "rows.cu", "consensus.cu", "mismap.cu", "exchange.cu", "capi.cu", "selftest.cu"]
CPP_SOURCES = ["mismatch_table.cpp", "host/refdata.cpp", "host/ingest.cpp", "host/annotate.cpp", "host/viral.cpp", "host/pipeline.cpp", "host/events.cpp", "host/output.cpp", "host/shard.cpp", "host/host_capi.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--fmad=false",
              "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function", "-Xptxas", "-v"]
GXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-Wall", "-Wno-unused-function", "-ffp-contract=off"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _all_sources():
    out = [os.path.join(ROOT, "include", "arriba_b200.h")]
    for d, _, files in os.walk(CSRC):
        out += [os.path.join(d, f) for f in files]
    return out


def _run(cmd, log=None):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log is not None:
        log.append(" ".join(cmd) + "\n" + r.stdout)
    if r.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def nvcc_path():
    for p in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if p and os.path.exists(p):
            return p
    raise RuntimeError("nvcc not found")


def build_product(force=False, verbose=False):
    """Cross-compiles every CUDA source for sm_100a (works without a GPU) and links the C-ABI shared library."""
    if not force and not _newer(PRODUCT_LIB, _all_sources()):
        return PRODUCT_LIB
    objdir = os.path.join(ROOT, "build", "product")
    os.makedirs(objdir, exist_ok=True)
    nvcc = nvcc_path()
    log = []
    jobs = []
    for s in CU_SOURCES:
        o = os.path.join(objdir, s + ".o")
        jobs.append([nvcc] + NVCC_FLAGS + ["-I", os.path.join(ROOT, "include"), "-c", os.path.join(CSRC, s), "-o", o])
    for s in CPP_SOURCES:
        o = os.path.join(objdir, s.replace("/", "_") + ".o")
        jobs.append(["g++"] + GXX_FLAGS + ["-I", os.path.join(ROOT, "include"), "-c", os.path.join(CSRC, s), "-o", o])
    with ThreadPoolExecutor(8) as ex:
        list(ex.map(lambda c: _run(c, log), jobs))
    objs = [os.path.join(objdir, s.replace("/", "_") + ".o") for s in CU_SOURCES + CPP_SOURCES]
    _run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", PRODUCT_LIB] + objs + ["-lcudart", "-lz", "-lpthread"], log)
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return PRODUCT_LIB


def build_cli(force=False):
    """The `arriba` executable: a thin C++ front end over the C ABI of the product library."""
    src = os.path.join(CSRC, "host", "cli_main.cpp")
    if force or _newer(CLI_BIN, [src, PRODUCT_LIB]):
        os.makedirs(os.path.dirname(CLI_BIN), exist_ok=True)
        _run(["g++"] + GXX_FLAGS + ["-o", CLI_BIN, src, "-L", os.path.dirname(PRODUCT_LIB), "-larriba_b200", "-Wl,-rpath,$ORIGIN/..", "-lpthread"])
    return CLI_BIN


HOSTSIM_CLI = os.path.join(ROOT, "tests", "hostsim", "arriba_hostsim")


def build_cli_hostsim(force=False):
    """The same `arriba` front end linked against the CPU stand-in: lets the CPU test-suite drive the command line. Test-only, lives under tests/."""
    lib = build_hostsim()
    src = os.path.join(CSRC, "host", "cli_main.cpp")
    if force or _newer(HOSTSIM_CLI, [src, lib]):
        _run(["g++"] + GXX_FLAGS + ["-o", HOSTSIM_CLI, src, "-L", os.path.dirname(lib), "-l:" + os.path.basename(lib), "-Wl,-rpath,$ORIGIN", "-lpthread"])
    return HOSTSIM_CLI


def build_hostsim(force=False):
    """CPU test-suite stand-in: same rule functors, sequential primitives. Never loaded by the package or the bench."""
    if not force and not _newer(HOSTSIM_LIB, _all_sources()):
        return HOSTSIM_LIB
    os.makedirs(os.path.dirname(HOSTSIM_LIB), exist_ok=True)
    objdir = os.path.join(ROOT, "build", "hostsim")
    os.makedirs(objdir, exist_ok=True)
    jobs = []
    for s in CU_SOURCES:
        jobs.append(["g++", "-x", "c++"] + GXX_FLAGS + ["-DARB_HOSTSIM", "-I", os.path.join(ROOT, "include"), "-c", os.path.join(CSRC, s), "-o", os.path.join(objdir, s + ".o")])
    for s in CPP_SOURCES:
        jobs.append(["g++"] + GXX_FLAGS + ["-DARB_HOSTSIM", "-I", os.path.join(ROOT, "include"), "-c", os.path.join(CSRC, s), "-o", os.path.join(objdir, s.replace("/", "_") + ".o")])
    with ThreadPoolExecutor(8) as ex:
        list(ex.map(_run, jobs))
    objs = [os.path.join(objdir, s.replace("/", "_") + ".o") for s in CU_SOURCES + CPP_SOURCES]
    _run(["g++", "-shared", "-o", HOSTSIM_LIB] + objs + ["-lz", "-lpthread"])
    return HOSTSIM_LIB


def build_tools(force=False):
    src = os.path.join(ROOT, "tools", "synth.cpp")
    if force or _newer(SYNTH_BIN, [src]):
        os.makedirs(os.path.dirname(SYNTH_BIN), exist_ok=True)
        _run(["g++", "-O2", "-std=c++17", "-o", SYNTH_BIN, src, "-lz"])
    return SYNTH_BIN


def oracle_available():
    return os.path.isdir(REFERENCE) or os.path.exists(ORACLE_BIN)


def build_oracle(force=False):
    """Compiles the unmodified reference against the shim where its sources are readable; elsewhere a prebuilt
    oracle/_ref/arriba is used as is. Only recording the reference's results (tests/worldutil.py) and bench.py's
    CPU baseline run it."""
    if os.path.isdir(REFERENCE):
        _run(["make", "-C", os.path.join(ROOT, "oracle"), "-j8"])
    if not os.path.exists(ORACLE_BIN):
        raise RuntimeError("oracle/_ref/arriba is missing and the reference sources are not available to build it")
    return ORACLE_BIN


if __name__ == "__main__":
    what = sys.argv[1:] or ["product", "cli", "hostsim", "tools", "oracle"]
    for w in what:
        print(w, "->", {"product": build_product, "cli": build_cli, "hostsim": build_hostsim, "tools": build_tools, "oracle": build_oracle}[w](force=True))
