"""Builds the in-tree native artefacts of bammmotif2_b200 with nvcc / g++ (no torch, no JIT cache):

    libbamm_b200.so   the C-ABI library (include/bamm_b200.h): csrc/capi.cu (+ capi_*.inl, one translation unit) + csrc/*.cuh, sm_100a only
    bin/BaMMmotif     the C++ host side (host/*.cpp: the reference's class surface over the C ABI) as the drop-in CLI
    bin/BaMMScan      the occurrence scan over the same host classes (host/mainScan.cpp)
    bin/host_check    test helper for the CPU-only parts of the host classes

Run as `python -m bammmotif2_b200.build` or through __graft_entry__.build().
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libbamm_b200.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-fmad=false",            # keep the reference's operation order (no FMA contraction) in the model update
    "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-misleading-indentation",
    "-shared",
]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _newer(target, deps):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


# translation units of the library: capi.cu carries the C ABI and the small kernels, each launch_*.cu one family of heavily
# templated kernels (csrc/launch.h); every unit depends on every header (cheap to state, the units build in parallel)
LIB_UNITS = ["capi", "launch_estep", "launch_mstep", "launch_score"]


def build_lib(force=False, verbose=False):
    from concurrent.futures import ThreadPoolExecutor
    cdir = os.path.join(HERE, "csrc")
    odir = os.path.join(HERE, "build", "lib")
    os.makedirs(odir, exist_ok=True)
    headers = [os.path.join(cdir, f) for f in sorted(os.listdir(cdir)) if f.endswith((".cuh", ".inl", ".h"))] + \
              [os.path.join(ROOT, "include", "bamm_b200.h"), __file__]
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)          # the image exports a gcc wrapper without libgomp specs
    ccbin = ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    jobs = []
    objs = []
    for u in LIB_UNITS:
        src, obj = os.path.join(cdir, u + ".cu"), os.path.join(odir, u + ".o")
        objs.append(obj)
        if force or not _newer(obj, [src] + headers):
            jobs.append([nvcc_path()] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj] + ccbin)
    if jobs:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            for rc in ex.map(lambda cmd: subprocess.call(cmd, env=env), jobs):
                if rc:
                    raise RuntimeError("nvcc failed")
    if jobs or not _newer(LIB, objs):
        subprocess.check_call([nvcc_path(), "-shared", "-o", LIB] + objs + ccbin, env=env)
    return LIB


HOST_SOURCES = ["Alphabet", "SequenceSet", "BackgroundModel", "Motif", "MotifSet", "EM", "ScoreSeqSet", "SeqGenerator", "FDR", "Global"]
# -ffp-contract=off: the host arithmetic (background model, site initialisation, p-values) follows the reference's
# operation order in plain IEEE fp32, without fused multiply-adds
HOST_FLAGS = ["-std=c++17", "-O2", "-Wall", "-ffp-contract=off", "-pthread"]


def build_host(force=False):
    """host/*.cpp -> bin/BaMMmotif, bin/BaMMScan and bin/host_check, linked against libbamm_b200.so (rpath $ORIGIN/..)."""
    hdir, bdir, odir = os.path.join(HERE, "host"), os.path.join(HERE, "bin"), os.path.join(HERE, "build", "host")
    os.makedirs(bdir, exist_ok=True)
    os.makedirs(odir, exist_ok=True)
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    headers = [os.path.join(hdir, f) for f in os.listdir(hdir) if f.endswith(".h")] + [os.path.join(ROOT, "include", "bamm_b200.h"), __file__]
    objs = {}
    for name in HOST_SOURCES + ["mainBaMM", "mainScan", "host_check"]:
        src, obj = os.path.join(hdir, name + ".cpp"), os.path.join(odir, name + ".o")
        if force or not _newer(obj, [src] + headers):
            subprocess.check_call([gxx] + HOST_FLAGS + ["-c", src, "-o", obj], env=env)
        objs[name] = obj
    outs = []
    for exe, main in (("BaMMmotif", "mainBaMM"), ("BaMMScan", "mainScan"), ("host_check", "host_check")):
        out = os.path.join(bdir, exe)
        deps = [objs[n] for n in HOST_SOURCES] + [objs[main]]
        if force or not _newer(out, deps + [LIB]):
            subprocess.check_call([gxx, "-o", out, objs[main]] + [objs[n] for n in HOST_SOURCES] +
                                  ["-L" + HERE, "-lbamm_b200", "-Wl,-rpath,$ORIGIN/..", "-pthread"], env=env)
        outs.append(out)
    return outs


def build_all(force=False, verbose=False):
    return [build_lib(force, verbose)] + build_host(force)


if __name__ == "__main__":
    for p in build_all(force="--force" in sys.argv, verbose="-v" in sys.argv):
        print(p)
