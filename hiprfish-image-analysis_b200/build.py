"""Builds libhipr_b200.so in-tree with nvcc for sm_100a (no other architecture, no JIT cache)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libhipr_b200.so")
SOURCES = ["chansum.cu", "register.cu", "nlm2d.cu", "nlm3d.cu", "lne2d.cu", "lne2d_q.cu", "fused2d.cu", "pipeline2d.cu", "mosaic_p2p.cu", "lne3d.cu", "cell_spectra.cu", "cell_geometry.cu", "kmeans1d.cu", "xcorr2d.cu", "label.cu", "watershed.cu", "morphology.cu", "host_api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "hipr_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, ptxas_verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    build_dir = os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
              [os.path.join(INCLUDE, "hipr_b200.h"), os.path.abspath(__file__)]
    newest_header = max(os.path.getmtime(h) for h in headers)
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        # per-object incremental build: an object is reused when it is newer than its source and every header
        if not force and os.path.exists(obj) and \
                os.path.getmtime(obj) > max(newest_header, os.path.getmtime(os.path.join(CSRC, src))):
            continue
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if ptxas_verbose else []) + \
              ["-I", INCLUDE, "-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose or ptxas_verbose:
            sys.stdout.write(out)
        if p.returncode != 0:
            failed = True
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, ptxas_verbose="--ptxas" in sys.argv))
