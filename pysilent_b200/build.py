"""Build libsilent_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsilent_b200.so")
SOURCES = ["plan.cu", "pyramid.cu", "conv.cu", "stack_fused.cu", "emit.cu", "display.cu", "pipeline.cu", "gather.cu", "nv12.cu", "points.cu", "match.cu", "motion.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                      # canonical order: every FMA in the library is an explicit fmaf()
    "-Xcompiler", "-fPIC,-ffp-contract=off", "-Xptxas", "-v",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "silent_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile every .cu of the library into pysilent_b200/libsilent_b200.so. Returns the path."""
    if not force and not needs_build():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append("== %s\n%s" % (src, out))
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError("nvcc failed on %s" % src)
    with open(os.path.join(HERE, "build", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    subprocess.check_call([_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"])
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
