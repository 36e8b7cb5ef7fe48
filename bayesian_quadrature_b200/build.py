"""Builds libbq_b200.so in-tree with nvcc for sm_100a (no torch dependency in the library)."""
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbq_b200.so")
SOURCES = ["bq_setup2.cu", "bq_score.cu", "bq_score_generic.cu", "bq_reduce.cu", "bq_round.cu", "bq_sort.cu", "bq_capi.cu"]
HEADERS = ["bq_common.cuh", os.path.join("..", "..", "include", "bq_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--fmad=true", "-Xptxas", "-v"]
#: bq_score.cu is compiled once per observation-capacity class (its instantiations only) plus once as the dispatcher,
#: so that the classes build in parallel
SCORE_CLASSES = [16, 64, 128, 160, 256]
#: ... and the band-relative kernels of the large classes in units of their own
REL_CLASSES = [128, 160, 256]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def _units():
    """(source, object, extra flags) of every translation unit."""
    units = []
    for src in SOURCES:
        base = src.replace(".cu", "")
        if src == "bq_score.cu":
            units.append((src, base + ".o", []))
            units += [(src, "%s_%d.o" % (base, c), ["-DBQB_SCORE_CLASS=%d" % c]) for c in SCORE_CLASSES]
            units += [(src, "%s_%d_rel.o" % (base, c), ["-DBQB_SCORE_CLASS=%d" % c, "-DBQB_SCORE_REL=1"]) for c in REL_CLASSES]
        else:
            units.append((src, base + ".o", []))
    return units


def _compile(unit):
    src, obj, extra = unit
    obj = os.path.join(CSRC, obj)
    r = subprocess.run([_nvcc()] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return unit, obj, r.returncode, r.stdout


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    units = _units()
    with ThreadPoolExecutor(max_workers=min(len(units), os.cpu_count() or 1)) as pool:
        results = list(pool.map(_compile, units))
    objs, log = [], []
    for (src, _, extra), obj, rc, out in results:
        log.append("==== %s %s\n%s" % (src, " ".join(extra), out))
        if rc:
            raise RuntimeError("nvcc failed on %s %s:\n%s" % (src, " ".join(extra), out))
        objs.append(obj)
    r = subprocess.run([_nvcc(), "-shared", "-o", LIB] + objs + ["-lcudart"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        raise RuntimeError("link failed:\n" + r.stdout)
    with open(os.path.join(CSRC, "ptxas.log"), "w") as fh:
        fh.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
