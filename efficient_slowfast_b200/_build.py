"""In-tree build of libesf_b200.so (hand-written sm_100a CUDA behind the C ABI in include/esf.h).

nvcc cross-compiles for sm_100a without a GPU; the resulting .so lives next to the sources (git-ignored), so that a
copy of the built tree runs on a GPU machine without compiling again.  ESF_NVCC_EXTRA adds nvcc flags (instrumented
builds such as -DESF_ATTN_TIMING); the library itself reads no environment variables at run time.
"""
import hashlib
import os
import shutil
import subprocess

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB = os.path.join(CSRC, "libesf_b200.so")
SOURCES = ["esf_api.cu", "esf_igemm.cu", "esf_simt.cu", "esf_attention.cu", "esf_attn_tc.cu", "esf_precise.cu", "esf_roi.cu", "esf_crop.cu",
           "esf_jpeg.cu"]
HEADERS = ["esf_common.cuh", "esf_host.h", os.path.join("..", "..", "include", "esf.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-DESF_NO_FAST_MATH",
] + os.environ.get("ESF_NVCC_EXTRA", "").split()


def _nvcc():
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found (set NVCC or put it on PATH)")
    return cand


def _digest():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu into objects and link libesf_b200.so; skipped when sources are unchanged."""
    stamp = LIB + ".stamp"
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, out))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s" % r.stdout)
    with open(stamp, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
