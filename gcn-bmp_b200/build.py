"""Build libgcnbmp.so in-tree with nvcc for sm_100a (no torch extension machinery:
the boundary is a plain C-ABI shared library loaded with ctypes)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "gcnbmp", "libgcnbmp.so")
SOURCES = ["misc.cu", "gemm.cu", "heads.cu", "ggnn.cu", "ggnn_x3.cu", "ggnn_tc.cu", "ggnn_tc256.cu", "ggnn_tc_bwd.cu", "wgrad_tc.cu", "wgrad_tc2.cu", "relgcn.cu", "relgcn_tc.cu", "readout.cu", "readout_tc.cu", "coattn.cu", "coattn_big.cu", "coattn_tc.cu", "bimpm.cu", "pair.cu", "det.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--use_fast_math=false"]
FLAGS = [f for f in FLAGS if f != "--use_fast_math=false"]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "gcnbmp.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc, "-shared", "-o", OUT] + objs)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
