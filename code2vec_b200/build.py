"""nvcc build of libc2v_b200.so (sm_100a only), in-tree so the .so travels with gpurun.

    python -m code2vec_b200.build [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.environ.get("C2V_LIB_OUT", os.path.join(HERE, "libc2v_b200.so"))   # variant builds (scripts/sanitize.sh)
EXTRA = os.environ.get("C2V_NVCC_EXTRA", "").split()
SOURCES = ["c2v_api.cu", "c2v_session.cu", "c2v_encode_ffma.cu", "c2v_encode_tm.cu", "c2v_label_tcgen05.cu", "c2v_label_backward_tc.cu", "c2v_head.cu",
           "c2v_backward.cu", "c2v_backward_dw_tc.cu", "c2v_backward_dc_tc.cu", "c2v_batch.cu", "c2v_adam.cu", "c2v_corpus.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr"]


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".cpp"))]
    deps.append(os.path.join(HERE, "..", "include", "c2v_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + (".o" if not EXTRA else ".var.o"))
        cmd = [NVCC] + FLAGS + EXTRA + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([NVCC, "-shared", "-o", OUT] + objs)   # static cudart (nvcc default)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
