"""In-tree build of the sm_100a C-ABI library (nvcc cross-compiles without a GPU).

``python -m e2fgvi_b200.build`` or ``__graft_entry__.build()``.  Output: ``e2fgvi_b200/libe2fgvi_b200.so``
(git-ignored, shipped to the GPU box with the tree).  No torch headers are involved: the boundary is plain C.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libe2fgvi_b200.so")
STAMP = LIB_PATH + ".stamp"

SOURCES = ["api.cu", "flow_warp.cu", "dcn.cu", "focal_attn.cu", "t2t.cu", "gemm.cu", "conv.cu", "elementwise.cu", "video.cu", "spynet.cu", "conv_kxn.cu", "peer.cu", "metrics.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "-I", os.path.join(os.path.dirname(HERE), "include"),
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256()
    names = sorted(os.listdir(CSRC))
    for n in names:
        if n.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(CSRC, n), "rb") as f:
                h.update(n.encode())
                h.update(f.read())
    with open(os.path.join(os.path.dirname(HERE), "include", "e2fgvi_b200.h"), "rb") as f:
        h.update(f.read())
    # flags without the checkout's absolute path: a built tree that is moved or copied stays up to date
    h.update(" ".join(NVCC_FLAGS).replace(os.path.dirname(HERE), ".").encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu into one shared library. Returns the path. Skips when sources are unchanged."""
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == digest:
                return LIB_PATH
    objs = []
    log = []
    os.makedirs(os.path.join(os.path.dirname(HERE), "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(os.path.dirname(HERE), "build", src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, obj, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    cmd = [_nvcc(), "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static",
                                                          "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append(r.stdout)
    if r.returncode != 0:
        sys.stderr.write("\n".join(log))
        raise RuntimeError("link failed")
    with open(STAMP, "w") as f:
        f.write(digest)
    with open(os.path.join(os.path.dirname(HERE), "build", "nvcc.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
