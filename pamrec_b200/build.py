"""Builds libpamrec_b200.so (sm_100a only) in-tree with nvcc.  No JIT cache: the .so travels with the repo."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpamrec_b200.so")
SOURCES = ["api.cu", "prof.cu", "comm.cu", "kernels_encoder.cu", "kernels_attn_mma.cu", "kernels_head.cu", "kernels_head2.cu", "kernels_sibling.cu", "kernels_sasrec.cu", "kernels_optim.cu", "kernels_sparse2.cu", "kernels_shard.cu", "kernels_p2p.cu", "batcher.cu", "tokenizer.cu", "crc32c.cu"]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith((".h", ".cuh", ".inl"))) + [os.path.join("..", "..", "include", "pamrec_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr",
]


def nccl_include():
    """nccl.h matching the libnccl.so.2 that PyTorch loads (types only: the functions are resolved with dlsym)."""
    try:
        import nvidia
        for p in nvidia.__path__:
            inc = os.path.join(p, "nccl", "include")
            if os.path.exists(os.path.join(inc, "nccl.h")):
                return ["-I", inc]
    except Exception:
        pass
    return []


def nccl_library():
    try:
        import nvidia
        for p in nvidia.__path__:
            lib = os.path.join(p, "nccl", "lib", "libnccl.so.2")
            if os.path.exists(lib):
                return lib
    except Exception:
        pass
    return None


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose=False, force=False, extra=()):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs = []
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = [nvcc, *NVCC_FLAGS, *nccl_include(), *extra, "-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
        if verbose and out.strip():
            print(out, file=sys.stderr)
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}")
    return LIB


if __name__ == "__main__":
    print(build(verbose=True, force="--force" in sys.argv, extra=["-Xptxas", "-v"] if "--ptxas" in sys.argv else ()))
