"""Build libdmt.so (hand-written sm_100a CUDA + C ABI) in-tree with nvcc.  No GPU needed to compile.

    python build.py [--force] [-v]                     -> libdmt.so
    python build.py --tag tpb32 -DDMT_FWD_TPB=32 ...   -> libdmt_tpb32.so (tuning variants; select with DMT_LIB=<path>)
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "dmt_api.cu")
DEPS = [os.path.join(HERE, "csrc", f) for f in sorted(os.listdir(os.path.join(HERE, "csrc"))) if f.endswith((".cu", ".cuh"))] + [
    os.path.join(os.path.dirname(HERE), "include", "dmt.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "-shared", "-ccbin", "/usr/bin/g++"]


def lib_path(tag=None):
    return os.path.join(HERE, "libdmt%s.so" % ("_" + tag if tag else ""))


def up_to_date(out):
    return os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(d) for d in DEPS)


def build(force=False, verbose=False, tag=None, defines=()):
    out = lib_path(tag)
    if not force and up_to_date(out):
        return out
    cmd = [NVCC] + FLAGS + list(defines) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out, SRC, "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building %s" % out)
    if verbose:
        sys.stderr.write(r.stderr)
    return out


if __name__ == "__main__":
    tag = sys.argv[sys.argv.index("--tag") + 1] if "--tag" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, tag=tag, defines=[a for a in sys.argv[1:] if a.startswith("-D")]))
