"""Build libthor_b200.so (sm_100a only) in-tree with nvcc.  Used by __graft_entry__.build() and the tests."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libthor_b200.so")
SOURCES = ["tb_api.cu", "tb_rdo.cu"]
DEPS = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))) + [os.path.join("..", "..", "include", "thor_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--std=c++17", "-shared", "-Xcompiler", "-fPIC",
              "-Xptxas", "-v", "--use_fast_math=false"]


def nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def _compile(src, obj, flags):
    cmd = [nvcc()] + flags + ["-c", "-o", obj, os.path.join(CSRC, src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return r.returncode, " ".join(cmd) + "\n" + r.stdout + r.stderr


def build(force=False, verbose=False, out=None):
    """one object per translation unit (compiled in parallel, kept under thor_b200/build/ and reused while its sources are older), then one link"""
    if not force and not stale() and out is None:
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math") and f != "-shared"]
    objdir = os.path.join(HERE, "build", "default" if out is None else os.path.basename(out))
    os.makedirs(objdir, exist_ok=True)
    newest = max(os.path.getmtime(os.path.join(CSRC, d)) for d in DEPS)
    jobs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest:
            jobs.append((s, obj))
    log = ""
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        for rc, text in ex.map(lambda j: _compile(j[0], j[1], flags), jobs):
            log += text
            if rc != 0:
                sys.stderr.write(text)
                raise RuntimeError("nvcc failed building libthor_b200.so")
    cmd = [nvcc(), "-shared", "-o", out or LIB] + [os.path.join(objdir, s.replace(".cu", ".o")) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log += " ".join(cmd) + "\n" + r.stdout + r.stderr
    with open(os.path.join(HERE, "build.log") if out is None else out + ".log", "w") as f:  # A/B builds log next to their output (ab_libs/)
        f.write(log)
    if r.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed linking libthor_b200.so")
    if verbose:
        print(log)
    return out or LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
