"""Builds libb200match.so in-tree with nvcc for sm_100a (B200) -- no JIT cache, so the
library travels with the source tree.  Used by __graft_entry__.build() and by the tests.

    python -m lidar_global_registration_b200.build [--force]
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200match.so")
SOURCES = ["api.cu", "pack.cu", "exact.cu", "filter.cu", "candidates_tc.cu", "multiscale.cu", "cluster.cu", "wide.cu", "multi.cu", "local.cu", "batch.cu", "wide_batch.cu", "plan.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
LINK_VERSION = "cudart-shared-2-dl-pthread"
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xcompiler", "-Wall",
         "-diag-suppress", "177"]
if os.environ.get("B200M_TC_TRACE"):   # cycle-stamp tracing of the candidate kernel (tools/run_trace.sh)
    FLAGS.append("-DB200M_TC_TRACE")


STAMP = LIB + ".stamp"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def source_hash():
    """Content hash of everything the library is built from (sources, headers, flags)."""
    h = hashlib.sha256((" ".join(FLAGS) + LINK_VERSION).encode())
    files = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(CSRC, "internal.cuh"),
                                                       os.path.join(HERE, "..", "include", "b200match.h")]
    for f in files:
        h.update(open(f, "rb").read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu to an object (parallel nvcc processes) and link the shared library.
    A library whose stamp matches the current sources is kept as is (so the .so built in the
    dev container is the one loaded on the GPU box, whatever happened to file mtimes)."""
    digest = source_hash()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == digest:
        return LIB
    headers = [os.path.join(CSRC, "internal.cuh"), os.path.join(HERE, "..", "include", "b200match.h")]
    # objects are reused by mtime, which knows nothing about the flags they were compiled with
    flags_stamp = os.path.join(CSRC, ".flags")
    flags_now = " ".join(FLAGS)
    if not os.path.exists(flags_stamp) or open(flags_stamp).read() != flags_now:
        force = True
    objs, procs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src[:-3] + ".o")
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed on %s:\n%s\n" % (src, out))
        elif verbose:
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("libb200match build failed")
    with open(flags_stamp, "w") as f:
        f.write(flags_now)
    # The stamp did not match, so always relink.  One CUDA runtime per process: bind to the shared libcudart.so.12
    # (the one torch has already loaded when the library is used next to torch; /usr/local/cuda/lib64 for
    # stand-alone C++ users) instead of a private static copy -- two runtimes in one process can disagree about
    # the current device on multi-GPU ranks.
    cmd = [NVCC, "-shared", "-cudart", "shared", "-o", LIB] + objs + [
        "-gencode", "arch=compute_100a,code=sm_100a", "-Xlinker", "-rpath,/usr/local/cuda/lib64", "-ldl", "-lpthread"]
    subprocess.run(cmd, check=True)
    with open(STAMP, "w") as f:
        f.write(digest + "\n")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
