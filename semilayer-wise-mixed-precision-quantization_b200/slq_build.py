"""slq_build.py -- compiles csrc/*.cu into libslq_b200.so (in-tree, next to this file) for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the build container; the resulting .so travels
to the GPU box with the repo snapshot (it is git-ignored, not gpurun-ignored).
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libslq_b200.so")
STAMP = os.path.join(HERE, "build", "sources.sha256")
SOURCES = ["quantizer.cu", "layers.cu", "conv_umma.cu", "stem_umma.cu", "eval_tail.cu", "probe.cu", "tail_umma.cu",
           "block_tail.cu", "tma_host.cu", "calib.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-I", os.path.join(ROOT, "include"), "-I", CSRC,
]


def _digest():
    h = hashlib.sha256()
    names = sorted(os.listdir(CSRC)) + ["../../include/slq.h"]
    for n in names:
        p = os.path.join(CSRC, n)
        if os.path.isfile(p):
            h.update(n.encode())
            h.update(open(p, "rb").read())
    # the flags WITHOUT the checkout's own path: the snapshot on a GPU box lives under another root and must not
    # look stale there (several ranks would then rebuild the same objects at once)
    h.update(" ".join(f.replace(ROOT, "<root>") for f in NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build():
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    return open(STAMP).read().strip() != _digest()


def build(force=False, verbose=False, debug=False):
    """Builds libslq_b200.so if the sources changed.  Returns the library path.
    debug=True builds libslq_b200_dbg.so instead: the same kernels with the timeline tracer / wait
    statistics compiled in (-DSLQ_DEBUG_TRACE=1), used by tools/trace_*.py and tools/wait_stats.py."""
    if debug:
        return _build_debug(verbose)
    if not force and not needs_build():
        return LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    # one builder at a time (the ranks of a torchrun job all call this): the others wait, then find the stamp current
    import fcntl
    with open(os.path.join(HERE, "build", ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not needs_build():
            return LIB
        return _build_locked(verbose)


def _build_locked(verbose):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode())
            raise RuntimeError("nvcc failed on %s" % src)
    cmd = [nvcc, "-shared", "-o", LIB + ".tmp"] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(cmd)
    os.replace(LIB + ".tmp", LIB)  # a process that already mapped the old library keeps its inode
    with open(STAMP, "w") as f:
        f.write(_digest())
    return LIB


LIB_DBG = os.path.join(HERE, "libslq_b200_dbg.so")


def _build_debug(verbose=False):
    stamp = os.path.join(HERE, "build", "dbg", "sources.sha256")
    if os.path.exists(LIB_DBG) and os.path.exists(stamp) and open(stamp).read().strip() == _digest():
        return LIB_DBG
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(os.path.join(HERE, "build", "dbg"), exist_ok=True)
    procs, objs = [], []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", "dbg", src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-DSLQ_DEBUG_TRACE=1", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode())
            raise RuntimeError("nvcc failed on %s" % src)
    subprocess.check_call([nvcc, "-shared", "-o", LIB_DBG] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    with open(stamp, "w") as f:
        f.write(_digest())
    return LIB_DBG


def build_variant(name, defines, verbose=False):
    """A/B build of the same sources with extra -D flags -> libslq_b200_<name>.so (developer tools load it with
    $SLQ_LIB_VARIANT=<name>; never the product path).  `python slq_build.py --variant resi2f SLQ_RES_I2F`"""
    lib = os.path.join(HERE, "libslq_b200_%s.so" % name)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    bdir = os.path.join(HERE, "build", name)
    os.makedirs(bdir, exist_ok=True)
    procs, objs = [], []
    for src in SOURCES:
        obj = os.path.join(bdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-D%s" % d for d in defines] + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode())
            raise RuntimeError("nvcc failed on %s" % src)
    subprocess.check_call([nvcc, "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return lib


if __name__ == "__main__":
    if "--variant" in sys.argv:
        i = sys.argv.index("--variant")
        print(build_variant(sys.argv[i + 1], sys.argv[i + 2:], verbose=True))
        sys.exit(0)
    print(build(force="--force" in sys.argv, verbose=True, debug="--debug" in sys.argv))
