"""In-tree build of libphovo_b200.so (nvcc, sm_100a only).  No torch involved.

    python -m <package>.build        or        build.build()
"""
import fcntl
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libphovo_b200.so")
SOURCES = ["phovo_api.cu", "phovo_batch.cu", "kernels_pyramid.cu", "kernels_align.cu", "kernels_batch.cu", "yaml_config.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function", "-Xptxas", "-v"]


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


_DEP_SUFFIXES = (".cu", ".cpp", ".h", ".cuh")


def needs_build():
    """Out of date iff a SOURCE file is newer than the library (ptxas_v.log and the objects, which the
    build itself writes, are not dependencies)."""
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(_DEP_SUFFIXES)]
    deps.append(os.path.join(HERE, "..", "include", "phovo_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compiles and links under an exclusive file lock (several ranks of one job may call this at the
    same time: one builds, the others wait and then find the library up to date); the library is
    linked to a temporary name and renamed into place, so a process that is dlopen-ing it never
    sees a half-written file."""
    if not force and not needs_build():
        return LIB
    with open(os.path.join(HERE, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():      # another process built it while we waited
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    log = []
    for src in _sources():
        obj = os.path.join(CSRC, os.path.basename(src) + ".o")
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append(r.stderr)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed on %s" % src)
        objs.append(obj)
    with open(os.path.join(CSRC, "ptxas_v.log"), "w") as f:
        # compile times differ from run to run: keep logs of two builds comparable
        f.write("\n".join(ln for chunk in log for ln in chunk.splitlines() if "Compile time" not in ln) + "\n")
    tmp = LIB + ".tmp.%d" % os.getpid()
    cmd = [nvcc, "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        if os.path.exists(tmp):
            os.remove(tmp)
        raise RuntimeError("link failed")
    os.replace(tmp, LIB)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
