"""Builds the CUDA C-ABI library in-tree for sm_100a (no torch dependency).

    python -m lcp_physics_b200.build        # or __graft_entry__.build()

nvcc cross-compiles without a GPU. The resulting `csrc/liblcpb200.so` is
git-ignored but travels to the GPU box with the gpurun snapshot.
Objects are rebuilt only when one of their sources changed (per-object digests
under csrc/build/).
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJDIR = os.path.join(CSRC, "build")
LIB = os.path.join(CSRC, "liblcpb200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]

DUAL_DEPS = ["lcp_kernels.cu", "lcp_launch.h", "lcp_device.cuh", "lcp_lu.cuh", "lcp_solver.cuh"]
COND_DEPS = ["lcp_cond_kernels.cu", "lcp_cond_launch.h", "lcp_device.cuh", "lcp_condensed.cuh"]
BAND_DEPS = ["lcp_band_kernels.cu", "lcp_band_launch.h", "lcp_device.cuh", "lcp_condensed.cuh", "lcp_banded.cuh"]
API_DEPS = ["lcpb200.cu", "lcp_assemble.cuh", "lcp_contacts.cuh", "lcp_joints.cuh", "../../include/lcpb200.h"] + DUAL_DEPS[1:] + COND_DEPS[1:] + BAND_DEPS[1:]

# dual-form kernels: one TU per (dtype, residency mode); condensed kernels: one per (dtype, NS)
DUAL_VARIANTS = [(t, m) for t in ("float", "double") for m in (0, 1, 2)]
COND_VARIANTS = [(t, ns) for t in ("float", "double") for ns in (2, 3, 4, 6, 8)]


def _jobs():
    jobs = []
    for t, m in DUAL_VARIANTS:
        jobs.append(("kernels_%s_m%d.o" % (t, m), "lcp_kernels.cu", ["-DLCP_T=%s" % t, "-DLCP_MODE=%d" % m], DUAL_DEPS))
    for t, ns in COND_VARIANTS:
        jobs.append(("cond_%s_%d.o" % (t, ns), "lcp_cond_kernels.cu", ["-DLCP_T=%s" % t, "-DLCP_NS=%d" % ns], COND_DEPS))
    # LCPB200_BAND_DEFS: extra -D flags for the banded kernel (debug builds, e.g. -DLCP_BAND_LUPROF)
    jobs.append(("band.o", "lcp_band_kernels.cu", os.environ.get("LCPB200_BAND_DEFS", "").split(), BAND_DEPS))
    jobs.append(("api.o", "lcpb200.cu", [], API_DEPS))
    return jobs


def _digest(deps, extra):
    h = hashlib.sha256()
    for d in deps:
        with open(os.path.join(CSRC, d), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS + extra).encode())
    return h.hexdigest()


def _stale(obj, digest):
    stamp = os.path.join(OBJDIR, obj + ".sha")
    if not (os.path.exists(os.path.join(OBJDIR, obj)) and os.path.exists(stamp)):
        return True
    with open(stamp) as f:
        return f.read().strip() != digest


STAMP = LIB + ".sha"      # digest of every source + flag the library was built from (git-ignored, travels with the .so)


def _lib_digest():
    h = hashlib.sha256()
    for obj, _, defs, deps in _jobs():
        h.update((obj + ":" + _digest(deps, defs)).encode())
    return h.hexdigest()


def is_fresh():
    """True when liblcpb200.so was built from the current sources and flags -- also on a box that received the
    library without the object directory (gpurun ships *.so, not csrc/build/)."""
    if not os.path.exists(LIB):
        return False
    if os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == _lib_digest():
                return True
    return not any(_stale(obj, _digest(deps, defs)) for obj, _, defs, deps in _jobs())


def build(force=False, verbose=True, max_parallel=None):
    if not force and is_fresh():
        if not os.path.exists(STAMP):
            with open(STAMP, "w") as f:
                f.write(_lib_digest())
        return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    todo = []
    objs = []
    for obj, src, defs, deps in _jobs():
        objs.append(os.path.join(OBJDIR, obj))
        dg = _digest(deps, defs)
        if force or _stale(obj, dg):
            todo.append((obj, dg, [nvcc] + NVCC_FLAGS + defs + ["-c", os.path.join(CSRC, src), "-o",
                                                               os.path.join(OBJDIR, obj)]))
    if not todo and os.path.exists(LIB):
        return LIB
    max_parallel = max_parallel or max(1, (os.cpu_count() or 4))
    running = []
    failed = []

    def reap(block):
        for item in list(running):
            obj, dg, proc = item
            rc = proc.wait() if block else proc.poll()
            if rc is None:
                continue
            running.remove(item)
            if rc:
                failed.append(obj)
            else:
                with open(os.path.join(OBJDIR, obj + ".sha"), "w") as f:
                    f.write(dg)
            if block:
                return

    for obj, dg, cmd in todo:
        while len(running) >= max_parallel:
            reap(True)
        if verbose:
            print("[lcp_physics_b200.build]", " ".join(cmd), flush=True)
        stamp = os.path.join(OBJDIR, obj + ".sha")
        if os.path.exists(stamp):
            os.remove(stamp)
        running.append((obj, dg, subprocess.Popen(cmd, cwd=CSRC)))
    while running:
        reap(True)
    if failed:
        raise RuntimeError("nvcc failed for %s" % failed)
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs
    if verbose:
        print("[lcp_physics_b200.build]", " ".join(link), flush=True)
    subprocess.check_call(link, cwd=CSRC)
    with open(STAMP, "w") as f:
        f.write(_lib_digest())
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    print(LIB)
