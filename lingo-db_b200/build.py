"""In-tree build recipe for every native artefact of the package.

  libldb_datagen_host.so  host generator (g++, no CUDA)                     csrc/datagen_host.cpp
  libldb_gpu.so           sm_100a kernels + C++ host runtime + C-ABI        csrc/*.cu csrc/*.cpp

`nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo` cross-compiles here without a GPU; the
built .so files are git-ignored but travel to the GPU box with the gpurun snapshot.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
INCLUDE = os.path.join(ROOT, "include")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CXX = os.environ.get("LDB_CXX", "/usr/bin/g++")  # not $CXX: the image exports a static-libstdc++ wrapper there

GPU_LIB = os.path.join(HERE, "libldb_gpu.so")
GEN_LIB = os.path.join(HERE, "libldb_datagen_host.so")
ARROW_LIB = os.path.join(HERE, "libldb_arrow_io.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unused-function",
    "--expt-relaxed-constexpr", "-cudart", "static", "-I", INCLUDE, "-I", CSRC,
]


def _sources(exts):
    out = []
    for dirpath, _, files in os.walk(CSRC):
        for f in sorted(files):
            if f.endswith(exts):
                out.append(os.path.join(dirpath, f))
    return sorted(out)


def _stamp(paths, extra=""):
    h = hashlib.sha256(extra.encode())
    for p in paths:
        h.update(os.path.relpath(p, ROOT).encode())  # relative: the stamp must survive the move to the GPU box
        with open(p, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def _up_to_date(target, stamp):
    sfile = target + ".stamp"
    return os.path.exists(target) and os.path.exists(sfile) and open(sfile).read() == stamp


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd[:3]) + " …")
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr)


class _Lock:
    """One builder at a time (torchrun starts N ranks that all import the package)."""

    def __enter__(self):
        import fcntl
        self.fh = open(os.path.join(HERE, ".build.lock"), "w")
        fcntl.flock(self.fh, fcntl.LOCK_EX)
        return self

    def __exit__(self, *a):
        import fcntl
        fcntl.flock(self.fh, fcntl.LOCK_UN)
        self.fh.close()


def build_datagen_host(verbose=False, force=False):
    # an up-to-date library is returned without the lock: loading must work from a read-only tree
    if not force and _up_to_date(GEN_LIB, _datagen_host_stamp()):
        return GEN_LIB
    with _Lock():
        return _build_datagen_host(verbose, force)


def build_gpu(verbose=False, force=False, ptxas_verbose=False):
    if not force and _up_to_date(GPU_LIB, _gpu_stamp()):
        return GPU_LIB
    with _Lock():
        return _build_gpu(verbose, force, ptxas_verbose)


def _datagen_host_stamp():
    deps = [os.path.join(CSRC, f) for f in ("datagen_host.cpp", "tpch_gen.h", "dbgen_gen.h")] + [os.path.join(INCLUDE, "ldb_datagen.h")]
    return _stamp(deps)


def _build_datagen_host(verbose=False, force=False):
    srcs = [os.path.join(CSRC, "datagen_host.cpp")]
    stamp = _datagen_host_stamp()
    if not force and _up_to_date(GEN_LIB, stamp):
        return GEN_LIB
    _run([CXX, "-std=c++17", "-O3", "-fPIC", "-pthread", "-shared", "-Wall", "-I", INCLUDE, "-o", GEN_LIB] + srcs, verbose)
    open(GEN_LIB + ".stamp", "w").write(stamp)
    return GEN_LIB


def _gpu_sources():
    cu = _sources((".cu",))
    cpp = [p for p in _sources((".cpp",)) if not p.endswith("_host.cpp")]
    host_cpp = [p for p in _sources((".cpp",)) if p.endswith("_host.cpp") and not p.endswith("datagen_host.cpp")]  # g++ only (function multi-versioning)
    hdr = _sources((".h", ".cuh")) + [os.path.join(INCLUDE, f) for f in sorted(os.listdir(INCLUDE))]
    return cu, cpp, host_cpp, hdr


def _gpu_stamp():
    cu, cpp, host_cpp, hdr = _gpu_sources()
    return _stamp(cu + cpp + host_cpp + hdr, " ".join(NVCC_FLAGS).replace(ROOT, "$ROOT"))


def _build_gpu(verbose=False, force=False, ptxas_verbose=False):
    cu, cpp, host_cpp, _ = _gpu_sources()
    stamp = _gpu_stamp()
    if not force and _up_to_date(GPU_LIB, stamp):
        return GPU_LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in cu + cpp:
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        objs.append(obj)
        cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if ptxas_verbose else []) + ["-x", "cu", "-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src in host_cpp:
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        objs.append(obj)
        cmd = [CXX, "-std=c++17", "-O3", "-fPIC", "-Wall", "-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(out)
        elif (verbose or ptxas_verbose) and out:
            print(out)
    if failed:
        raise RuntimeError("nvcc failed")
    _run([NVCC, "-shared", "-cudart", "static", "-o", GPU_LIB + ".tmp"] + objs, verbose)
    os.replace(GPU_LIB + ".tmp", GPU_LIB)
    open(GPU_LIB + ".stamp", "w").write(stamp)
    return GPU_LIB


def build_arrow_io(verbose=False, force=False):
    """libldb_arrow_io.so: Arrow IPC file → backend table (csrc_arrow/), linked against the Arrow C++ that ships inside pyarrow."""
    import pyarrow
    src = os.path.join(HERE, "csrc_arrow", "arrow_table_io.cpp")
    deps = [src, os.path.join(INCLUDE, "ldb_arrow_io.h"), os.path.join(INCLUDE, "ldb_gpu.h")]
    if not force and _up_to_date(ARROW_LIB, _stamp(deps, pyarrow.__version__)):
        return ARROW_LIB
    with _Lock():
        pa_dir = os.path.dirname(pyarrow.__file__)
        stamp = _stamp(deps, pyarrow.__version__)
        if not force and _up_to_date(ARROW_LIB, stamp):
            return ARROW_LIB
        libs = [f for f in os.listdir(pa_dir) if f.startswith("libarrow.so.") and f.count(".") == 2]
        _run([CXX, "-std=c++20", "-O2", "-fPIC", "-shared", "-Wall", "-I", INCLUDE, "-I", os.path.join(pa_dir, "include"), "-o", ARROW_LIB, src,
              "-L", pa_dir, "-l:" + sorted(libs)[0], "-Wl,-rpath," + pa_dir], verbose)
        open(ARROW_LIB + ".stamp", "w").write(stamp)
        return ARROW_LIB


def build_all(verbose=False, force=False):
    return build_datagen_host(verbose, force), build_gpu(verbose, force), build_arrow_io(verbose, force)


if __name__ == "__main__":
    build_all(verbose=True, force="--force" in sys.argv)
