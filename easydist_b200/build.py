"""Build libedb.so (the C-ABI CUDA runtime) in-tree for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the CPU container (`__graft_entry__.build()`)
and the resulting .so travels to the GPU box with the repo snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB_PATH = os.path.join(HERE, "libedb.so")
BUILD_DIR = os.path.join(HERE, "csrc", "_build")

HEADERS = ["edb_internal.cuh", "edb_vec.cuh"]
SOURCES = ["edb_runtime.cu", "edb_reshard.cu", "edb_ll.cu", "edb_norm.cu", "edb_loss.cu", "edb_optim.cu", "edb_gemm.cu"]

NVCC_FLAGS = [
    "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC",
    "-I", INCLUDE, "-I", CSRC,
]


def _nvcc():
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    return cand if os.path.exists(cand) else None


def _digest(paths):
    h = hashlib.sha256()
    # paths relative to the repository: a built tree stays current when it is moved or copied
    rel = lambda s: os.path.relpath(s, ROOT) if os.path.isabs(s) else s
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(rel(p).encode())
            h.update(f.read())
    h.update(" ".join(map(rel, NVCC_FLAGS)).encode())
    return h.hexdigest()


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build():
    stamp = os.path.join(BUILD_DIR, "stamp")
    if not os.path.exists(LIB_PATH) or not os.path.exists(stamp):
        return True
    deps = sources() + [os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(INCLUDE, "edb.h")]
    with open(stamp) as f:
        return f.read().strip() != _digest(deps)


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ and link libedb.so. Returns the library path.

    Safe under torchrun (N ranks importing at once): the build is serialised with an exclusive
    file lock and re-checked under the lock, objects go to a private temporary directory, and the
    library and its stamp are moved into place with os.replace (atomic), so no rank can link
    against half-written objects or dlopen a half-written .so."""
    if not force and not needs_build():
        return LIB_PATH
    import fcntl
    os.makedirs(BUILD_DIR, exist_ok=True)
    with open(os.path.join(BUILD_DIR, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB_PATH  # another process built it while we waited
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
    import tempfile
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libedb.so")
    srcs = sources()
    tmp = tempfile.mkdtemp(prefix="tmp_", dir=BUILD_DIR)
    objs = [os.path.join(tmp, os.path.basename(s)[:-3] + ".o") for s in srcs]

    def compile_one(args):
        src, obj = args
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return r.stderr

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        logs = list(ex.map(compile_one, zip(srcs, objs)))
    if verbose:
        sys.stderr.write("\n".join(logs))
    tmp_lib = os.path.join(tmp, "libedb.so")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp_lib, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    deps = srcs + [os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(INCLUDE, "edb.h")]
    tmp_stamp = os.path.join(tmp, "stamp")
    with open(tmp_stamp, "w") as f:
        f.write(_digest(deps))
    os.replace(tmp_lib, LIB_PATH)
    os.replace(tmp_stamp, os.path.join(BUILD_DIR, "stamp"))
    shutil.rmtree(tmp, ignore_errors=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
