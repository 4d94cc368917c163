"""Build libprmf_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import contextlib
import fcntl
import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libprmf_b200.so")
HEADER = os.path.join(HERE, "..", "include", "prmf_b200.h")
# translation unit -> headers it depends on
SOURCES = {
    "prmf_b200.cu": ["kernels.cuh", "block_params.h", "tf32.cuh", "nccl_dyn.h", "nnls_init.cuh"],
    "block.cu": ["kernels.cuh", "block_params.h", "block.cuh"],
    "preprocess.cu": [],
    "cv.cu": [],
    "host_logic.cpp": [],
}
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libprmf_b200.so cannot be built")


def _mtime(path):
    return os.path.getmtime(path) if os.path.exists(path) else 0.0


def _obj(src):
    return os.path.join(OBJDIR, os.path.splitext(src)[0] + ".o")


def _stale_objects():
    out = []
    for src, deps in SOURCES.items():
        newest = max([_mtime(os.path.join(CSRC, src)), _mtime(HEADER)] + [_mtime(os.path.join(CSRC, d)) for d in deps])
        if _mtime(_obj(src)) < newest:
            out.append(src)
    return out


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for src, deps in SOURCES.items():
        for f in [src] + deps:
            if _mtime(os.path.join(CSRC, f)) > t:
                return True
    return _mtime(HEADER) > t


@contextlib.contextmanager
def _build_lock():
    """One builder at a time (torchrun ranks and restart workers all reach `_lib.load()` at once): an exclusive
    flock for the whole compile + link."""
    os.makedirs(OBJDIR, exist_ok=True)
    with open(os.path.join(OBJDIR, ".lock"), "w") as fh:
        fcntl.flock(fh, fcntl.LOCK_EX)
        try:
            yield
        finally:
            fcntl.flock(fh, fcntl.LOCK_UN)


def build_library(force=False, verbose=False):
    """Compile the CUDA sources (one object per translation unit, rebuilt only when stale) and link
    prmf_b200/libprmf_b200.so.  Returns the path.  Safe to call from several processes at once: the build runs
    under a file lock, whoever gets the lock second finds the library fresh, and the library appears
    atomically (linked to a temporary name, then renamed), so nobody can dlopen a half-written file."""
    if not force and not is_stale():
        return LIB
    with _build_lock():
        if not force and not is_stale():         # built by another process while we waited for the lock
            return LIB
        return _build_locked(force, verbose)


def _build_locked(force, verbose):
    nvcc = nvcc_path()
    todo = list(SOURCES) if force else (_stale_objects() or [s for s in SOURCES if not os.path.exists(_obj(s))])

    def compile_one(src):
        cmd = [nvcc, "-O3", "-std=c++17"] + ARCH + ["-lineinfo", "-Xcompiler", "-fPIC,-ffp-contract=off", "-c", "-o",
                                                     _obj(src), os.path.join(CSRC, src)]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        return src, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        for src, res in pool.map(compile_one, todo):
            if res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
                raise RuntimeError("nvcc failed on %s" % src)
            if verbose:
                sys.stderr.write(res.stdout + res.stderr)
    fd, tmp = tempfile.mkstemp(prefix=".libprmf_b200.", suffix=".so.tmp", dir=HERE)
    os.close(fd)
    try:
        link = [nvcc, "-shared"] + ARCH + ["-o", tmp] + [_obj(s) for s in SOURCES] + ["-ldl"]
        res = subprocess.run(link, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("linking libprmf_b200.so failed")
        os.chmod(tmp, 0o755)
        os.replace(tmp, LIB)
    finally:
        if os.path.exists(tmp):
            os.unlink(tmp)
    return LIB


def build_debug_library(defines, out_path, sources=("block.cu",)):
    """Developer builds with instrumentation macros (tools/*.py): a second library next to the product one, e.g.
    python -m prmf_b200.build --debug PRMF_BLOCK_TIMING  ->  tools/libprmf_dbg.so  (recompiles `sources` with -D...)"""
    build_library()
    nvcc = nvcc_path()
    objs = []
    for src in SOURCES:
        if src not in sources:
            objs.append(_obj(src))
            continue
        obj = os.path.join(OBJDIR, os.path.splitext(src)[0] + "_dbg.o")
        cmd = [nvcc, "-O3", "-std=c++17"] + ARCH + ["-lineinfo", "-Xcompiler", "-fPIC,-ffp-contract=off"] + \
              ["-D" + d for d in defines] + ["-c", "-o", obj, os.path.join(CSRC, src)]
        subprocess.run(cmd, check=True)
        objs.append(obj)
    subprocess.run([nvcc, "-shared"] + ARCH + ["-o", out_path] + objs + ["-ldl"], check=True)
    return out_path


if __name__ == "__main__":
    if "--debug" in sys.argv:
        defs = sys.argv[sys.argv.index("--debug") + 1:]
        print(build_debug_library(defs, os.path.join(HERE, "..", "tools", "libprmf_dbg.so")))
    else:
        print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
