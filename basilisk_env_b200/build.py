"""In-tree build of the CUDA library (libbskenv.so) for sm_100a with plain nvcc.

nvcc cross-compiles without a GPU, so this runs on the CPU build box; the .so travels to the GPU box
with the repo snapshot (git-ignored, not gpurun-ignored).  Staleness is decided on a content hash of
the sources and flags (written next to the library), not on mtimes: a fresh checkout next to a shipped
.so has arbitrary mtimes."""
import hashlib
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("BSKENV_LIB") or os.path.join(HERE, "libbskenv.so")   # BSKENV_LIB: load a tuning variant instead
SOURCES = ["bskenv.cu", "opnav.cu"]
DEPS = ["bskenv.cu", "batch_common.cuh", "leo_core.cuh", "leo_split.cuh", "leo_f32.cuh", "leo_params.h", "leo_host.h", "opnav.cu",
        "opnav_core.cuh", "opnav_params.h", "opnav_host.h", os.path.join("..", "..", "include", "bskenv.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: cannot build libbskenv.so")
    return p


def source_hash(extra_flags=()):
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS + list(extra_flags)).encode())
    for d in DEPS:
        p = os.path.join(CSRC, d)
        if os.path.exists(p):
            h.update(d.encode())
            h.update(open(p, "rb").read())
    return h.hexdigest()


def is_stale(lib=None):
    lib = lib or LIB
    stamp = lib + ".stamp"
    if not os.path.exists(lib) or not os.path.exists(stamp):
        return True
    return open(stamp).read().strip() != source_hash()


def build(force=False, extra_flags=(), verbose=False, out=None):
    if out is None and not force and not is_stale():
        return LIB
    out = out or LIB
    objdir = os.path.join(HERE, "build", os.path.basename(out) + ".obj")
    os.makedirs(objdir, exist_ok=True)
    nvcc = nvcc_path()
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(s):
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + ["-c", "-o", obj, os.path.join(CSRC, s)]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd, cwd=CSRC)
        return obj

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:      # one nvcc per translation unit, side by side
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out] + objs
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd, cwd=CSRC)
    if not extra_flags:
        with open(out + ".stamp", "w") as f:
            f.write(source_hash())
    return out


LITERAL_LIB = os.path.join(HERE, "libbskenv_literal.so")


def build_literal(force=False):
    """PARITY BUILD (tests only): the same library with -DLEO_LITERAL_ECLIPSE, i.e. the penumbra evaluated exactly as
    Basilisk's eclipse.cpp writes it instead of the regrouped production form (DESIGN.md section 9, deviation D7).
    Loaded through BSKENV_LIB by tests/eclipse_probe.py; never by the product."""
    stamp = LITERAL_LIB + ".stamp"
    want = source_hash(("-DLEO_LITERAL_ECLIPSE",))
    if not force and os.path.exists(LITERAL_LIB) and os.path.exists(stamp) and open(stamp).read().strip() == want:
        return LITERAL_LIB
    build(extra_flags=("-DLEO_LITERAL_ECLIPSE",), out=LITERAL_LIB)
    with open(stamp, "w") as f:
        f.write(want)
    return LITERAL_LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
