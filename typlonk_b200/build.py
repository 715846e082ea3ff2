"""Build libtyplonk_b200.so in-tree with nvcc for sm_100a (no torch involved).

    python -m typlonk_b200.build [--force]

The .so lands in typlonk_b200/lib/ (git-ignored, travels to the GPU box with the snapshot).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "csrc"
LIBDIR = ROOT / "lib"
LIB = LIBDIR / "libtyplonk_b200.so"
SOURCES = ["api.cu", "comm.cu", "ntt.cu", "msm.cu", "poly.cu", "prove_batch.cu", "prove_v2.cu", "srs.cu", "srs_ceremony.cu", "selftest.cu", "verify.cu", "verify_batch.cu", "verify_key.cu", "wire.cu", "trace.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O2",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stamp():
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cpp")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) +
                    [ROOT.parent / "include" / "typlonk_b200.h"]):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, defines=(), tag: str = "") -> Path:
    """`defines` / `tag` build an experimental variant libtyplonk_b200_<tag>.so (selected at run
    time with TYPLONK_B200_LIB); the default build takes neither."""
    LIBDIR.mkdir(exist_ok=True)
    lib = LIBDIR / ("libtyplonk_b200_%s.so" % tag) if tag else LIB
    # The hash of every source + flag is compiled INTO the library (tp_build_stamp, api.cu) and compared with the
    # sources on disk: a stale .so left behind by a checkout can never pass for a current one (no side file).
    stamp = hashlib.sha256((_stamp() + "|" + " ".join(defines)).encode()).hexdigest()
    if not force and lib.exists() and ("tp-build-stamp:" + stamp).encode() in lib.read_bytes():
        return lib
    nvcc = _nvcc()
    objdir = LIBDIR / ("obj" + ("_" + tag if tag else ""))
    objdir.mkdir(exist_ok=True)

    def compile_one(src):
        obj = objdir / (src.rsplit(".", 1)[0] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *["-D" + d for d in defines], "-c", str(CSRC / src), "-o", str(obj)]
        if src == "api.cu":
            cmd.insert(1, '-DTP_BUILD_STAMP="%s"' % stamp)
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, res.stdout, res.stderr))
        if verbose:
            print(res.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    # NCCL is loaded with dlopen at run time (comm.cu): only libdl is linked
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(lib), *map(str, objs), "-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (res.stdout, res.stderr))
    return lib


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    tags = [a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--tag=")]
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs, tag=tags[0] if tags else "")
    print(path)
