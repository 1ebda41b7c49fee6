"""In-tree build of libmcskin_cuda.so (nvcc, sm_100a).  No JIT cache: the .so lives
next to the package so it travels with the repo snapshot to the GPU box."""
from __future__ import annotations

import fcntl
import hashlib
import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "_lib"
LIB_PATH = LIB_DIR / "libmcskin_cuda.so"

# kernels_plain.cu / wavefront_plain.cu: the same kernels built without pose code (csrc/dev_types.cuh)
# kernels_counter.cu / wavefront_counter.cu: the general kernels with counter-based random streams (McConfig::rng_mode 1)
CUDA_SOURCES = ["kernels.cu", "wavefront.cu", "kernels_plain.cu", "wavefront_plain.cu", "kernels_counter.cu",
                "wavefront_counter.cu", "capi.cu", "context.cu", "frame.cu", "host_out.cu", "batch.cu"]
HOST_SOURCES = ["host_prep.cpp", "skin_scene.cpp", "host_copy.cpp"]

# --fmad=false: the geometry chain must round like the x86-64 reference build (no FMA);
# IEEE division and sqrt are nvcc's defaults and are left alone (no -use_fast_math).
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo", "--fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; the CUDA extension cannot be built")


def _source_digest() -> str:
    """Hash of everything the library is built from (file contents, not mtimes: the snapshot that
    travels to the GPU box does not preserve a meaningful order of timestamps)."""
    h = hashlib.sha1(" ".join(NVCC_FLAGS).encode())
    for path in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.cpp")) +
                       list(CSRC.glob("*.hpp")) + [ROOT / "include" / "mcskin_cuda.h"]):
        h.update(path.name.encode())
        h.update(path.read_bytes())
    return h.hexdigest()


def needs_build() -> bool:
    stamp = LIB_DIR / "build.hash"
    return not LIB_PATH.exists() or not stamp.exists() or stamp.read_text().strip() != _source_digest()


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB_PATH
    LIB_DIR.mkdir(exist_ok=True)
    # one builder at a time (torchrun starts one process per GPU, all of which may get here)
    with open(LIB_DIR / ".build.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB_PATH
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> Path:
    obj_dir = LIB_DIR / "obj"
    obj_dir.mkdir(exist_ok=True)
    nvcc = _nvcc()
    inc = ["-I", str(ROOT / "include"), "-I", str(CSRC)]
    procs = []
    objs = []
    for src in CUDA_SOURCES + HOST_SOURCES:
        obj = obj_dir / (src.rsplit(".", 1)[0] + ".o")
        objs.append(str(obj))
        cmd = [nvcc, *NVCC_FLAGS, *inc, "-c", str(CSRC / src), "-o", str(obj)]
        if src.endswith(".cu"):
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    (LIB_DIR / "build.log").write_text("\n".join(log))
    tmp = LIB_DIR / f".libmcskin_cuda.{os.getpid()}.so"
    link = [nvcc, "-shared", "-o", str(tmp), *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB_PATH)  # atomic: a concurrent dlopen sees the old or the new file, never half of one
    (LIB_DIR / "build.hash").write_text(_source_digest())
    if verbose:
        print("\n".join(log))
    return LIB_PATH


def build_variant(name: str, extra_flags: list[str]) -> Path:
    """A tuning variant of the library: _lib/variants/libmcskin_cuda_<name>.so (select with MCSKIN_LIB)."""
    vdir = LIB_DIR / "variants"
    obj_dir = vdir / f"obj_{name}"
    obj_dir.mkdir(parents=True, exist_ok=True)
    nvcc = _nvcc()
    inc = ["-I", str(ROOT / "include"), "-I", str(CSRC)]
    procs, objs = [], []
    for src in CUDA_SOURCES + HOST_SOURCES:
        obj = obj_dir / (src.rsplit(".", 1)[0] + ".o")
        objs.append(str(obj))
        procs.append((src, subprocess.Popen([nvcc, "-Xptxas", "-v", *NVCC_FLAGS, *extra_flags, *inc, "-c", str(CSRC / src), "-o", str(obj)],
                                            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    out_path = vdir / f"libmcskin_cuda_{name}.so"
    r = subprocess.run([nvcc, "-shared", "-o", str(out_path), *objs, "-gencode", "arch=compute_100a,code=sm_100a"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(r.stderr)
    (vdir / f"build_{name}.log").write_text("\n".join(log))
    return out_path


if __name__ == "__main__":
    print(build(force=True, verbose=True))
