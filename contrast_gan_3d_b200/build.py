"""Build libcgan3d.so in-tree with nvcc for sm_100a (no torch/pybind involved: plain C ABI)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
OBJ = PKG / "build"
LIB = PKG / "libcgan3d.so"
SOURCES = ["api_misc.cu", "conv_api.cu", "conv_generic.cu", "conv_tc.cu", "conv_tc_prog.cu", "conv_tc_prog_ks1.cu", "conv_tc_prog_ks2.cu", "conv_tc_prog_ks4.cu", "conv_tc_prog_ks8.cu", "conv_thin_tc.cu", "wgrad7_v2.cu", "conv_d1_tc.cu", "wgrad_tc.cu", "wgrad_s2_tc.cu", "norm_act.cu", "loss_optim.cu", "augment.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "--expt-extended-lambda", "-I", str(ROOT / "include"), "-I", str(CSRC)]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and Path(c).exists():
            return c
    raise RuntimeError("nvcc not found")


def _digest(paths) -> str:
    """Digest of the sources and of the flags that shape the binary.  Location-independent: the repository is checked out
    under different roots (authoring container, GPU box), and a digest that contained the absolute -I paths made every
    process on the GPU box rebuild the shipped library — eight ranks at once, racing on the same output file."""
    h = hashlib.sha256()
    for p in sorted(paths):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(f for f in NVCC_FLAGS if not f.startswith(str(ROOT))).encode())
    return h.hexdigest()


def _deps():
    return list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [ROOT / "include" / "cgan3d.h"]


def have_nvcc() -> bool:
    try:
        _nvcc()
        return True
    except RuntimeError:
        return False


def is_current() -> bool:
    """True when libcgan3d.so exists and was built from exactly the sources that are in the tree now."""
    stamp = OBJ / "stamp"
    return LIB.exists() and stamp.exists() and stamp.read_text() == _digest(_deps())


def build(force: bool = False, verbose: bool = False) -> Path:
    stamp = OBJ / "stamp"
    dig = _digest(_deps())
    if not force and LIB.exists() and stamp.exists() and stamp.read_text() == dig:
        return LIB
    OBJ.mkdir(exist_ok=True)
    # one builder at a time (ranks of one job share the tree): the others wait, then find the stamp up to date
    import fcntl

    with open(OBJ / "lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and LIB.exists() and stamp.exists() and stamp.read_text() == dig:
            return LIB
        return _build_locked(dig, stamp, verbose)


def _build_locked(dig: str, stamp: Path, verbose: bool) -> Path:
    nvcc = _nvcc()

    def compile_one(src: str):
        obj = OBJ / (src[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return str(obj)

    with ThreadPoolExecutor(max_workers=min(os.cpu_count() or 8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = LIB.with_suffix(".so.tmp")
    r = subprocess.run([nvcc, "-shared", "-o", str(tmp), *objs, "-lcudart"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB)  # atomic: a concurrent dlopen sees the old or the new library, never a partial one
    stamp.write_text(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
