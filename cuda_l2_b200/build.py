"""In-tree builds of the native pieces (nvcc cross-compiles sm_100a without a GPU).

Artifacts land in ``cuda_l2_b200/lib/`` (git-ignored, shipped to the GPU box by gpurun):

* ``libb200_hgemm.so``  — the C-ABI product library (include/b200_hgemm.h)
* ``libb200_baselines.so`` — cuBLAS / cuBLASLt comparators behind a C ABI (include/b200_baselines.h)
* ``dev_check``         — standalone bring-up / tuning binary (developer tool)

Every step is skipped when the artifact is newer than all of its inputs.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
REPO = PKG_DIR.parent
CSRC = PKG_DIR / "csrc"
LIB_DIR = PKG_DIR / "lib"

ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-gnu-unique"]


def nvcc_path() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(cand).exists():
        raise RuntimeError("nvcc not found: the B200 HGEMM library cannot be built")
    return cand


def _stale(out: Path, inputs: list[Path]) -> bool:
    if not out.exists():
        return True
    t = out.stat().st_mtime
    return any(p.stat().st_mtime > t for p in inputs if p.exists())


def _run(cmd: list[str], verbose: bool) -> None:
    if verbose:
        print("+", " ".join(cmd), flush=True)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError(f"build step failed ({r.returncode}): {' '.join(cmd)}")
    if verbose and r.stdout.strip():
        print(r.stdout)


def _headers() -> list[Path]:
    return sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.inc")) + sorted((REPO / "include").glob("*.h"))


def build_capi(verbose: bool = False, force: bool = False) -> Path:
    LIB_DIR.mkdir(exist_ok=True)
    out = LIB_DIR / "libb200_hgemm.so"
    src = CSRC / "b200_hgemm_capi.cu"
    if force or _stale(out, [src] + _headers()):
        _run([nvcc_path(), *ARCH_FLAGS, *COMMON, "--shared", "-o", str(out), str(src)], verbose)
    return out


def build_baselines(verbose: bool = False, force: bool = False) -> Path:
    LIB_DIR.mkdir(exist_ok=True)
    out = LIB_DIR / "libb200_baselines.so"
    src = CSRC / "b200_baselines_capi.cu"
    if force or _stale(out, [src] + _headers()):
        _run([nvcc_path(), *ARCH_FLAGS, *COMMON, "--shared", "-o", str(out), str(src), "-lcublas", "-lcublasLt"],
             verbose)
    return out


def build_dev_check(verbose: bool = False, force: bool = False) -> Path:
    lib = build_capi(verbose, force)
    build_baselines(verbose, force)
    out = LIB_DIR / "dev_check"
    src = CSRC / "dev_check.cu"
    if force or _stale(out, [src, lib] + _headers()):
        _run([nvcc_path(), *ARCH_FLAGS, "-std=c++17", "-O3", "-lineinfo", "-o", str(out), str(src),
              f"-L{LIB_DIR}", "-lb200_hgemm", "-lb200_baselines", "-lcublas", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"], verbose)
    return out


def build_variant(name: str, defines: list[str], verbose: bool = False, force: bool = False) -> Path:
    """Developer build of the library and of dev_check with extra -D flags: libb200_hgemm_<name>.so + dev_check_<name>.

    Not part of build_all(): the product library is always the plain build."""
    LIB_DIR.mkdir(exist_ok=True)
    build_baselines(verbose, force)
    flags = [f"-D{d}" for d in defines]
    lib = LIB_DIR / f"libb200_hgemm_{name}.so"
    src = CSRC / "b200_hgemm_capi.cu"
    if force or _stale(lib, [src] + _headers()):
        _run([nvcc_path(), *ARCH_FLAGS, *COMMON, *flags, "--shared", "-o", str(lib), str(src)], verbose)
    out = LIB_DIR / f"dev_check_{name}"
    dsrc = CSRC / "dev_check.cu"
    if force or _stale(out, [dsrc, lib] + _headers()):
        _run([nvcc_path(), *ARCH_FLAGS, "-std=c++17", "-O3", "-lineinfo", *flags, "-o", str(out), str(dsrc),
              f"-L{LIB_DIR}", f"-lb200_hgemm_{name}", "-lb200_baselines", "-lcublas", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"],
             verbose)
    return out


def build_trace(verbose: bool = False, force: bool = False) -> Path:
    """Per-CTA phase timestamps (-DB200_HGEMM_TRACE): libb200_hgemm_trace.so + dev_check_trace."""
    return build_variant("trace", ["B200_HGEMM_TRACE"], verbose, force)


def build_all(verbose: bool = False, force: bool = False) -> dict[str, Path]:
    out = {"capi": build_capi(verbose, force)}
    if (CSRC / "b200_baselines_capi.cu").exists():
        out["baselines"] = build_baselines(verbose, force)
    out["dev_check"] = build_dev_check(verbose, force)
    return out


if __name__ == "__main__":
    for k, v in build_all(verbose=True, force="--force" in sys.argv).items():
        print(f"{k}: {v}")
