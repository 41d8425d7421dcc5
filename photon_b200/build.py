"""In-tree build of the sm_100a extension ``photon_b200/_C*.so``.

Plain ``nvcc`` / ``g++`` invocations (parallel, mtime-incremental) so that the
exact arch flags are under our control: ``-gencode arch=compute_100a,code=sm_100a
-lineinfo`` (tcgen05/TMA need the arch-specific ``a`` target).  The product is
kept in-tree so the GPU box sees it and the driver can record it as loaded.
"""
from __future__ import annotations

import os
import subprocess
import sys
import sysconfig
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "csrc"
OBJ = ROOT / "build" / "obj"
EXT_NAME = "_C"

CU_SOURCES = ["gemm_tcgen05.cu", "gemm_mxfp8.cu", "attention_tcgen05.cu", "fused_ops.cu", "fp8_ops.cu", "comm.cu", "decode.cu"]
CPP_SOURCES = ["bindings.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--use_fast_math", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def ext_path() -> Path:
    return ROOT / "photon_b200" / (EXT_NAME + sysconfig.get_config_var("EXT_SUFFIX"))


def _newer(src: Path, dst: Path, deps: list[Path]) -> bool:
    if not dst.exists():
        return True
    t = dst.stat().st_mtime
    return any(p.stat().st_mtime > t for p in [src, *deps] if p.exists())


def _run(cmd: list[str], log: Path | None = None) -> None:
    r = subprocess.run(cmd, capture_output=True, text=True)
    if log is not None:
        log.write_text(r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build step failed: " + " ".join(cmd[:6]) + " ...")


def build(force: bool = False, verbose: bool = True) -> Path:
    from torch.utils.cpp_extension import CUDA_HOME, include_paths, library_paths

    nvcc = str(Path(CUDA_HOME or "/usr/local/cuda") / "bin" / "nvcc")
    OBJ.mkdir(parents=True, exist_ok=True)
    headers = sorted(CSRC.glob("*.h")) + sorted(CSRC.glob("*.cuh"))
    incs = [f"-I{p}" for p in include_paths("cuda")] + [f"-I{sysconfig.get_paths()['include']}", f"-I{CSRC}"]
    jobs = []
    objs = []
    for s in CU_SOURCES:
        src, dst = CSRC / s, OBJ / (s + ".o")
        objs.append(dst)
        if force or _newer(src, dst, headers):
            jobs.append(([nvcc, *NVCC_FLAGS, f"-I{CSRC}", "-c", str(src), "-o", str(dst)], OBJ / (s + ".log")))
    defs = [f"-DTORCH_EXTENSION_NAME={EXT_NAME}", "-DTORCH_API_INCLUDE_EXTENSION_H", "-D_GLIBCXX_USE_CXX11_ABI=1"]
    for s in CPP_SOURCES:
        src, dst = CSRC / s, OBJ / (s + ".o")
        objs.append(dst)
        if force or _newer(src, dst, headers):
            jobs.append((["g++", "-O2", "-std=c++17", "-fPIC", "-w", *defs, *incs, "-c", str(src), "-o", str(dst)], None))
    if verbose and jobs:
        print(f"[photon_b200.build] compiling {len(jobs)} translation unit(s) for sm_100a ...", flush=True)
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 2)) as ex:
        list(ex.map(lambda j: _run(*j), jobs))
    out = ext_path()
    if force or jobs or not out.exists():
        libs = [f"-L{p}" for p in library_paths("cuda")]
        rpath = [f"-Wl,-rpath,{p}" for p in library_paths("cuda")]
        _run(["g++", "-shared", "-o", str(out), *[str(o) for o in objs], *libs, *rpath,
              "-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch", "-ltorch_python", "-lcudart"])
        if verbose:
            print(f"[photon_b200.build] linked {out}", flush=True)
    return out


def ptxas_report() -> str:
    """Concatenated ``-Xptxas -v`` logs (registers / spills / smem per kernel)."""
    return "\n".join(p.read_text() for p in sorted(OBJ.glob("*.log")))


def main() -> None:
    """Console entry point (``photon-build-kernels [--force]``)."""
    build(force="--force" in sys.argv)


if __name__ == "__main__":
    main()
