"""In-tree native builds for vcfx_b200 (no JIT cache: everything is built ahead of use, next to its sources).

* ``libvcfx_cuda.so``  — the product: hand-written sm_100a kernels + the C ABI
  (``include/vcfx_cuda.h``).  nvcc cross-compiles it without a GPU.
* ``libvcfx_synth.so`` — synthetic-input generator (plain C).
* ``bin/VCFX_*``       — the five drop-in command-line tools (C++ host code over the C ABI).
* ``oracle/_ref/``     — test infrastructure: the CPU restatement and, when ``VCFX_REFERENCE`` names
  a VCFX source tree, the unmodified reference tools.  Building the checker is
  not using it; nothing in this package imports it.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "vcfx_b200"
CSRC = PKG / "csrc"
TOOLS = PKG / "tools"
BIN = PKG / "bin"
INCLUDE = ROOT / "include"
ORACLE = ROOT / "oracle"

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUDA_LIB = PKG / "libvcfx_cuda.so"
SYNTH_LIB = PKG / "libvcfx_synth.so"
TOOL_NAMES = ["allele_freq_calc", "allele_counter", "missing_detector", "variant_counter", "hwe_tester", "nonref_filter", "indexer", "phase_checker", "inbreeding_calculator", "genotype_query", "dosage_calculator", "plink_bed"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",            # FP64 text must follow the reference's FMA-less op sequence
    "-Xcompiler", "-fPIC,-O2,-Wall",
    "-shared", "-cudart", "static",
]


def _newer(target: Path, sources) -> bool:
    if not target.exists():
        return False
    t = target.stat().st_mtime
    return all(Path(s).stat().st_mtime <= t for s in sources)


def _run(cmd, **kw):
    """Runs a compiler.  The file behind "-o" is written under a private name and renamed when it is complete: several
    processes (parallel test workers) may build the same target at once, and none of them may load a half-written one."""
    cmd = [str(c) for c in cmd]
    final = tmp = None
    if "-o" in cmd:
        i = cmd.index("-o") + 1
        final = Path(cmd[i]); tmp = final.with_name(f".{final.name}.{os.getpid()}")
        cmd[i] = str(tmp)
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    if r.returncode != 0:
        if tmp is not None and tmp.exists():
            tmp.unlink()
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError(f"build step failed: {cmd[0]}")
    if tmp is not None:
        os.replace(tmp, final)
    return r


def build_cuda(force: bool = False, verbose_ptxas: bool = False) -> Path:
    srcs = sorted(CSRC.glob("*.cu"))
    deps = srcs + sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) + sorted(INCLUDE.glob("*.h"))
    if not force and _newer(CUDA_LIB, deps):
        return CUDA_LIB
    flags = list(NVCC_FLAGS)
    if verbose_ptxas:
        flags += ["-Xptxas", "-v"]
    r = _run([NVCC, *flags, "-I", INCLUDE, "-I", CSRC, "-o", CUDA_LIB, *srcs])
    if verbose_ptxas:
        sys.stderr.write(r.stderr)
    return CUDA_LIB


def build_synth(force: bool = False) -> Path:
    src = CSRC / "vcfx_synth.c"
    if not force and _newer(SYNTH_LIB, [src]):
        return SYNTH_LIB
    _run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-o", SYNTH_LIB, src, "-lpthread"])
    return SYNTH_LIB


def build_tools(force: bool = False):
    BIN.mkdir(exist_ok=True)
    common = sorted(p for p in TOOLS.glob("*.cpp") if not p.name.startswith("VCFX_"))
    hdrs = sorted(TOOLS.glob("*.h")) + sorted(INCLUDE.glob("*.h"))
    out = []
    for t in TOOL_NAMES:
        src = TOOLS / f"VCFX_{t}.cpp"
        if not src.exists():
            continue
        exe = BIN / f"VCFX_{t}"
        if force or not _newer(exe, [src, *common, *hdrs, CUDA_LIB]):
            _run(["g++", "-O2", "-std=c++17", "-Wall", "-I", INCLUDE, "-I", TOOLS, src, *common,
                  "-o", exe, f"-L{PKG}", "-lvcfx_cuda", f"-Wl,-rpath,$ORIGIN/..", "-lz", "-lpthread", "-ldl", "-lrt"])
        out.append(exe)
    return out


def build_oracle(force: bool = False) -> Path:
    """Test infrastructure (see oracle/vcfx_oracle.h): the CPU restatement, and the unmodified reference tools
    (oracle/_ref/VCFX_*) when VCFX_REFERENCE names a VCFX source tree.  Without them the tests compare with recorded
    outputs (tests/reference_runs.py) and bench.py's reference legs fall back to the oracle or are left out."""
    if force:
        shutil.rmtree(ORACLE / "_ref" / "liboracle.so", ignore_errors=True)
    _run(["make", "-C", ORACLE, "all"])
    reference = os.environ.get("VCFX_REFERENCE")
    if reference:
        _run(["make", "-C", ORACLE, "ref", f"REFERENCE={reference}"])
    return ORACLE / "_ref" / "liboracle.so"


def build_all(force: bool = False):
    build_cuda(force)
    build_synth(force)
    build_tools(force)
    build_oracle(force)
