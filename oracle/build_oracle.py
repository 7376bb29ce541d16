"""Build the oracle's C restatement (TEST INFRASTRUCTURE): oracle/libwavernn_twin.so.

gcc -O2 -ffp-contract=off so that every a*b+c stays two rounded operations unless written as
fmaf() - the arithmetic contract shared with the CUDA kernel (include/mb_wavernn_math.h).
The reference is pure Python with ONE compiled piece on the edge of the path: monotonic_align/core.pyx (Cython, 42 lines;
SURVEY.md 8f row N4).  build_ref() compiles THAT FILE, from where it lies in the reference tree (ref_harness.REFERENCE_ROOT),
with `cython` + gcc into oracle/_ref/monotonic_align_core*.so (git-ignored) - the real reference for that row, whose outputs
oracle/make_golden_pinned.py stores for the tests; nothing of the reference is copied into the repo.  Everything else has no
C/C++ reference to compile.
"""
from __future__ import annotations

import subprocess
from pathlib import Path

from ref_harness import REFERENCE_ROOT

HERE = Path(__file__).resolve().parent
SRC = HERE / "wavernn_twin.c"
LIB = HERE / "libwavernn_twin.so"


def build(force: bool = False) -> Path:
    hdr = HERE.parent / "include" / "mb_wavernn_math.h"
    if not force and LIB.is_file() and LIB.stat().st_mtime >= max(SRC.stat().st_mtime, hdr.stat().st_mtime):
        return LIB
    cmd = ["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-fopenmp", "-fPIC", "-shared",
           "-o", str(LIB), str(SRC), "-lm"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return LIB


REF_DIR = HERE / "_ref"
REF_PYX = REFERENCE_ROOT / "monotonic_align" / "core.pyx"


def ref_so():
    """path of the compiled reference module if it exists (oracle/_ref/monotonic_align_core.*.so)"""
    hits = sorted(REF_DIR.glob("monotonic_align_core*.so")) if REF_DIR.is_dir() else []
    return hits[0] if hits else None


def build_ref(force: bool = False):
    """compile the reference's own monotonic_align/core.pyx into oracle/_ref (needs the reference tree)"""
    import sysconfig

    if not REF_PYX.is_file():
        return ref_so()
    if not force and ref_so() is not None:
        return ref_so()
    REF_DIR.mkdir(exist_ok=True)
    c_file = REF_DIR / "monotonic_align_core.c"
    # cython names the module after the OUTPUT file: the init symbol becomes PyInit_monotonic_align_core
    subprocess.run(["cython", "-3", str(REF_PYX), "-o", str(c_file)], check=True, capture_output=True, text=True)
    ext = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    out = REF_DIR / ("monotonic_align_core" + ext)
    inc = sysconfig.get_paths()["include"]
    subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", inc, "-o", str(out), str(c_file)], check=True,
                   capture_output=True, text=True)
    c_file.unlink()
    return out


if __name__ == "__main__":
    print(build(force=True))
    print(build_ref(force=True))
