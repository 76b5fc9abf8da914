"""Build oracle/_ref/libgsr_refshaders{,_libm}.so: the reference's six compute shaders compiled for the CPU.

TEST INFRASTRUCTURE.  Recipe (the reference compiled from the sources where they lie):
  $GSR_REFERENCE_DIR/resources/shaders/compute/*.glsl --translate.py--> C++ in a temporary directory
  --g++ -ffp-contract=off, glsl_emu.hpp--> oracle/_ref/*.so        (git-ignored; travels to the GPU box)
No reference source is written into the repository; the temporary C++ is deleted after the link.
Two variants: exp()/pow() from the oracle's deterministic orc_exp/orc_pow (bit-exact comparisons with gsr_oracle.c),
and `_libm` with glibc expf/powf (an independent implementation of the implementation-defined built-ins).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.dirname(HERE)
OUT_DIR = os.path.join(ORACLE_DIR, "_ref")
# a checkout of the original project; without it only prebuilt libraries count (tests use tests/golden instead)
REFERENCE_DIR = os.environ.get("GSR_REFERENCE_DIR", "")
REFERENCE_SHADERS = os.path.join(REFERENCE_DIR, "resources", "shaders", "compute")
SHADERS = ("gsplat_projection", "radix_sort_upsweep", "radix_sort_spine", "radix_sort_downsweep", "gsplat_boundaries",
           "gsplat_render")
CXX = os.environ.get("ORC_CXX", "/usr/bin/g++")
CXXFLAGS = ["-std=gnu++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fwrapv", "-fPIC", "-w"]


def lib_path(libm: bool = False) -> str:
    return os.path.join(OUT_DIR, "libgsr_refshaders_libm.so" if libm else "libgsr_refshaders.so")


def reference_available() -> bool:
    return bool(REFERENCE_DIR) and all(os.path.isfile(os.path.join(REFERENCE_SHADERS, s + ".glsl")) for s in SHADERS)


def build(force: bool = False, verbose: bool = False) -> bool:
    """Returns True when both libraries exist afterwards.  Without the reference only prebuilt files count."""
    have = os.path.isfile(lib_path(False)) and os.path.isfile(lib_path(True))
    if not reference_available():
        return have
    deps = [os.path.join(HERE, f) for f in ("glsl_emu.hpp", "translate.py", "build_ref.py")]
    deps += [os.path.join(REFERENCE_SHADERS, s + ".glsl") for s in SHADERS]
    if have and not force:
        newest = max(os.path.getmtime(d) for d in deps)
        if min(os.path.getmtime(lib_path(False)), os.path.getmtime(lib_path(True))) >= newest:
            return True
    sys.path.insert(0, HERE)
    try:
        from translate import translate
    finally:
        sys.path.pop(0)
    os.makedirs(OUT_DIR, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="gsr_refshaders_")
    try:
        sources = []
        for s in SHADERS:
            with open(os.path.join(REFERENCE_SHADERS, s + ".glsl")) as f:
                cpp = translate(f.read(), s)
            path = os.path.join(tmp, s + ".cpp")
            with open(path, "w") as f:
                f.write(cpp)
            sources.append(path)
        for libm in (False, True):
            cmd = [CXX, *CXXFLAGS, "-I", HERE, "-shared", "-o", lib_path(libm), *sources]
            if libm:
                cmd += ["-DGLSL_EMU_LIBM", "-lm"]
            else:
                cmd += ["-L", ORACLE_DIR, "-l:libgsr_oracle.so", "-Wl,-rpath,$ORIGIN/..", "-lm"]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return True


if __name__ == "__main__":
    ok = build(force="--force" in sys.argv, verbose=True)
    print("refshaders:", "built" if ok else "unavailable (GSR_REFERENCE_DIR unset and no prebuilt oracle/_ref)")
