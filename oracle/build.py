"""Build recipe for the oracle (TEST INFRASTRUCTURE ONLY -- see oracle/oracle.cpp header).

    python oracle/build.py        ->  oracle/liboracle.so

The reference itself (C# + GLSL) cannot be compiled in this image (no dotnet/mono, no GL, no glslang), so there is
no oracle/_ref: the oracle is a CPU restatement ("port") and parity is unpinned by the reference (DESIGN.md).
"""
import os
import subprocess

ORACLE_DIR = os.path.dirname(os.path.abspath(__file__))
LIBORACLE = os.path.join(ORACLE_DIR, "liboracle.so")


def build(force=False, verbose=False):
    src = os.path.join(ORACLE_DIR, "oracle.cpp")
    deps = [src] + [os.path.join(ORACLE_DIR, f) for f in ("oracle_vxgi.inc", "oracle_post.inc")] + [os.path.join(ORACLE_DIR, "..", "include", f) for f in ("idkpt.h", "idkvx.h", "idk_gpu_types.h")]
    if not force and os.path.exists(LIBORACLE) and all(os.path.getmtime(d) <= os.path.getmtime(LIBORACLE) for d in deps):
        return LIBORACLE
    cmd = ["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread",
           "-fvisibility=hidden", "-o", LIBORACLE, src]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIBORACLE


if __name__ == "__main__":
    print(build(force=True, verbose=True))
