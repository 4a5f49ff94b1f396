"""Build recipe for the compiled checker under oracle/ (test infrastructure; never the product path).

`oracle/ref_eigen/regenie_ref_eigen.cpp` (our C++ restatement of the reference's level-0 / score-test arithmetic) is
compiled against the reference's OWN vendored Eigen, where it lies: /root/reference/external_libs/eigen-3.4.0.  Flags
follow the reference Makefile (:33 `-O3 -ffast-math`, :49 `-fopenmp`).  Outputs go to oracle/_ref/ only (git-ignored,
shipped to the GPU box with the snapshot; /root/reference does not exist there, so the prebuilt files are used).

Also built here: the reference's vendored pgenlib itself (external_libs/pgenlib, plain g++ over its own few sources, no
cmake / external libraries) behind oracle/ref_pgenlib/pgen_ref_shim.cpp -> oracle/_ref/libpgenlib_ref.so, the reference
reader of the .pgen path.

Two Eigen objects are built: the reference's default code generation (no -march: SSE2 Eigen kernels, what `make` gives), and
an AVX2+FMA build that the wrapper prefers when the host CPU has it (the faster, more generous CPU baseline).
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
SRC = os.path.join(HERE, "ref_eigen", "regenie_ref_eigen.cpp")
EIGEN = os.environ.get("RG_REF_EIGEN", "/root/reference/external_libs/eigen-3.4.0")
LIBS = {"libregenie_ref_eigen.so": [], "libregenie_ref_eigen_avx2.so": ["-mavx2", "-mfma"]}


PGENLIB = os.environ.get("RG_REF_PGENLIB", "/root/reference/external_libs/pgenlib")
PGEN_SHIM = os.path.join(HERE, "ref_pgenlib", "pgen_ref_shim.cpp")
PGEN_LIB = os.path.join(OUT, "libpgenlib_ref.so")


def _skip(name, src):
    """Without the reference's sources the checker is optional: the tests compare with its stored outputs
    (tests/golden/ref/) and bench.py leaves out its CPU baseline."""
    sys.stderr.write("oracle/_ref/%s not built: the reference's sources (%s) are not available\n" % (name, src))


def build_pgenlib(verbose=False):
    """The reference's vendored pgenlib, from its own sources where they lie (its Makefile: g++ -O3 -std=c++11 over
    include/*.cc, *.cpp, *.cc with -I simde -I include), plus oracle/ref_pgenlib/pgen_ref_shim.cpp -> oracle/_ref/."""
    import glob
    gxx = shutil.which("g++")
    if not (os.path.isdir(PGENLIB) and gxx):
        if not os.path.exists(PGEN_LIB):
            _skip("libpgenlib_ref.so", PGENLIB)
        return                                 # a prebuilt checker is used as it is
    if os.path.exists(PGEN_LIB) and os.path.getmtime(PGEN_LIB) > max(os.path.getmtime(PGEN_SHIM), os.path.getmtime(__file__)):
        return
    os.makedirs(OUT, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(PGENLIB, "include", "*.cc")) + glob.glob(os.path.join(PGENLIB, "*.cpp")) +
                  glob.glob(os.path.join(PGENLIB, "*.cc")))
    cmd = [gxx, "-O3", "-std=c++11", "-fPIC", "-shared", "-w", "-I", PGENLIB, "-I", os.path.join(PGENLIB, "simde"),
           "-I", os.path.join(PGENLIB, "include"), "-o", PGEN_LIB, PGEN_SHIM] + srcs
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("oracle build failed: " + " ".join(cmd))


def build(verbose=False):
    build_pgenlib(verbose)
    gxx = shutil.which("g++")
    have_src = os.path.isdir(EIGEN) and gxx is not None
    for name, extra in LIBS.items():
        lib = os.path.join(OUT, name)
        if not have_src:
            if not os.path.exists(lib):
                _skip(name, EIGEN)
            continue                           # a prebuilt checker is used as it is
        if os.path.exists(lib) and os.path.getmtime(lib) > max(os.path.getmtime(SRC), os.path.getmtime(__file__)):
            continue
        os.makedirs(OUT, exist_ok=True)
        cmd = [gxx, "-O3", "-ffast-math", "-fopenmp", "-std=c++14", "-fPIC", "-shared", "-Wall", "-Wno-unused-local-typedefs",
               "-Wno-deprecated-declarations", "-DNDEBUG", "-I", EIGEN] + extra + ["-o", lib, SRC]
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("oracle build failed: " + " ".join(cmd))


if __name__ == "__main__":
    build(verbose=True)
