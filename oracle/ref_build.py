#!/usr/bin/env python
"""TEST INFRASTRUCTURE: build oracle/_ref/libmadigan_ref.so from the REFERENCE's own sources.

The reference's C++ env needs Eigen, HighFive/HDF5 and CMake with hard-coded conda paths
(environments/cpp/CMakeLists.txt:5-15); none of that exists here and there is no network.  Its env path,
however, compiles from a handful of its source files with g++ directly once `Eigen/Core` and the HighFive
headers resolve -- oracle/ref_shim provides a small eager Eigen subset (left-to-right folds) and throwing
HighFive stubs.  The reference sources are compiled WHERE THEY LIE, in the madigan checkout that MADIGAN_REFERENCE
names (never copied); without it there is nothing to build.
pybind11 + Python headers are real (the reference headers include them).  Strict IEEE flags instead of the
reference's -ffast-math -mfma, so that the result is reproducible and comparable bit for bit.
"""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.environ["MADIGAN_REFERENCE"], "madigan", "environments", "cpp") \
    if os.environ.get("MADIGAN_REFERENCE") else None
OUT = os.path.join(HERE, "_ref")
LIB = os.path.join(OUT, "libmadigan_ref.so")
SOURCES = ["Portfolio.cpp", "Account.cpp", "Broker.cpp", "DataSource.cpp", "Config.cpp"]


def build(verbose=False):
    if not REF or not os.path.isdir(REF):
        return None
    import pybind11
    os.makedirs(OUT, exist_ok=True)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-w",
           "-I", os.path.join(HERE, "ref_shim"), "-I", REF, "-I", pybind11.get_include(),
           "-I", sysconfig.get_paths()["include"],
           os.path.join(HERE, "ref_driver.cpp")] + [os.path.join(REF, s) for s in SOURCES] + ["-o", LIB]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stderr[-6000:])
        raise RuntimeError("reference build failed")
    if verbose:
        print(LIB)
    return LIB


if __name__ == "__main__":
    build(verbose=True)
