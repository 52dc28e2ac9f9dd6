"""Builds the C++ drop-in layer (Matcher / BA with the reference's interfaces,
bodies over the C ABI) together with the test harness into
lorb_slam_b200/lib/libhost_dropin.so.  Uses the shim headers because this image
has no OpenCV-C++; in a LORB-SLAM checkout the same two .cpp files compile
against the real include/ directory (INTEGRATION.md)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
LIBDIR = os.path.join(HERE, "..", "lib")
OUT = os.path.join(LIBDIR, "libhost_dropin.so")
SRCS = [os.path.join(HERE, "src", "matcher.cpp"), os.path.join(HERE, "src", "bundle_adjust.cpp"),
        os.path.join(HERE, "src", "ORBextractor.cpp"), os.path.join(HERE, "src", "local_map_index.cpp"),
        os.path.join(HERE, "src", "pose_optimization.cpp"), os.path.join(HERE, "src", "pose_from_matches.cpp"),
        os.path.join(HERE, "test", "harness.cpp")]


def _deps():
    d = list(SRCS)
    for root, _, files in os.walk(HERE):
        d += [os.path.join(root, f) for f in files if f.endswith((".h", ".hpp", ".inc"))]
    d.append(os.path.join(HERE, "..", "..", "include", "lorb_cuda.h"))
    return d


def build(force=False):
    from lorb_slam_b200 import build as libbuild
    libbuild.build_library()
    if not force and os.path.exists(OUT) and all(
            os.path.getmtime(p) <= os.path.getmtime(OUT) for p in _deps()):
        return OUT
    cmd = ["/usr/bin/g++", "-std=c++11", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-pthread",
           "-I", os.path.join(HERE, "shim"), "-o", OUT] + SRCS + [
        "-L", LIBDIR, "-llorb_cuda", "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building libhost_dropin.so")
    return OUT


if __name__ == "__main__":
    print(build(force=True))
