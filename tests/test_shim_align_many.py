"""The C++ multi-align entry points of include/lgs/registration.hpp build against liblgs_b200.so with plain g++ (no GPU needed;
tests/test_gpu_ndt_align_many.py runs them)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_shim_align_many(tmpdir):
    exe = os.path.join(str(tmpdir), "shim_align_many")
    libdir = os.path.join(ROOT, "lidar_graph_slam_b200")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "shim_align_many.cpp"),
                           "-o", exe, "-L" + libdir, "-l:liblgs_b200.so", "-Wl,-rpath," + libdir, "-ldl", "-lpthread", "-lrt"])
    return exe


def test_cpp_align_many_shim_compiles_and_links(tmp_path):
    from lidar_graph_slam_b200 import _lib
    _lib.load()
    exe = build_shim_align_many(tmp_path)
    assert "shim compiled" in subprocess.check_output([exe]).decode()
