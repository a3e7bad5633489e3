"""Host logic of the balanced plans (``bodge_b200/csrc/work_lists.h``): the planner that cuts the (panel, patch column, plane)
space of a two-step launch into one chunk per CTA slot is plain C++ -- ``tests/cpp/work_lists_check.cpp`` compiles it with
the host compiler and checks 13 k plans for exact cover, bounds, slot count and the cost it reports, and the choice between
the classic and the balanced plan (``choose_work_plan``) with the lists it uploads.  No GPU."""

import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)


def test_balanced_plans_cover_the_launch_exactly_once(tmp_path):
    cxx = os.environ.get("CXX") or shutil.which("g++")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if not cxx or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA headers (host-only compile)")
    exe = str(tmp_path / "work_lists_check")
    subprocess.run([cxx, "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(REPO, "bodge_b200", "csrc"),
                    "-I", os.path.join(REPO, "include"), "-I", cuda_inc, "-o", exe,
                    os.path.join(HERE, "cpp", "work_lists_check.cpp")], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout + out.stderr
