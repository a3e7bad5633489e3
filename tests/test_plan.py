"""Host logic of the stepping planner (``bodge_b200/csrc/cheb_plan.h``): which stepping, matrix format and panel width a
recursion runs on, or why it is refused, is plain C++ -- ``tests/cpp/plan_check.cpp`` compiles it with the host compiler and
checks ``plan_stepping`` over every consistent set of matrix facts, kernel number, column count and auto switch: the
refusals and their messages, the stepping and format each rule gives, the panel widths, and the bench systems' plans.
No GPU."""

import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)


def test_stepping_plans_follow_the_rules(tmp_path):
    cxx = os.environ.get("CXX") or shutil.which("g++")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if not cxx or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA headers (host-only compile)")
    exe = str(tmp_path / "plan_check")
    subprocess.run([cxx, "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(REPO, "bodge_b200", "csrc"),
                    "-I", os.path.join(REPO, "include"), "-I", cuda_inc, "-o", exe,
                    os.path.join(HERE, "cpp", "plan_check.cpp")], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok"), out.stdout + out.stderr
