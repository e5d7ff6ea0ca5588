"""CPU: the result-block layout shared by the lane buffers and the pinned result sets
(irmv_detection_b200/csrc/result_layout.h), compiled on its own with g++."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_result_layout_and_copy_plan(tmp_path):
    exe = tmp_path / "result_layout_test"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                    "-I", os.path.join(ROOT, "irmv_detection_b200", "csrc"),
                    os.path.join(ROOT, "tests", "cpp", "result_layout_test.cpp"), "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "RESULT_LAYOUT_OK" in r.stdout, r.stdout[-2000:]
