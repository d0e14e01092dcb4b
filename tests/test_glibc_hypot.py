"""glibc_hypot (navigation_b200/csrc/glibc_hypot.cuh), the hypot the TrajectoryPlanner's device fleet step computes,
against the running libm's hypot bit for bit, without a GPU: tests/cpp/glibc_hypot_check.cpp built with g++ compares
17 x 10^6 pairs (whole exponent range, the planner's range, integers, equal arguments, zeros, subnormals, the cutoffs of
the scaled paths, +-inf / NaN).  On glibc 2.35+ every pair agrees and glibc_hypot_matches_libm() says so; on a libm that
computes hypot another way some pair differs, and the probe must then say so too."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_glibc_hypot_matches_libm_bit_for_bit(tmp_path):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    exe = tmp_path / "glibc_hypot_check"
    subprocess.check_call([gxx, "-O2", "-ffp-contract=off", "-std=c++17", "-o", str(exe),
                           os.path.join(ROOT, "tests", "cpp", "glibc_hypot_check.cpp"), "-lm"])
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    m = re.search(r"pairs (\d+) mismatches (\d+) probe (\d)", out)
    assert m, out
    pairs, mismatches, probe = (int(g) for g in m.groups())
    assert pairs >= 10_000_000
    if mismatches:  # another libm: the device step must refuse, so the probe has to notice
        assert probe == 0, out
    else:
        assert probe == 1, out
