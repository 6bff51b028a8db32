"""GPU test (-m gpu) of the straight-line arithmetic of the map-point unary (csrc/unary_obs.cuh) against the library
sequences it replaces.  tests/cuda/unary_obs_check.cu is compiled with the library's own nvcc flags (from the
Makefile) into a temporary directory and run once; it prints one line of counters:
  * the fast reciprocal over all 2^32 bit patterns: equal to __frcp_rn wherever it is not flagged, and flagged
    exactly for the exponent fields outside [1, 252];
  * the Newton square root at the decision boundary (every offset within +-2^15 double ulps of float rounding
    midpoints, midpoints included) and on 2^30 log-uniform inputs: (float)y equal to (float)__dsqrt_rn(s) wherever
    not flagged; its largest error in double ulps must stay within half the +-2^13-ulp window that flags;
  * the limits of the range check and the special values: flagged;
  * observe_fast against observe on 2^28 random and crafted tuples: bit-identical wherever not flagged."""
import os
import re
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lc-crf-slam_b200", "csrc")


def makefile_flags():
    """ARCH and the code-generation part of NVFLAGS as the library is built with them"""
    text = open(os.path.join(CSRC, "Makefile")).read().replace("\\\n", " ")
    var = dict(re.findall(r"^(\w+)\s*:=\s*(.*)$", text, re.M))
    flags = var["NVFLAGS"].replace("$(ARCH)", var["ARCH"]).split()
    keep, skip = [], False
    for f in flags:
        if skip:
            skip = False
        elif f in ("-Xcompiler", "-Xptxas"):
            skip = True   # host warnings and the ptxas report are not needed here
        elif not f.startswith("$("):
            keep.append(f)
    for f in ("-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false", "sm_100a"):
        assert any(f in k for k in keep), f
    return keep


def nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    pytest.fail("nvcc not found")


def test_unary_fast_path_arithmetic(tmp_path):
    exe = str(tmp_path / "unary_obs_check")
    subprocess.run([nvcc(), *makefile_flags(), "-I", CSRC, "-o", exe, os.path.join(ROOT, "tests", "cuda", "unary_obs_check.cu")],
                   check=True, timeout=300)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    print(p.stdout, p.stderr)
    assert p.returncode == 0, p.stderr
    line = [l for l in p.stdout.splitlines() if l.startswith("unary_obs ")]
    assert len(line) == 1, p.stdout
    c = {k: int(v) for k, v in re.findall(r"(\w+)=(-?\d+)", line[0])}
    # reciprocal: all 2^32 patterns; flagged = exponent fields 0, 253, 254, 255
    assert c["rcp_n"] == 1 << 32
    assert c["rcp_flag_bad"] == 0 and c["rcp_bad"] == 0
    assert c["rcp_flagged"] == 4 << 23 << 1
    # square root at the decision boundary: 60 binades x 64 floats x (2^16 + 1) offsets
    assert c["bnd_n"] == 60 * 64 * ((1 << 16) + 1)
    assert c["bnd_bad"] == 0
    # the window flags +-2^13 ulps around each midpoint: at least the offsets within it minus the Newton error
    assert c["bnd_flagged"] >= 60 * 64 * (1 << 13)
    assert 0 < c["bnd_margin_ulps"] <= 1 << 12, "Newton error %d double ulps" % c["bnd_margin_ulps"]
    # random inputs: flagged at about the window's share 2^-15
    assert c["rnd_n"] >= 1 << 30 and c["rnd_bad"] == 0
    rate = c["rnd_flagged"] / c["rnd_n"]
    assert 0.5 * 2 ** -15 < rate < 2 * 2 ** -15, rate
    assert c["rnd_margin_ulps"] <= 1 << 12
    assert c["spc_n"] == 22 and c["spc_bad"] == 0
    # end to end
    assert c["e2e_n"] >= 1 << 28
    assert c["e2e_bad"] == 0, "first differing tuple %d" % c["first_bad_e2e"]
    assert c["e2e_flagged"] > 0 and c["e2e_kept"] > c["e2e_n"] // 8 and c["e2e_nan"] > 0
