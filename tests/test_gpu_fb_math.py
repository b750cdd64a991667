"""The framebuffer kernel's launch-constant arithmetic (csrc/fb_math.cuh), checked on the GPU by tests/fb_math_check.cu:
the camera divides split at the divisor equal __fdiv_rn for every frame width and height, and the per-block colour tables
equal the oracle's packing for every hit count of every sample count up to the table's cap."""
import os
import re
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(os.path.dirname(HERE), "bih-gpu-raytracer_b200")


def nvcc():
    return os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")


def table_cap():
    with open(os.path.join(PKG, "csrc", "fb_math.cuh")) as f:
        return int(re.search(r"#define COLOUR_TABLE_MAX (\d+)", f.read()).group(1))


@pytest.fixture(scope="module")
def checked(tmp_path_factory):
    d = tmp_path_factory.mktemp("fb_math")
    exe, tables = str(d / "fb_math_check"), str(d / "tables.bin")
    subprocess.check_call([nvcc(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                           os.path.join(HERE, "fb_math_check.cu")])
    p = subprocess.run([exe, tables], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout, np.fromfile(tables, np.uint32)


@pytest.mark.gpu
def test_camera_divide_equals_fdiv_rn(checked):
    out, _ = checked
    m = re.search(r"^div (\d+) (\d+) (\S+)$", out, re.M)
    assert m, out
    assert int(m.group(1)) == 0, "camera_div != __fdiv_rn: %s mismatches, first at w = %s, x = %s" % m.groups()


@pytest.mark.gpu
def test_colour_table_equals_oracle_packing(checked, oracle):
    _, tab = checked
    cap = table_cap()
    assert tab.size == (cap + 1) * (cap + 2) // 2 - 1
    for n in range(1, cap + 1):
        # pixel h of a 1-row frame with n samples per pixel: its first h samples hit
        hits = np.where(np.arange(n)[None, :] < np.arange(n + 1)[:, None], 0, -1).astype(np.int32)
        want = oracle.pack_framebuffer(hits.ravel(), n + 1, 1, n)
        off = n * (n + 1) // 2 - 1
        np.testing.assert_array_equal(tab[off:off + n + 1], want, err_msg="colour table for %d samples per pixel" % n)
