"""C_gprc_gpr_append of src/gprc_shim.c (the `.Call` behind GPR$add_points) EXECUTED against libgprc on the GPU, through
the miniature R runtime of tests/stubs/mini_r.c; tests/shim_append_exec.c plays the R host code (known answers of
test-gpr.R reached by appending, return shapes, the info > 0 path, the non-conformable error)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "gaussian-process-regression_b200")


def build(tmp_path):
    exe = str(tmp_path / "shim_append_exec")
    cmd = ["gcc", "-std=c11", "-Wall", "-Werror", "-D_GNU_SOURCE", "-I" + os.path.join(ROOT, "tests", "stubs"),
           "-I" + os.path.join(ROOT, "include"), os.path.join(PKG, "src", "gprc_shim.c"),
           os.path.join(ROOT, "tests", "stubs", "mini_r.c"), os.path.join(ROOT, "tests", "shim_append_exec.c"),
           "-L" + PKG, "-lgprc", "-lm", "-o", exe]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return exe


def test_append_shim_driver_compiles_and_links(tmp_path):
    """CPU tier: the shim, the miniature runtime and the append driver build warning-free and link against libgprc.so"""
    build(tmp_path)


@pytest.mark.gpu
def test_append_shim_executes_against_the_library(tmp_path):
    exe = build(tmp_path)
    env = dict(os.environ, LD_LIBRARY_PATH=PKG + os.pathsep + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and "ALL OK" in out.stdout and "FAIL" not in out.stdout, out.stdout + out.stderr
    assert out.stdout.count(" ok\n") >= 10, out.stdout
