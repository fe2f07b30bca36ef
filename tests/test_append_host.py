"""CPU tier of the append (GPR.add_points / gprc_gpr_append): the substitution kernel behind it runs on the FP64 tensor
cores, and add_points rejects malformed arguments on the host before the library is called."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "gaussian-process-regression_b200")


def kernel_sass(name):
    """the SASS of the kernel function(s) of libgprc.so whose symbol contains `name`"""
    out = subprocess.run(["cuobjdump", "-sass", os.path.join(PKG, "libgprc.so")], capture_output=True, text=True).stdout
    body, keep = [], False
    for line in out.splitlines():
        if "Function : " in line:
            keep = name in line
        if keep:
            body.append(line)
    return "\n".join(body)


def test_trsm_flow_kernel_runs_on_the_fp64_tensor_cores():
    sass = kernel_sass("trsm_flow_kernel")
    assert "Function : " in sass, "trsm_flow_kernel is not in libgprc.so"
    assert "DMMA.8x8x4" in sass
    assert "UBLKCP" in sass  # operands staged by the TMA engine


@pytest.fixture
def model(gprc):
    # a model object as the constructor leaves it, without a device: the argument checks come before any library call
    g = gprc.GPR.__new__(gprc.GPR)
    g._X = np.arange(6, dtype=float).reshape(2, 3)
    g._y = np.zeros(3)
    g._k = gprc.cov_func(gprc.sqrexp, l=1.0)
    g._handle = None
    return g


@pytest.mark.parametrize("X_new,y_new,match", [
    (np.zeros(3), np.zeros(1), r"length\(X_new\) %% nrow\(self\$X\) == 0"),           # length not a multiple of D
    (np.array(["a", "b"]), np.zeros(1), r"is.numeric\(X_new\)"),                       # non-numeric
    (np.array([True, False]), np.zeros(1), r"is.numeric\(X_new\)"),                    # logical is not numeric in R
    (np.zeros((3, 2)), np.zeros(2), r"non-conformable arrays"),                         # wrong number of rows
    (np.zeros(4), np.zeros(1), r"length\(y_new\) == ncol\(X_new\)"),                   # 2 points, 1 value
    (np.zeros(4), np.array(["a", "b"]), r"is.numeric\(y_new\)"),                       # non-numeric y
    (np.zeros(2), np.zeros((1, 1)), r"is.vector\(y_new\)"),                            # y not a vector
])
def test_add_points_argument_checks(model, X_new, y_new, match):
    with pytest.raises(ValueError, match=match):
        model.add_points(X_new, y_new)
    assert model._X.shape == (2, 3) and len(model._y) == 3


def test_add_points_with_no_points_is_a_no_op(model):
    assert model.add_points(np.zeros(0), np.zeros(0)) is model
    assert model._X.shape == (2, 3)
