"""GPR.add_points / gprc_gpr_append: appending training points to a fitted model extends its Cholesky factor in place
(rows from the last full 128-block boundary are recomputed; the new rows are solved against the old factor by
trsm_flow_kernel).  Afterwards the model must be GPR(cbind(X, X_new), c(y, y_new), noise, k): checked against the reference's
known answers, the oracle on the concatenated data, and fresh GPU fits."""
import ctypes as C
import math
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def data(rng, D, n, noise_sd=0.1):
    X = rng.uniform(-2, 2, (D, n))
    y = np.sum(np.sin(X), axis=0) + rng.normal(0, noise_sd, n)
    return X, y


def assert_matches(g, ref, Xs, check_L):
    """logp 1e-8 relative, alpha 1e-9 max|alpha|, L 1e-12 max|L|, predictive mean / variance 1e-9 (the repo's tolerances)"""
    assert g.logp.shape == (1, 1)
    assert abs(g.logp[0, 0] - float(ref.logp)) <= 1e-8 * abs(float(ref.logp))
    assert np.max(np.abs(g.alpha - ref.alpha)) <= 1e-9 * np.max(np.abs(ref.alpha))
    if check_L:
        assert np.max(np.abs(g.L - ref.L)) <= 1e-12 * np.max(np.abs(ref.L))
    got, want = g.predict(Xs), ref.predict(Xs)
    assert np.max(np.abs(got[:, 0] - want[:, 0])) <= 1e-9 * max(np.max(np.abs(want[:, 0])), 1.0)
    assert np.max(np.abs(got[:, 1] - want[:, 1])) <= 1e-9


def test_known_answers_through_append(gprc):
    # tests/testthat/test-gpr.R:12-15, one point fitted and the second appended
    g = gprc.GPR.constant(np.array([[1.0]]), np.array([1.0]), 1, c=1)
    assert g.add_points(np.array([2.0]), np.array([3.0])) is g
    np.testing.assert_allclose(g.predict(3.0), [[4 / 3, 1 / 3]], rtol=0, atol=1.5e-8)
    # :23-27
    g = gprc.GPR.sqrexp(np.array([[1.0]]), np.array([0.0]), 1, l=1).add_points([2.0], [1.0])
    e = math.exp
    var = 1 - (2 * e(-1) - 2 * e(-3) + 2 * e(-4)) / (4 - e(-1))
    np.testing.assert_allclose(g.predict(0.0), [[(2 * e(-2) - e(-1)) / (4 - e(-1)), var]], rtol=0, atol=1.5e-8)
    assert isinstance(g, gprc.GPR.sqrexp)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 1000, 5000])
@pytest.mark.parametrize("k", [1, 2, 127, 128, 300])
def test_against_the_oracle_on_the_concatenated_data(gprc, oracle, n, k):
    """128 boundaries on both sides, growth of the padding and none, and n0 = 0 (n < 128)"""
    rng = np.random.default_rng(1000 * n + k)
    X, y = data(rng, 3, n + k)
    Xs = rng.uniform(-2, 2, (3, 50))
    g = gprc.GPR(X[:, :n], y[:n], 0.05, gprc.cov_func(gprc.sqrexp, l=0.8))
    g.add_points(X[:, n:], y[n:])
    ref = oracle.GPR(X, y, 0.05, oracle.cov_func(oracle.sqrexp, l=0.8))
    assert_matches(g, ref, Xs, check_L=n + k <= 1500)
    assert g.X.shape == (3, n + k) and np.array_equal(g.X, X) and np.array_equal(g.y, y) and g.noise == 0.05
    assert g._ctx.lib.gprc_gpr_n(g._handle) == n + k


@pytest.mark.parametrize("name,par,D", [
    ("rationalquadratic", dict(l=1.0, alpha=1.5), 4),
    ("polynomial", dict(sigma=1.0, p=2.0), 3),
    ("linear", dict(sigma=np.array([0.5, 1.0, 2.0])), 3),
    ("gammaexp", dict(l=1.0, gamma=1.5), 2),
])
@pytest.mark.parametrize("n,k", [(127, 2), (300, 200), (1000, 129)])
def test_other_kernels_against_the_oracle(gprc, oracle, name, par, D, n, k):
    rng = np.random.default_rng(n + 7 * k + D)
    X, y = data(rng, D, n + k)
    Xs = rng.uniform(-2, 2, (D, 40))
    noise = 0.5 if name in ("polynomial", "linear") else 0.05
    g = gprc.GPR(X[:, :n], y[:n], noise, gprc.cov_func(getattr(gprc, name), **par))
    g.add_points(X[:, n:], y[n:])
    ref = oracle.GPR(X, y, noise, oracle.cov_func(getattr(oracle, name), **par))
    assert_matches(g, ref, Xs, check_L=True)


def test_many_single_point_appends(gprc):
    """300 appends of one point from n = 500: crosses the 128 boundaries at 512, 640, 768; agrees with one fresh fit"""
    rng = np.random.default_rng(5)
    X, y = data(rng, 8, 800)
    k = gprc.cov_func(gprc.sqrexp, l=1.0)
    g = gprc.GPR(X[:, :500], y[:500], 0.01, k)
    for i in range(500, 800):
        g.add_points(X[:, i], y[i:i + 1])
    fresh = gprc.GPR(X, y, 0.01, k)
    assert abs(g.logp[0, 0] - fresh.logp[0, 0]) <= 1e-11 * abs(fresh.logp[0, 0])
    assert np.max(np.abs(g.alpha - fresh.alpha)) <= 1e-9 * np.max(np.abs(fresh.alpha))
    Xs = rng.uniform(-2, 2, (8, 100))
    assert np.max(np.abs(g.predict(Xs) - fresh.predict(Xs))) <= 1e-9


@pytest.mark.parametrize("k", [1, 128, 1000, 20000])
def test_large_n(gprc, k):
    """n = 20 480 (160 row blocks): one group of right-hand sides, several groups, and more than one wave of units"""
    rng = np.random.default_rng(20480 + k)
    n, D = 20480, 6
    X = rng.uniform(-1, 1, (D, n + k))
    y = np.sum(np.sin(3 * X), axis=0) + rng.normal(0, 0.1, n + k)
    kern = gprc.cov_func(gprc.sqrexp, l=1.0)
    g = gprc.GPR(X[:, :n], y[:n], 0.01, kern)
    g.add_points(X[:, n:], y[n:])
    a = g.alpha.copy()
    idx = np.concatenate([rng.integers(0, n, 32), rng.integers(n, n + k, 32)])
    Krows = np.exp(-0.5 * np.sum((X[:, idx, None] - X[:, None, :]) ** 2, axis=0))
    Krows[np.arange(len(idx)), idx] += 0.01
    assert np.max(np.abs(Krows @ a - y[idx])) < 1e-8 * np.max(np.abs(a))
    lp = g.logp[0, 0]
    del g
    fresh = gprc.GPR(X, y, 0.01, kern)
    assert abs(lp - fresh.logp[0, 0]) <= 1e-11 * abs(fresh.logp[0, 0])
    assert np.max(np.abs(a - fresh.alpha)) <= 1e-9 * np.max(np.abs(fresh.alpha))


def test_derived_state_is_rebuilt_after_an_append(gprc, ctx):
    """W = L^-1 (path 1) and the INT8 digit planes (path 4) exist before the append; every path agrees with a fresh model
    afterwards"""
    rng = np.random.default_rng(9)
    X, y = data(rng, 4, 700)
    Xs = rng.uniform(-2, 2, (4, 300))
    kern = gprc.cov_func(gprc.sqrexp, l=1.0)
    g = gprc.GPR(X[:, :600], y[:600], 0.01, kern)
    opt = gprc._lib.OPT_PREDICT_PATH
    try:
        for path in (1, 4):
            ctx.set_option(opt, path)
            g.predict(Xs)
            assert ctx.last_predict_path() == path
        g.add_points(X[:, 600:], y[600:])
        fresh = gprc.GPR(X, y, 0.01, kern)
        for path in (1, 2, 3, 4):
            ctx.set_option(opt, path)
            got = g.predict(Xs)
            assert ctx.last_predict_path() == path
            want = fresh.predict(Xs)
            assert np.max(np.abs(got[:, 0] - want[:, 0])) <= 1e-9 * np.max(np.abs(want[:, 0])), path
            assert np.max(np.abs(got[:, 1] - want[:, 1])) <= 1e-9, path
    finally:
        ctx.set_option(opt, 0)


def test_failed_append_leaves_the_model_intact(gprc, oracle):
    """constant kernel c = 1, noise 0: the Schur complement of the second point is 1 - 1 * 1^-1 * 1 = 0 exactly"""
    g = gprc.GPR.constant(np.array([[1.0]]), np.array([2.0]), 0, c=1)
    Xs = np.array([[0.0, 3.0, 7.0]])
    lp0, a0, p0 = g.logp.copy(), g.alpha.copy(), g.predict(Xs)
    lib = g._ctx.lib
    xp, yp = np.array([5.0]), np.array([-1.0])
    logp, info = C.c_double(0.0), C.c_long(0)
    rc = lib.gprc_gpr_append(g._handle, xp.ctypes.data_as(C.POINTER(C.c_double)), 1,
                             yp.ctypes.data_as(C.POINTER(C.c_double)), C.byref(logp), C.byref(info))
    assert rc == 0 and info.value == 2
    assert lib.gprc_gpr_n(g._handle) == 1
    g._alpha = None
    assert np.array_equal(g.logp, lp0) and np.array_equal(g.alpha, a0) and np.array_equal(g.predict(Xs), p0)
    # add_points then does what the constructor does on the same data: noise bumped to 0.01, with its warning
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        g.add_points([5.0], [-1.0])
        ref = gprc.GPR.constant(np.array([[1.0, 5.0]]), np.array([2.0, -1.0]), 0, c=1)
    msgs = [str(x.message) for x in w]
    assert msgs == ["Noise got changed to 0.01 to avoid errors in cholesky decomposition"] * 2
    assert g.noise == ref.noise == 0.01
    assert np.array_equal(g.logp, ref.logp) and np.array_equal(g.predict(Xs), ref.predict(Xs))
    assert g.X.shape == (1, 2) and np.array_equal(g.y, [2.0, -1.0])


def test_closure_kernel_takes_the_constructor_path(gprc):
    kappa = lambda x, y: np.exp(-3 * np.sum((x - y) ** 2, axis=0))
    rng = np.random.default_rng(3)
    X, y = data(rng, 2, 90)
    g = gprc.GPR(X[:, :60], y[:60], 0.1, kappa)
    lp = C.c_double(0.0)
    info = C.c_long(0)
    xp, yp = gprc._lib.points(X[:, 60:]), np.ascontiguousarray(y[60:])
    rc = g._ctx.lib.gprc_gpr_append(g._handle, gprc._lib.dptr(xp), 30, gprc._lib.dptr(yp), C.byref(lp), C.byref(info))
    assert rc < 0
    g.add_points(X[:, 60:], y[60:])
    ref = gprc.GPR(X, y, 0.1, kappa)
    Xs = rng.uniform(-2, 2, (2, 20))
    assert np.array_equal(g.logp, ref.logp) and np.array_equal(g.predict(Xs), ref.predict(Xs))
    assert g.k is kappa


def test_appends_are_reproducible(gprc):
    rng = np.random.default_rng(11)
    X, y = data(rng, 5, 3000)
    kern = gprc.cov_func(gprc.sqrexp, l=1.0)
    out = []
    for _ in range(2):
        g = gprc.GPR(X[:, :2000], y[:2000], 0.01, kern)
        g.add_points(X[:, 2000:2100], y[2000:2100]).add_points(X[:, 2100:], y[2100:])
        out.append((g.alpha.copy(), g.logp[0, 0]))
        del g
    assert np.array_equal(out[0][0], out[1][0]) and out[0][1] == out[1][1]
