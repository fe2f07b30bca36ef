"""The explicit inverse W = L^-1 (trtri_levels) and the results built on it, against float64 LAPACK / NumPy and the
oracle at the sizes and shapes where the blocked kernels change behaviour:

- W itself for 1 to 129 block rows (the level-wise inversion splits groups in two and clips the right part), with a
  padded leading dimension, and the plain DGEMM with padded operands;
- predict path 1 (the default route) at the full size of BASELINE config 4, and the other paths after the inversion has
  used the factor's upper block triangle as scratch;
- the full predictive covariance, the likelihood gradient and posterior sampling;
- the automatic mixed plan of large predicts (whole waves on path 2, the merged tail on path 3).

Every tolerance is fixed from the input (its conditioning, or the magnitudes the reference sums) before the library
runs.  No library kernel serves as the reference of another."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.linalg
from scipy.linalg import lapack

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
NB = 128
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c4_full_sample.npz")


def assert_mean_var(got, ref, kss):
    """the oracle tolerances of the GPR suite: |d mean| <= 1e-9 max(|mean|, max|mean|); |d var| <= 1e-9 max(|var|, k**)"""
    scale = np.maximum(np.abs(ref[:, 0]), np.max(np.abs(ref[:, 0])))
    assert np.all(np.abs(got[:, 0] - ref[:, 0]) <= 1e-9 * scale)
    assert np.all(np.abs(got[:, 1] - ref[:, 1]) <= 1e-9 * np.maximum(np.abs(ref[:, 1]), kss))


def _offset(p, nbytes):
    return C.c_void_p(p.value + nbytes)


# ---------------------------------------------------------------------------------------------------------------------
# W = L^-1 across block counts
# ---------------------------------------------------------------------------------------------------------------------
def _sqrexp_spd(gprc, ctx, n, seed):
    """K + 0.1 I for a sqrexp kernel on random points: W = L^-1 is dense (the points are in random order, so no block of
    W is negligible).  Returns A and a bound on kappa_2(L): lambda_min >= 0.1 (K is PSD), lambda_max <= the largest row
    sum (Gershgorin, K >= 0)."""
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1, 1, (3, n))
    A = gprc.covariance_matrix(X, X, gprc.cov_func(gprc.sqrexp, l=0.3), ctx=ctx)
    A[np.diag_indices(n)] += 0.1
    kappa_L = np.sqrt(np.max(np.sum(A, axis=1)) / 0.1)
    return A, kappa_L


def _factor_and_invert(ctx, A, n, ld, pad_value=0.0):
    """gprc_dev_potrf + gprc_dev_trtri on an ld x n buffer (rows n..ld-1 hold pad_value); W starts as zeros in its n x n
    part and pad_value below.  Returns the downloaded ld x n buffers of the factor and of W."""
    buf = np.full((ld, n), pad_value, order="F")
    buf[:n] = A
    dA = ctx.upload(buf)
    dinv = ctx.malloc(n * NB * 8)
    wbuf = np.full((ld, n), pad_value, order="F")
    wbuf[:n] = 0.0
    dW = ctx.upload(wbuf)
    try:
        info = C.c_long(-1)
        rc = ctx.lib.gprc_dev_potrf(ctx.handle, dA, n, ld, dinv, C.byref(info))
        assert rc == 0, ctx.lib.gprc_last_error()
        assert info.value == 0
        Lbuf = np.empty((ld, n), order="F")
        ctx.d2h(Lbuf, dA)
        rc = ctx.lib.gprc_dev_trtri(ctx.handle, dA, n, ld, dinv, dW, dA)  # scratch: the upper block triangle of L
        assert rc == 0, ctx.lib.gprc_last_error()
        ctx.d2h(wbuf, dW)
    finally:
        for p in (dA, dinv, dW):
            ctx.free(p)
    return Lbuf, wbuf


def _tile_errors(W, Wref):
    """max |W - Wref| over each 128 x 128 tile"""
    nt = W.shape[0] // NB
    return np.abs(W - Wref).reshape(nt, NB, nt, NB).max(axis=(1, 3))


@pytest.mark.parametrize("nt", [1, 2, 3, 5, 7, 8, 9, 13, 16, 17, 31, 33, 64, 65])
def test_trtri_matches_lapack_tile_by_tile(gprc, ctx, nt):
    n = nt * NB
    A, kappa_L = _sqrexp_spd(gprc, ctx, n, seed=nt)
    # normwise error of a triangular inverse: ~ n eps kappa(L) ||W|| (Higham, ch. 14); both sides carry it
    tol = n * EPS * kappa_L
    Lbuf, W = _factor_and_invert(ctx, A, n, n)
    L = np.tril(Lbuf)
    Wref, info = lapack.dtrtri(L, lower=1)
    assert info == 0
    Wref = np.tril(Wref)
    scale = np.max(np.abs(Wref))
    err = _tile_errors(W, Wref) / scale
    worst = np.unravel_index(np.argmax(err), err.shape)
    assert err.max() <= tol, "tile %s: %.3e > %.3e" % (worst, err.max(), tol)
    assert np.all(np.triu(W, 1) == 0.0)


def _partial_group_columns(nt):
    """first and last column of the left and of the clipped right part of every group whose right part is partial"""
    cols = set()
    s = 1
    while s < nt:
        for gl in range(0, nt, 2 * s):
            gr = gl + s
            r = min(s, nt - gr)
            if 0 < r < s:
                cols.update([gl * NB, gr * NB - 1, gr * NB, (gr + r) * NB - 1])
        s *= 2
    return sorted(cols)


@pytest.mark.parametrize("nt", [100, 129])
def test_trtri_sampled_columns_at_many_block_rows(gprc, ctx, nt):
    n = nt * NB
    A, kappa_L = _sqrexp_spd(gprc, ctx, n, seed=nt)
    tol = n * EPS * kappa_L
    cols = _partial_group_columns(nt)
    rng = np.random.default_rng(nt)
    rest = np.setdiff1d(np.arange(n), cols)
    J = np.sort(np.concatenate([cols, rng.choice(rest, 64 - len(cols), replace=False)]))
    dA = ctx.upload(np.asfortranarray(A))
    del A
    dinv = ctx.malloc(n * NB * 8)
    dW = ctx.upload(np.zeros((n, n), order="F"))
    try:
        info = C.c_long(-1)
        assert ctx.lib.gprc_dev_potrf(ctx.handle, dA, n, n, dinv, C.byref(info)) == 0, ctx.lib.gprc_last_error()
        assert info.value == 0
        L = np.empty((n, n), order="F")
        ctx.d2h(L, dA)
        assert ctx.lib.gprc_dev_trtri(ctx.handle, dA, n, n, dinv, dW, dA) == 0, ctx.lib.gprc_last_error()
        WJ = np.empty((n, len(J)), order="F")
        col = np.empty(n)
        for q, j in enumerate(J):                      # column j of W is contiguous on the device
            ctx.d2h(col, _offset(dW, int(j) * n * 8))
            WJ[:, q] = col
    finally:
        for p in (dA, dinv, dW):
            ctx.free(p)
    L = np.tril(L)
    E = np.zeros((n, len(J)), order="F")
    E[J, np.arange(len(J))] = 1.0
    ref = scipy.linalg.solve_triangular(L, E, lower=True, check_finite=False)
    scale = np.max(np.abs(ref))
    err = np.abs(WJ - ref).reshape(nt, NB, len(J)).max(axis=1) / scale      # (row tile, sampled column)
    worst = np.unravel_index(np.argmax(err), err.shape)
    assert err.max() <= tol, "row tile %d, column %d: %.3e > %.3e" % (worst[0], J[worst[1]], err.max(), tol)


def test_potrf_and_trtri_with_a_padded_leading_dimension(gprc, ctx):
    """ld = n + 256 with NaN in the padding rows: the factor and W are right and no padding entry is written"""
    nt = 9
    n, ld = nt * NB, nt * NB + 256
    A, kappa_L = _sqrexp_spd(gprc, ctx, n, seed=3)
    tol = n * EPS * kappa_L
    Lbuf, Wbuf = _factor_and_invert(ctx, A, n, ld, pad_value=np.nan)
    assert np.all(np.isnan(Lbuf[n:])) and np.all(np.isnan(Wbuf[n:]))
    L = np.tril(Lbuf[:n])
    Lref = scipy.linalg.cholesky(A, lower=True)
    assert np.max(np.abs(L - Lref)) <= tol * np.max(np.abs(Lref))
    Wref = np.tril(lapack.dtrtri(L, lower=1)[0])
    assert np.max(_tile_errors(Wbuf[:n], Wref)) <= tol * np.max(np.abs(Wref))
    assert np.all(np.triu(Wbuf[:n], 1) == 0.0)


@pytest.mark.parametrize("transb", [1, 0])
def test_dgemm_with_padded_operands(ctx, transb):
    M, N, K = 256, 384, 16
    lda, ldb, ldc = M + 128, (N if transb else K) + 64, M + 130
    rng = np.random.default_rng(17 + transb)
    A = np.full((lda, K), np.nan, order="F")
    A[:M] = rng.standard_normal((M, K))
    rows_b, cols_b = (N, K) if transb else (K, N)
    B = np.full((ldb, cols_b), np.nan, order="F")
    B[:rows_b] = rng.standard_normal((rows_b, cols_b))
    Cm = np.full((ldc, N), np.nan, order="F")
    Cm[:M] = rng.standard_normal((M, N))
    dA, dB, dC = ctx.upload(A), ctx.upload(B), ctx.upload(Cm)
    try:
        rc = ctx.lib.gprc_dev_dgemm(ctx.handle, transb, M, N, K, -1.5, dA, lda, dB, ldb, 0.5, dC, ldc)
        assert rc == 0, ctx.lib.gprc_last_error()
        out = np.empty((ldc, N), order="F")
        ctx.d2h(out, dC)
    finally:
        for p in (dA, dB, dC):
            ctx.free(p)
    Bv = B[:rows_b]
    ref = 0.5 * Cm[:M] - 1.5 * (A[:M] @ (Bv.T if transb else Bv))
    bound = 0.5 * np.abs(Cm[:M]) + 1.5 * (np.abs(A[:M]) @ np.abs(Bv.T if transb else Bv))
    assert np.all(np.abs(out[:M] - ref) <= 4 * (K + 2) * EPS * bound)
    assert np.all(np.isnan(out[M:]))


# ---------------------------------------------------------------------------------------------------------------------
# predict path 1 at full size; the other paths after the inversion
# ---------------------------------------------------------------------------------------------------------------------
def test_path_one_and_persistent_substitution_at_c4_size(gprc, ctx):
    """BASELINE config 4 (n = 50 000) against the committed oracle sample: the automatic route of a small predict is
    path 1 (W = L^-1), and path 3 on the same model; tolerances of test_gpu_c4_golden.py"""
    import bench
    z = np.load(GOLDEN)
    n, m, d, M = int(z["n"]), int(z["m"]), int(z["d"]), int(z["M"])
    X, y, Xs = bench.make_inputs(n, m, d)
    np.testing.assert_array_equal(Xs[:, :M], z["Xs_head"])
    model = gprc.GPR(X, y, float(z["noise"]), gprc.cov_func(gprc.sqrexp, l=float(z["l"])), ctx=ctx)
    out = {}
    out[1] = model.predict(Xs[:, :M])
    assert ctx.last_predict_path() == 1
    ctx.set_option(gprc._lib.OPT_PREDICT_PATH, 3)
    try:
        out[3] = model.predict(Xs[:, :M])
        assert ctx.last_predict_path() == 3
    finally:
        ctx.set_option(gprc._lib.OPT_PREDICT_PATH, 0)
    del model
    for path, got in out.items():
        emean = np.max(np.abs(got[:, 0] - z["mean"])) / np.max(np.abs(z["mean"]))
        evar = np.max(np.abs(got[:, 1] - z["var"]) / np.maximum(np.abs(z["var"]), 1.0))
        assert emean <= 1e-9 and evar <= 1e-9, "path %d: mean %.3e, var %.3e" % (path, emean, evar)


def test_substitution_paths_are_unaffected_by_the_inverse_scratch(gprc, ctx):
    """trtri_levels uses the strictly upper blocks of L's buffer as scratch: paths 2, 3 and 4 give the same bits
    before and after a path-1 predict has built W"""
    rng = np.random.default_rng(61)
    n, m, D = 1500, 148 * 64 + 333, 4
    X = rng.uniform(-1, 1, (D, n))
    y = np.sum(np.sin(2 * X), axis=0) + rng.normal(0, 0.1, n)
    Xs = rng.uniform(-1.2, 1.2, (D, m))
    g = gprc.GPR(X, y, 0.05, gprc.cov_func(gprc.rationalquadratic, l=0.7, alpha=1.5), ctx=ctx)

    def run(path):
        ctx.set_option(gprc._lib.OPT_PREDICT_PATH, path)
        try:
            out = g.predict(Xs)
            assert ctx.last_predict_path() == path
        finally:
            ctx.set_option(gprc._lib.OPT_PREDICT_PATH, 0)
        return out

    first = {p: run(p) for p in (2, 3, 4)}
    again = {p: run(p) for p in (2, 3, 4)}
    for p in (2, 3, 4):
        np.testing.assert_array_equal(again[p], first[p], err_msg="path %d is not reproducible without an inverse" % p)
    run(1)
    for p in (2, 3, 4):
        np.testing.assert_array_equal(run(p), first[p], err_msg="path %d changed after the inversion" % p)


# ---------------------------------------------------------------------------------------------------------------------
# full predictive covariance
# ---------------------------------------------------------------------------------------------------------------------
def _check_full_cov(gprc, ctx, oracle, g, okern, X, y, noise, Xs, host_mean=False):
    mean, cov = g.predict(Xs, pointwise_var=False)
    pw = g.predict(Xs)
    omean, ocov = oracle.GPR(X, y, noise, okern).predict(Xs, pointwise_var=False)
    kss = np.abs(np.asarray(okern(Xs, Xs), dtype=float))
    skk = np.sqrt(np.outer(kss, kss))
    mean, omean = mean[:, 0], omean[:, 0]
    assert np.max(np.abs(mean - omean)) <= 1e-9 * np.max(np.abs(omean))
    assert np.all(np.abs(cov - ocov) <= 1e-9 * skk)
    assert np.all(np.abs(np.diag(cov) - pw[:, 1]) <= 1e-12 * kss)
    assert np.all(np.abs(cov - cov.T) <= 1e-12 * skk)
    mean_tol = 1e-14 * np.max(np.abs(pw[:, 0]))
    if host_mean:
        # the closure route forms K_star' alpha on the host: the same dot products as the device, summed in another
        # order, so they agree to n eps |K_star|' |alpha| (the built-in route shares the device's partial sums)
        Ks = oracle.covariance_matrix(X, Xs, okern)
        mean_tol = np.maximum(mean_tol, X.shape[1] * EPS * (np.abs(Ks).T @ np.abs(g.alpha)))
    assert np.all(np.abs(mean - pw[:, 0]) <= mean_tol)


@pytest.mark.parametrize("n,m,D,name,params,gram", [
    (129, 129, 2, "gammaexp", dict(l=1.1, gamma=1.4), 1),
    (700, 1, 3, "sqrexp", dict(l=0.8), 1),
    (1500, 1000, 4, "rationalquadratic", dict(l=0.9, alpha=2.0), 1),
    (3000, 2177, 8, "sqrexp", dict(l=1.0), 2),
    (1, 300, 2, "polynomial", dict(sigma=1.0, p=2.0), 1),
])
def test_full_covariance_matches_the_oracle(gprc, oracle, ctx, n, m, D, name, params, gram):
    rng = np.random.default_rng(n + m)
    X = rng.uniform(-1, 1, (D, n))
    y = np.sum(np.cos(2 * X), axis=0) + rng.normal(0, 0.1, n)
    Xs = rng.uniform(-1.2, 1.2, (D, m))
    Xs[:, 0] = X[:, 0]
    noise = 0.05
    ctx.set_option(gprc._lib.OPT_GRAM_DMMA, gram)
    try:
        g = gprc.GPR(X, y, noise, gprc.cov_func(getattr(gprc, name), **params), ctx=ctx)
        _check_full_cov(gprc, ctx, oracle, g, oracle.cov_func(getattr(oracle, name), **params), X, y, noise, Xs)
    finally:
        ctx.set_option(gprc._lib.OPT_GRAM_DMMA, 1)


def test_full_covariance_of_a_closure_kernel(gprc, oracle, ctx):
    """an opaque kernel takes the host route through gprc_gpr_get(GET_LINV)"""
    kappa = lambda x, y: np.exp(-2.0 * np.sum((x - y) ** 2, axis=0))
    rng = np.random.default_rng(7)
    n, m = 700, 250
    X = rng.uniform(-1, 1, (2, n))
    y = np.sin(3 * X[0]) + X[1] + rng.normal(0, 0.1, n)
    Xs = rng.uniform(-1.2, 1.2, (2, m))
    g = gprc.GPR(X, y, 0.1, kappa, ctx=ctx)
    _check_full_cov(gprc, ctx, oracle, g, kappa, X, y, 0.1, Xs, host_mean=True)


# ---------------------------------------------------------------------------------------------------------------------
# likelihood gradient
# ---------------------------------------------------------------------------------------------------------------------
def _sqdist(X):
    s = np.zeros((X.shape[1], X.shape[1]))
    for row in X:                       # direct differences, as the kernels of the library evaluate them
        s += (row[:, None] - row[None, :]) ** 2
    return s


def _kernel_and_derivs(name, v, X):
    """K and dK/dv_p for the parameter vector v in the kernel's own order, from the kernel definitions
    (sqrexp exp(-r2 / 2l^2); gammaexp exp(-(r/l)^gamma); rationalquadratic (1 + r2 / (2 alpha l^2))^-alpha;
    polynomial (x.y + sigma)^p)"""
    if name == "polynomial":
        sigma, p = v
        b = X.T @ X + sigma
        K = b ** p
        return K, [p * b ** (p - 1), K * np.log(b)]
    s = _sqdist(X)
    if name == "sqrexp":
        (l,) = v
        K = np.exp(-s / (2 * l * l))
        return K, [K * s / l ** 3]
    if name == "gammaexp":
        l, gam = v
        r = np.sqrt(s)
        q = (r / l) ** gam
        K = np.exp(-q)
        with np.errstate(divide="ignore", invalid="ignore"):
            dgam = np.where(r > 0, -K * q * np.log(r / l), 0.0)
        return K, [K * q * gam / l, dgam]
    l, a = v
    base = 1 + s / (2 * a * l * l)
    K = base ** -a
    return K, [K * s / (l ** 3 * base), K * (-np.log(base) + s / (2 * a * l * l * base))]


GRAD_CASES = dict(sqrexp=[0.6], rationalquadratic=[0.7, 1.6], gammaexp=[0.8, 1.5], polynomial=[1.0, 2.5])


@pytest.mark.parametrize("name", list(GRAD_CASES))
def test_kernel_derivatives_of_the_reference_match_central_differences(name):
    rng = np.random.default_rng(5)
    X = rng.uniform(-0.5, 0.5, (3, 40))
    v = np.array(GRAD_CASES[name])
    _, dK = _kernel_and_derivs(name, v, X)
    for p in range(len(v)):
        h = 1e-5 * v[p]
        vp, vm = v.copy(), v.copy()
        vp[p] += h
        vm[p] -= h
        fd = (_kernel_and_derivs(name, vp, X)[0] - _kernel_and_derivs(name, vm, X)[0]) / (2 * h)
        np.testing.assert_allclose(dK[p], fd, rtol=0, atol=1e-8 * max(1.0, np.max(np.abs(dK[p]))))


def _grad_inputs(n, D, seed):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-0.5, 0.5, (D, n))
    y = np.sum(np.sin(3 * X), axis=0) + rng.normal(0, 0.1, n)
    return X, y


@pytest.mark.parametrize("name", list(GRAD_CASES))
@pytest.mark.parametrize("n", [129, 700, 1500, 3000])
def test_textbook_gradient_matches_numpy(gprc, ctx, n, name):
    """0.5 (alpha' dK alpha - tr(Ky^-1 dK)) with Ky = K + noise I (the gradient fit() runs BFGS on)"""
    X, y = _grad_inputs(n, 3, n)
    noise = 0.1
    v = GRAD_CASES[name]
    K, dKs = _kernel_and_derivs(name, v, X)
    Ky = K + noise * np.eye(n)
    Kinv = np.linalg.inv(Ky)
    alpha = scipy.linalg.cho_solve(scipy.linalg.cho_factor(Ky, lower=True), y)
    ref = np.array([0.5 * (alpha @ dK @ alpha - np.sum(Kinv * dK)) for dK in dKs])
    tol = np.array([1e-9 * (np.abs(alpha) @ np.abs(dK) @ np.abs(alpha) + np.sum(np.abs(Kinv * dK))) for dK in dKs])
    got = gprc.Objective(X, y, noise, ctx=ctx).dens_deriv(name, v, formula=gprc._lib.GRAD_TEXTBOOK)
    assert np.all(np.abs(got - ref) <= tol), (got, ref, tol)


def _as_coded_dk(name, v, X):
    """dK of R/fit.R (cov_dict[[name]]$deriv called positionally with v) for the two kernels tested as coded"""
    s = _sqdist(X)
    if name == "sqrexp":
        (l,) = v
        return [s / l ** 3 * np.exp(-s / (l * l * 2))]
    a, l = v                            # rationalquadratic's deriv reads v as (alpha, l)
    t = 2 * l * l * a
    base = s / t + 1
    return [base ** -a * (s - (t + s) * np.log(base)) / (t + s), s * base ** (-a - 1) / l ** 3]


@pytest.mark.parametrize("n,name,v", [(129, "sqrexp", [0.05]), (700, "sqrexp", [0.05]), (1500, "sqrexp", [0.05]),
                                      (129, "rationalquadratic", [0.05, 1.5]), (700, "rationalquadratic", [0.05, 1.5])])
def test_as_coded_gradient_matches_the_oracle(gprc, oracle, ctx, n, name, v):
    """dens_deriv as coded (noise-free K, diag(K^-1)) at a short length scale, where K is well conditioned"""
    X, y = _grad_inputs(n, 3, n + 1)
    K = oracle.covariance_matrix(X, X, lambda a, b: oracle.cov_dict[name]["func"](a, b, *v))
    assert np.linalg.cond(K) < 1e6
    Kinv = np.linalg.inv(K)
    alpha = Kinv @ y
    tol = np.array([1e-9 * (np.abs(alpha) @ np.abs(dK) @ np.abs(alpha) + np.sum(np.abs(Kinv * dK)))
                    for dK in _as_coded_dk(name, v, X)])
    ref = oracle.dens_deriv(X, y, 0.1, name, v)
    got = gprc.Objective(X, y, 0.1, ctx=ctx).dens_deriv(name, v)
    assert np.all(np.abs(got - ref) <= tol), (got, ref, tol)


# ---------------------------------------------------------------------------------------------------------------------
# posterior sampling
# ---------------------------------------------------------------------------------------------------------------------
def _check_samples(gprc, m, ns, seed):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((m, m))
    S = G @ G.T / m + 0.5 * np.eye(m)
    mean = np.linspace(-3.0, 5.0, m) + 0.25
    w = np.linalg.eigvalsh(S)
    kappa = w[-1] / w[0]
    got = gprc.multivariate_normal(ns, mean, S, rng=np.random.default_rng(seed + 1))
    Z = np.random.default_rng(seed + 1).standard_normal((m, ns))
    L = scipy.linalg.cholesky(S, lower=True)
    ref = mean[:, None] + L @ Z
    # the factor differs from LAPACK's by ~ m eps kappa(S) |L| (perturbation bound of the Cholesky factor); the product
    # and the mean add a few ulp of |L||Z| + |mean|
    bound = 4 * m * EPS * kappa * (np.abs(L) @ np.abs(Z)) + 2 * EPS * np.abs(mean)[:, None]
    assert got.shape == (m, ns)
    bad = np.abs(got - ref) > bound
    assert not np.any(bad), "%d of %d entries off, worst column %d" % (bad.sum(), bad.size, np.argmax(bad.any(axis=0)))


@pytest.mark.parametrize("ns", [1, 129])
@pytest.mark.parametrize("m", [1, 127, 129, 1000])
def test_multivariate_normal_matches_mean_plus_cholesky_times_normals(gprc, m, ns):
    _check_samples(gprc, m, ns, seed=m * 1000 + ns)


def test_multivariate_normal_with_more_draws_than_a_grid_row_holds(gprc, oracle):
    """70 000 draws are more than the 65 535 blocks of gridDim.y; afterwards the library keeps working"""
    _check_samples(gprc, 3, 70000, seed=70000)
    rng = np.random.default_rng(8)
    X = rng.uniform(-1, 1, (2, 200))
    y = np.sin(2 * X[0]) + rng.normal(0, 0.1, 200)
    Xs = rng.uniform(-1, 1, (2, 50))
    got = gprc.GPR(X, y, 0.1, gprc.cov_func(gprc.sqrexp, l=0.7)).predict(Xs)
    assert_mean_var(got, oracle.GPR(X, y, 0.1, oracle.cov_func(oracle.sqrexp, l=0.7)).predict(Xs), np.ones(50))


# ---------------------------------------------------------------------------------------------------------------------
# the automatic mixed plan
# ---------------------------------------------------------------------------------------------------------------------
def test_automatic_mixed_plan_matches_the_oracle(gprc, oracle, ctx):
    """300 tiles of 128 test points, no inverse, n < 4096: one whole wave (148 tiles) on path 2, then the last wave
    merged with the remainder (152 tiles) in one chunk of path 3"""
    rng = np.random.default_rng(71)
    n, m, D = 1000, 2 * 148 * NB + 3 * NB + 5, 3
    X = rng.uniform(-1, 1, (D, n))
    y = np.sum(np.sin(2 * X), axis=0) + rng.normal(0, 0.1, n)
    Xs = rng.uniform(-1.2, 1.2, (D, m))
    g = gprc.GPR(X, y, 0.05, gprc.cov_func(gprc.sqrexp, l=0.8), ctx=ctx)
    got = g.predict(Xs)
    assert ctx.last_predict_path() == 2
    assert ctx.last_predict_chunks() == 2
    ref = oracle.GPR(X, y, 0.05, oracle.cov_func(oracle.sqrexp, l=0.8)).predict(Xs)
    assert_mean_var(got, ref, np.ones(m))
