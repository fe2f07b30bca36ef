"""The blocked Cholesky above n = 16 384 (potrf_blocked: the launch sequence with two-stream lookahead, outer panels of
512 columns up to 199 block columns and of 1024 from 200 on), its first-bad-pivot report, the smallest leading-minor
determinant fit() reads, and the GPC Newton loop on the blocked route -- against float64 references computed with
torch (cuSOLVER / cuBLAS, code independent of libgprc) on the same device, and against the oracle.

Every tolerance has the form c kappa u scale, with u the unit roundoff, kappa an estimate of the condition number of
the matrix that was factored (lambda_max from power iterations, lambda_min bounded below by the added diagonal) and c
written next to it.  c = 8 sqrt(n) covers the sqrt(n) growth of the rounding errors of blocked sums; every such
tolerance stays below 1e-7 relative, so an error of 1e-6 relative in any tile fails it."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.linalg
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
NB = 128
DEV = "cuda"
F64 = torch.float64


@pytest.fixture(autouse=True)
def _release_torch_cache():
    yield
    if torch.cuda.is_initialized():
        torch.cuda.empty_cache()  # the factorisations below hold 10-50 GB; hand it back before the library allocates


def c_of(n):
    return 8.0 * math.sqrt(n)


def report(what, err, tol, scale):
    """print the observed error against its tolerance; the tolerance must stay below 1e-7 of the scale it is stated in"""
    assert tol < 1e-7 * scale, "%s: tolerance %.3e is too loose to catch a 1e-6 error" % (what, tol)
    print("%s: error %.3e, tolerance %.3e, ratio %.3e" % (what, err, tol, err / tol))


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def sqrexp(A, B, l=1.0):
    """exp(-|a - b|^2 / (2 l^2)) for the columns of A (d x n) and B (d x m), from explicit differences"""
    s = torch.zeros(A.shape[1], B.shape[1], dtype=F64, device=A.device)
    for a, b in zip(A, B):
        s.add_((a[:, None] - b[None, :]) ** 2)
    return torch.exp(s.mul_(-0.5 / (l * l)))


def lam_max(A, iters=30):
    """largest eigenvalue of the symmetric A with non-negative entries (power iterations from the Perron direction)"""
    v = torch.ones(A.shape[0], dtype=F64, device=A.device)
    for _ in range(iters):
        v = A @ v
        v /= torch.linalg.vector_norm(v)
    return float(v @ (A @ v))


def spd_matrix(n, seed):
    """A = K_sqrexp(X, X; l = 1) + I, X ~ U(-1, 1)^8, and kappa(A) <= lambda_max / 1"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    X = torch.rand(8, n, generator=g, dtype=F64, device=DEV) * 2 - 1
    A = sqrexp(X, X)
    A.diagonal().add_(1.0)
    return A, lam_max(A)


def ref_cholesky(A):
    L, info = torch.linalg.cholesky_ex(A)
    assert int(info) == 0
    return L


def potrf(ctx, buf, n, ld, dinv):
    """gprc_dev_potrf on the column-major ld x n matrix held by buf (n x ld, row-major: buf[c, r] = A[r, c])"""
    torch.cuda.synchronize()  # the library works on its own non-blocking streams
    info = C.c_long(-1)
    rc = ctx.lib.gprc_dev_potrf(ctx.handle, C.c_void_p(buf.data_ptr()), n, ld, C.c_void_p(dinv.data_ptr()),
                                C.byref(info))
    assert rc == 0, ctx.lib.gprc_last_error()
    return info.value


def factor(ctx, A, ld):
    """copy A into an ld x n buffer whose padding rows hold NaN, factor it; returns (buf, dinv, info, launches)"""
    n = A.shape[0]
    buf = torch.full((n, ld), float("nan"), dtype=F64, device=DEV)
    buf[:, :n] = A  # A is symmetric: its rows are its columns
    dinv = torch.zeros(n // NB, NB, NB, dtype=F64, device=DEV)
    ctx.reset_timers()
    info = potrf(ctx, buf, n, ld, dinv)
    return buf, dinv, info, ctx.timers()[1]


def worst_tile(Lt, Lref):
    """Lt: the factor transposed (row c holds column c of L, as the column-major buffer reads row by row).
    max |L - Lref| over the lower triangle -> (worst error, its 128 x 128 tile (i, j))"""
    n = Lref.shape[0]
    E = torch.triu(Lt)
    E.sub_(Lref.T).abs_()
    if n % NB:
        idx = int(torch.argmax(E))
        return float(E.reshape(-1)[idx]), (idx % n // NB, idx // n // NB)
    nt = n // NB
    T = E.reshape(nt, NB, nt, NB).amax(dim=(1, 3))  # T[tile of c, tile of r]
    idx = int(torch.argmax(T))
    tj, ti = divmod(idx, nt)
    return float(T.reshape(-1)[idx]), (ti, tj)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the raw factor on both routes and at the edges of the outer panels
# ---------------------------------------------------------------------------------------------------------------------
# (n, padded ld): nt = 128 is the last persistent size; 129 the first blocked one (its last outer panel has one block
# column); 157 = 4 * 39 + 1; 199 the last with 512-column panels; 200 the first with 1024-column panels (200 % 8 = 0:
# the last panel has no rest() update); 258 ends in a partial panel; 320 % 8 = 0
FACTOR_CASES = [(16384, False), (16512, False), (20096, True), (25472, False), (25600, False), (33024, True),
                (40960, False)]


@pytest.mark.parametrize("n,padded", FACTOR_CASES)
def test_factor_and_inverted_diagonal_blocks_match_cusolver(ctx, n, padded):
    nt = n // NB
    ld = n + NB if padded else n
    A, lmax = spd_matrix(n, seed=nt)
    kappa = lmax / 1.0
    Lref = ref_cholesky(A)
    buf, dinv, info, launches = factor(ctx, A, ld)
    del A
    assert info == 0
    # the route under test: one persistent launch up to 128 block columns, about three launches per block column beyond
    assert (launches == 1) if nt <= 128 else (launches > 2 * nt)
    if padded:
        assert bool(torch.isnan(buf[:, n:]).all()), "a padding row was written"
    c = c_of(n)
    tol = c * kappa * U * float(Lref.abs().max())
    err, (ti, tj) = worst_tile(buf[:, :n], Lref)
    report("n=%d L" % n, err, tol, float(Lref.abs().max()))
    assert err <= tol, "n = %d: tile (%d, %d) off by %.3e > %.3e" % (n, ti, tj, err, tol)
    del buf
    # the inverted diagonal blocks (column-major 128 x 128 each; zeros above the diagonal)
    ar = torch.arange(nt, device=DEV)
    Ld = Lref.view(nt, NB, nt, NB)[ar, :, ar, :]
    del Lref
    eye = torch.eye(NB, dtype=F64, device=DEV).repeat(nt, 1, 1)
    Wref = torch.linalg.solve_triangular(Ld, eye, upper=False)
    Wgot = dinv.transpose(1, 2)
    assert bool((torch.triu(Wgot, 1) == 0).all())
    E = (Wgot - Wref).abs().amax(dim=(1, 2))
    tol = c * kappa * U * float(Wref.abs().max())
    j = int(torch.argmax(E))
    report("n=%d dinv" % n, float(E[j]), tol, float(Wref.abs().max()))
    assert float(E[j]) <= tol, "n = %d: inverted diagonal block %d off by %.3e > %.3e" % (n, j, float(E[j]), tol)


def test_the_torch_reference_agrees_with_host_lapack(ctx):
    """pins the cuSOLVER reference once, at the first blocked size, against scipy's dpotrf"""
    n = 16512
    A, lmax = spd_matrix(n, seed=n // NB)
    Lt = ref_cholesky(A).cpu().numpy()
    Lh = scipy.linalg.cholesky(A.cpu().numpy(), lower=True, check_finite=False)
    del A
    tol = c_of(n) * lmax * U * np.max(np.abs(Lh))
    err = np.max(np.abs(Lt - Lh))
    report("torch vs LAPACK", err, tol, np.max(np.abs(Lh)))
    assert err <= tol


# ---------------------------------------------------------------------------------------------------------------------
# 2. the first failing pivot on the blocked route
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def spd_cache():
    cache = {}

    def get(n):
        if n not in cache:
            cache.clear()  # one at a time: 3 GB at n = 20 096, 8.7 GB at 33 024
            cache[n] = spd_matrix(n, seed=n // NB)[0]
        return cache[n]

    yield get
    cache.clear()


def first_bad_pivot(ctx, A, rows):
    """set A[r, r] = -5 for each r in rows and factor; returns (info, the first leading minor that is not positive
    definite).  The reference: the leading minor r0 = min(rows) is positive definite (cuSOLVER factors it) and the
    next pivot, A[r0, r0] - |L^-1 A[:r0, r0]|^2, is negative.  (cholesky_ex's own info is no reference here: on a B200
    with torch 2.11 it reports r + 2 for r = 127, 511, 1023 and 0 for r = n - 1.)"""
    B = A.clone()
    for r in rows:
        B[r, r] = -5.0
    r0 = min(rows)
    pivot = float(B[r0, r0])
    if r0 > 0:
        z = torch.linalg.solve_triangular(ref_cholesky(B[:r0, :r0]), B[:r0, r0:r0 + 1], upper=False)
        pivot -= float(torch.sum(z * z))
    assert pivot < 0
    n = A.shape[0]
    info = potrf(ctx, B, n, n, torch.zeros(n // NB, NB, NB, dtype=F64, device=DEV))
    return info, r0 + 1


# rows of n = 20 096 (4-column panels, nt = 157): first row; last row of block 0; last row of outer panel 0; first row
# of panel 1 (factored on the lookahead stream after LA(0)); inside the last, one-column panel; the last row.
# n = 33 024 (8-column panels, nt = 258): last row of panel 0, first of panel 1, a row beyond 30 000
@pytest.mark.parametrize("n,r", [(20096, 0), (20096, 127), (20096, 511), (20096, 512), (20096, 20000), (20096, 20095),
                                 (33024, 1023), (33024, 1024), (33024, 31001)])
def test_first_bad_pivot_is_reported_by_the_launch_sequence(ctx, spd_cache, n, r):
    info, want = first_bad_pivot(ctx, spd_cache(n), [r])
    assert info == want


def test_the_smallest_bad_pivot_wins_and_no_state_is_carried_over(ctx, spd_cache):
    n = 20096
    A = spd_cache(n)
    first, dinv1, info1, _ = factor(ctx, A, n)
    assert info1 == 0
    info, want = first_bad_pivot(ctx, A, [5000, 3000])
    assert info == want == 3001
    again, dinv2, info2, _ = factor(ctx, A, n)
    assert info2 == 0
    assert torch.equal(torch.triu(first), torch.triu(again)), "the factor changed after a failed call"
    assert torch.equal(dinv1, dinv2)


# ---------------------------------------------------------------------------------------------------------------------
# 3. through the model path: n not a multiple of 128 (identity padding of the covariance build)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,with_L", [(16385, True), (20000, True), (33000, False)])
def test_gpr_fit_matches_torch_on_the_blocked_route(gprc, oracle, ctx, n, with_L):
    noise = 0.01
    cfg = oracle.make_config("C4", n=n, m=1)
    X, y = cfg["X"], cfg["y"]
    model = gprc.GPR(X, y, noise, gprc.cov_func(gprc.sqrexp, l=1.0), ctx=ctx)
    assert model.noise == noise
    Xt, yt = torch.from_numpy(X).to(DEV), torch.from_numpy(y).to(DEV)
    K = sqrexp(Xt, Xt)
    K.diagonal().add_(noise)
    kappa = lam_max(K) / noise
    Lref = ref_cholesky(K)
    del K
    c = c_of(n)
    alpha = torch.cholesky_solve(yt[:, None], Lref)[:, 0]
    logdet = torch.log(torch.diagonal(Lref))
    logp = float(-0.5 * (yt @ alpha) - logdet.sum() - n / 2 * math.log(2 * math.pi))
    err = float((torch.from_numpy(model.alpha).to(DEV) - alpha).abs().max())
    tol = c * kappa * U * float(alpha.abs().max())
    report("n=%d alpha" % n, err, tol, float(alpha.abs().max()))
    assert err <= tol
    scale = float(0.5 * (yt.abs() @ alpha.abs()) + logdet.abs().sum()) + n / 2 * math.log(2 * math.pi)
    tol = c * kappa * U * scale
    report("n=%d logp" % n, abs(model.logp[0, 0] - logp), tol, scale)
    assert abs(model.logp[0, 0] - logp) <= tol
    if with_L:
        Lt = torch.from_numpy(model.L.T).to(DEV)  # model.L is column-major: its transpose is C-contiguous
        assert bool((torch.tril(Lt, -1) == 0).all())  # explicit zeros above the diagonal, like t(chol(.))
        tol = c * kappa * U * float(Lref.abs().max())
        err, (ti, tj) = worst_tile(Lt, Lref)
        report("n=%d model L" % n, err, tol, float(Lref.abs().max()))
        assert err <= tol, "n = %d: tile (%d, %d) off by %.3e > %.3e" % (n, ti, tj, err, tol)


# ---------------------------------------------------------------------------------------------------------------------
# 4. the leading-minor rule of fit()
# ---------------------------------------------------------------------------------------------------------------------
def logml(ctx, X, y, noise, name, v):
    """gprc_logml: (logp, min_leading_logdet, info)"""
    from gprc_b200 import _lib
    from gprc_b200.fit import _spec
    kc, keep = _spec(name, v).to_c()
    xp = _lib.points(X)
    logp, minlog, info = C.c_double(0.0), C.c_double(0.0), C.c_long(0)
    _lib.check(ctx.lib.gprc_logml(ctx.handle, kc, _lib.dptr(xp), X.shape[0], X.shape[1], _lib.dptr(y), noise,
                                  C.byref(logp), C.byref(minlog), C.byref(info)))
    return logp.value, minlog.value, info.value


@pytest.mark.parametrize("n", [1023, 1024, 1025, 3000, 20000])
def test_min_leading_logdet_is_the_prefix_minimum(ctx, n):
    """p points in a tiny cluster (pivots of K + I/2 just above 1/2: the prefix sums fall), then points far from every
    other point (pivots 3/2: they rise), so the minimum lies at p - 1, inside a chunk of gp_reduce_kernel that is neither
    the first nor the last"""
    noise = 0.5
    p = n // 2 + 37
    rng = np.random.default_rng(n)
    X = np.empty((8, n))
    X[:, :p] = 1e-3 * rng.uniform(-1, 1, (8, p))
    X[:, p:] = rng.uniform(-1000, 1000, (8, n - p))
    y = rng.normal(size=n)
    logp, minlog, info = logml(ctx, X, y, noise, "sqrexp", [1.0])
    assert info == 0
    Xt = torch.from_numpy(X).to(DEV)
    K = sqrexp(Xt, Xt)
    K.diagonal().add_(noise)
    kappa = lam_max(K) / noise
    Lref = ref_cholesky(K)
    del K
    prefix = torch.cumsum(2 * torch.log(torch.diagonal(Lref)), 0)
    arg = int(torch.argmin(prefix))
    chunk = (n + 1023) // 1024
    assert arg == p - 1 and chunk <= arg < (n - 1) // chunk * chunk  # interior, and below the full determinant
    assert float(prefix[-1] - prefix[arg]) > 1.0
    tol = c_of(n) * kappa * U * float(prefix.abs().max())
    report("n=%d min leading logdet" % n, abs(minlog - float(prefix[arg])), tol, float(prefix.abs().max()))
    assert abs(minlog - float(prefix[arg])) <= tol


def _min_leading_logdet_host(X, noise, l):
    K = np.exp(-0.5 * sum((row[:, None] - row[None, :]) ** 2 for row in X) / (l * l))
    K[np.diag_indices_from(K)] += noise
    return np.min(np.cumsum(2 * np.log(np.diag(scipy.linalg.cholesky(K, lower=True)))))


def _noise_for(X, l, target):
    """the noise at which the smallest leading-minor log determinant of K + noise I is `target` (it rises with noise)"""
    lo, hi = 1e-6, 1.0
    for _ in range(60):
        mid = math.sqrt(lo * hi)
        lo, hi = (mid, hi) if _min_leading_logdet_host(X, mid, l) < target else (lo, mid)
    return hi


# exp(-744.8) rounds to the smallest subnormal, so R's det() of that minor is > 0 and the literal rule accepts;
# exp(-745.5) rounds to 0 and it rejects
@pytest.mark.parametrize("n,where", [(150, "accept"), (200, -744.8), (200, -745.5), (200, "reject"), (300, -744.6)])
def test_literal_minor_rule_matches_the_oracle(gprc, oracle, ctx, n, where):
    cfg = oracle.make_config("C1", n=n, m=1)
    X, y, l = cfg["X"], cfg["y"], 1.0
    noise = {"accept": 0.2, "reject": 0.01}.get(where)
    if noise is None:
        noise = _noise_for(X, l, where)
        assert abs(_min_leading_logdet_host(X, noise, l) - where) < 0.05
    try:
        want = oracle.dens(X, y, noise, "sqrexp", [l], minors="literal")
    except oracle.OptimError:
        want = None
    from gprc_b200.fit import OptimError
    obj = gprc.Objective(X, y, noise, ctx=ctx, minors="literal")
    if want is None:
        with pytest.raises(OptimError):
            obj.dens("sqrexp", [l])
    else:
        assert abs(obj.dens("sqrexp", [l]) - want) <= 1e-8 * abs(want)
    if where == "reject":
        assert want is None
    if where == "accept":
        assert want is not None


# ---------------------------------------------------------------------------------------------------------------------
# 5. the GPC Newton loop on the blocked route
# ---------------------------------------------------------------------------------------------------------------------
def torch_gpc(X, y, l, eps=1e-5):
    """R/GPCclass.R:73-103 in float64 torch (guard off): returns iterations, objective trace, f_hat, the final factor of
    B = I + W^1/2 K W^1/2, logq and K"""
    Xt, yt = torch.from_numpy(X).to(DEV), torch.from_numpy(y).to(DEV)
    K = sqrexp(Xt, Xt, l)
    f = torch.zeros(len(y), dtype=F64, device=DEV)
    trace = []

    def chol_b(f):
        P = 1 / (1 + torch.exp(-f))
        W = (1 - P) * P
        sw = torch.sqrt(W)
        B = torch.outer(sw, sw) * K
        B.diagonal().add_(1.0)
        return P, W, sw, ref_cholesky(B)

    while True:
        P, W, sw, L = chol_b(f)
        b = W * f + (yt + 1) / 2 - P
        inter = torch.linalg.solve_triangular(L, (sw * (K @ b))[:, None], upper=False)
        inter = torch.linalg.solve_triangular(L.T, inter, upper=True)[:, 0]
        a = b - sw * inter
        f = K @ a
        trace.append(float(-torch.sum(a * f) / 2 - torch.sum(torch.log(1 + torch.exp(-yt * f)))))
        if len(trace) > 1 and abs(trace[-1] - trace[-2]) < eps:
            break
    P, W, sw, L = chol_b(f)
    return dict(iterations=len(trace), trace=np.array(trace), f_hat=f, P=P, sw=sw, L=L,
                logq=trace[-1] - float(torch.diagonal(L).sum()), K=K, X=Xt, y=yt)


def assert_gpc_fit(g, r):
    assert g.iterations == r["iterations"]
    np.testing.assert_allclose(g.objective_trace, r["trace"], rtol=1e-9)
    f = r["f_hat"].cpu().numpy()
    assert np.max(np.abs(g.f_hat - f)) <= 1e-9 * np.max(np.abs(f))
    assert abs(g.logq - r["logq"]) <= 1e-8 * abs(r["logq"])


def test_gpc_restatement_matches_the_oracle(oracle):
    c2 = oracle.make_config("C2", n=700, m=1)
    o = oracle.GPC(c2["X"], c2["y"], oracle.cov_func(oracle.sqrexp, l=0.3), guard=False)
    r = torch_gpc(c2["X"], c2["y"], 0.3)
    assert r["iterations"] == o.iterations
    np.testing.assert_allclose(r["trace"], o.objective_trace, rtol=1e-9)
    assert np.max(np.abs(r["f_hat"].cpu().numpy() - o.f_hat)) <= 1e-9 * np.max(np.abs(o.f_hat))
    assert abs(r["logq"] - o.logq) <= 1e-8 * abs(o.logq)
    assert np.max(np.abs(r["L"].cpu().numpy() - o.L)) <= 1e-10 * np.max(np.abs(o.L))


def test_gpc_fit_and_latent_predict_on_the_blocked_route(gprc, oracle, ctx):
    """n = 16 500 (n_pad = 16 512, 129 block columns); 20 000 test points take the INT8 variance pass (path 4, rows
    scaled by sqrt(W)) under the automatic plan"""
    l = 0.3
    c2 = oracle.make_config("C2", n=16500, m=1)
    X, y = c2["X"], c2["y"]
    g = gprc.GPC(X, y, gprc.cov_func(gprc.sqrexp, l=l), guard=False, verbose=False, ctx=ctx)
    r = torch_gpc(X, y, l)
    assert_gpc_fit(g, r)
    Xs = np.random.default_rng(16500).uniform(-4, 4, (2, 20000))
    fs, V = g.predict_latent(Xs)
    assert ctx.last_predict_path() == 4
    Ks = sqrexp(r["X"], torch.from_numpy(Xs).to(DEV), l)
    fs_ref = (Ks.T @ ((r["y"] + 1) / 2 - r["P"])).cpu().numpy()
    v = torch.linalg.solve_triangular(r["L"], r["sw"][:, None] * Ks, upper=False)
    V_ref = (1.0 - torch.sum(v * v, dim=0)).cpu().numpy()
    del Ks, v
    assert np.all(np.abs(fs - fs_ref) <= 1e-9 * np.max(np.abs(fs_ref)))
    assert np.all(np.abs(V - V_ref) <= 1e-9 * np.maximum(np.abs(V_ref), 1.0))
    sub = slice(0, 2000)
    labels = g.predict_class(Xs[:, sub]) >= 0.5
    want = np.array([oracle.logistic_gaussian_integral(m, s) for m, s in zip(fs_ref[sub], V_ref[sub])]) >= 0.5
    assert np.array_equal(labels, want)
