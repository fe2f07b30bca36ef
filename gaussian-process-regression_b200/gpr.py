"""GPR: host mirror of the R6 class of R/GPRclass.R:116-351 over the C ABI of libgprc.

The R host code of the drop-in (R/GPRclass.R in this package) has the same structure: argument checks, the noise-bump
retry loop and the return shapes live on the host; kernel-matrix build, Cholesky, solves and reductions are one
library call each."""
from __future__ import annotations

import ctypes as C
import warnings

import numpy as np

from . import _lib
from .kernels import (KernelSpec, as_matrix, cov_func, host_covariance_matrix, kernel_spec_of, constant, linear,
                      polynomial, sqrexp, gammaexp, rationalquadratic)


class _ReadOnly:
    """``stop("`$X` is read only")`` of the active bindings, R/GPRclass.R:230-280."""

    def __init__(self, name):
        self.name = name

    def __set_name__(self, owner, attr):
        self.attr = "_" + attr

    def __get__(self, obj, owner=None):
        if obj is None:
            return self
        return getattr(obj, self.attr)

    def __set__(self, obj, value):
        raise AttributeError("`$%s` is read only" % self.name)


class GPR:
    X = _ReadOnly("X")
    k = _ReadOnly("k")
    y = _ReadOnly("y")
    noise = _ReadOnly("noise")
    logp = _ReadOnly("logp")

    def __init__(self, X, y, noise=0.0, k=None, cov_names=None, ctx=None):
        # stopifnot(...) of R/GPRclass.R:129-133
        X = np.asarray(X)
        y = np.asarray(y)
        if not (np.issubdtype(X.dtype, np.number) and np.issubdtype(y.dtype, np.number) and y.ndim == 1):
            raise TypeError("is.numeric(X), is.vector(y), is.numeric(y) are not all TRUE")
        if not (np.isscalar(noise) or np.ndim(noise) == 0) or not float(noise) >= 0:
            raise ValueError("is.numeric(noise), length(noise) == 1, noise >= 0 are not all TRUE")
        X = as_matrix(X)
        y = y.astype(np.float64)
        noise = float(noise)
        if k is None:  # k = fit(X, y, noise, cov_names)$func                              R/GPRclass.R:127
            from .fit import fit
            k = fit(X, y, noise, cov_names)["func"]
        if len(y) != X.shape[1] or not callable(k):
            raise ValueError("length(y) == ncol(X), is.function(k) are not all TRUE")
        self._ctx = ctx or _lib.default_context()
        self._X, self._y, self._k = X, y, k
        self._handle = None
        lib = self._ctx.lib
        spec = kernel_spec_of(k)
        n = X.shape[1]
        xp = _lib.points(X)
        K = None if spec is not None else np.asfortranarray(host_covariance_matrix(X, X, k))
        new_noise = noise
        handle = _lib._P()
        logp = C.c_double(0.0)
        info = C.c_long(0)
        ok = False
        for i in range(1, 11):  # R/GPRclass.R:141-148
            if spec is not None:
                kc, keep = spec.to_c()
                _lib.check(lib.gprc_gpr_fit(self._ctx.handle, kc, _lib.dptr(xp), X.shape[0], n, _lib.dptr(y),
                                            new_noise, C.byref(handle), C.byref(logp), C.byref(info)))
            else:
                _lib.check(lib.gprc_gpr_fit_precomputed(self._ctx.handle, _lib.dptr(K), n, _lib.dptr(y), new_noise,
                                                        C.byref(handle), C.byref(logp), C.byref(info)))
            if info.value == 0 and np.isfinite(logp.value):
                if i > 1:
                    warnings.warn("Noise got changed to %s to avoid errors in cholesky decomposition" % _fmt(new_noise))
                ok = True
                break
            if handle:
                lib.gprc_gpr_free(handle)
                handle = _lib._P()
            new_noise = 0.01 * i + noise
        if not ok:  # R/GPRclass.R:149
            raise ValueError("Inputs lead to non positive definite covariance matrix. "
                             "Try using a larger noise or a smaller lengthscale.")
        self._handle = handle
        self._noise = new_noise
        self._logp = np.array([[logp.value]])  # a 1 x 1 matrix in R (y %*% alpha)
        self._alpha = None
        self._L = None

    # R6 spelling
    @classmethod
    def new(cls, *args, **kwargs):
        return cls(*args, **kwargs)

    def __del__(self):  # pragma: no cover
        try:
            if getattr(self, "_handle", None) and getattr(self._ctx, "handle", None):
                self._ctx.lib.gprc_gpr_free(self._handle)
                self._handle = None
        except Exception:
            pass

    @property
    def alpha(self):
        if self._alpha is None:
            a = np.empty(self._X.shape[1])
            _lib.check(self._ctx.lib.gprc_gpr_get(self._handle, _lib.GET_ALPHA, _lib.dptr(a)))
            self._alpha = a
        return self._alpha

    @alpha.setter
    def alpha(self, value):
        raise AttributeError("`$alpha` is read only")

    @property
    def L(self):
        """t(chol(K + noise I)): dense lower-triangular n x n, downloaded on first use (20 GB at n = 50k)."""
        if self._L is None:
            n = self._X.shape[1]
            out = np.empty((n, n), order="F")
            _lib.check(self._ctx.lib.gprc_gpr_get(self._handle, _lib.GET_L, _lib.dptr(out)))
            self._L = out
        return self._L

    @L.setter
    def L(self, value):
        raise AttributeError("`$L` is read only")

    def predict_grid(self, limits, per_dim):
        """$predict on the test grid simulate_regression() builds (R/simulation.R:101-102: per_dim points per dimension
        between the limits, combined by combine_all), generated on the device (gprc_gpr_predict_grid, SURVEY.md 8f-4):
        per_dim^D x 2 matrix cbind(mean, var) in the grid's own point order."""
        limits = np.ascontiguousarray(np.asarray(limits, dtype=np.float64).reshape(-1, 2))
        D = self._X.shape[0]
        if limits.shape[0] != D:
            raise ValueError("limits must have one (lower, upper) row per dimension")
        if kernel_spec_of(self._k) is None:
            raise TypeError("predict_grid needs a built-in kernel (cov_func of sqrexp, ...)")
        m = int(per_dim) ** D
        mean, var = np.empty(m), np.empty(m)
        _lib.check(self._ctx.lib.gprc_gpr_predict_grid(self._handle, _lib.dptr(limits), int(per_dim), _lib.dptr(mean),
                                                       _lib.dptr(var)))
        return np.column_stack([mean, var])

    def predict(self, X_star, pointwise_var=True):
        """R/GPRclass.R:155-170: m x 2 matrix cbind(mean, var), or list(mean (m x 1), cov (m x m))."""
        X_star = np.asarray(X_star, dtype=np.float64)
        D = self._X.shape[0]
        if X_star.size % D != 0:
            raise ValueError("is.numeric(X_star), length(X_star) %% nrow(self$X) == 0 are not all TRUE")
        if X_star.ndim < 2:
            X_star = X_star.reshape(-1, D).T  # dim(X_star) <- c(D, length / D)  (column-major fill)
        elif X_star.ndim != 2 or X_star.shape[0] != D:
            # a matrix with the wrong number of rows passes the length check of R/GPRclass.R:156 and then fails inside
            # covariance_matrix ("non-conformable arrays"): the library must never read d * m doubles from such a buffer
            raise ValueError("non-conformable arrays: nrow(X_star) = %d, nrow(self$X) = %d" % (X_star.shape[0], D))
        m = X_star.shape[1]
        lib, h = self._ctx.lib, self._handle
        spec = kernel_spec_of(self._k)
        mean = np.empty(m)
        if pointwise_var:
            var = np.empty(m)
            if spec is not None:
                xs = _lib.points(X_star)
                _lib.check(lib.gprc_gpr_predict(h, _lib.dptr(xs), m, _lib.dptr(mean), _lib.dptr(var)))
            else:
                Ks = np.asfortranarray(host_covariance_matrix(self._X, X_star, self._k))
                kss = np.ascontiguousarray(np.asarray(self._k(X_star, X_star), dtype=np.float64))
                _lib.check(lib.gprc_gpr_predict_precomputed(h, _lib.dptr(Ks), _lib.dptr(kss), m, _lib.dptr(mean),
                                                            _lib.dptr(var)))
            return np.column_stack([mean, var])
        cov = np.empty((m, m), order="F")
        if spec is not None:
            xs = _lib.points(X_star)
            _lib.check(lib.gprc_gpr_predict_cov(h, _lib.dptr(xs), m, _lib.dptr(mean), _lib.dptr(cov)))
        else:
            # closure kernel: v = L^-1 K_star column by column through the pointwise path, Sigma on the host
            Linv = np.empty((self._X.shape[1],) * 2, order="F")
            _lib.check(lib.gprc_gpr_get(h, _lib.GET_LINV, _lib.dptr(Linv)))
            Ks = host_covariance_matrix(self._X, X_star, self._k)
            v = Linv @ Ks
            mean = Ks.T @ self.alpha
            cov = host_covariance_matrix(X_star, X_star, self._k) - v.T @ v
        return [mean.reshape(-1, 1), cov]

    def add_points(self, X_new, y_new):
        """Append training points in place and return the model: afterwards it is GPR(cbind(X, X_new), c(y, y_new),
        noise = self.noise, k = self.k) (the kernel is kept, never re-fitted).  X_new follows predict's reshape rule.
        Built-in kernels extend the existing Cholesky factor on the device (gprc_gpr_append); if the enlarged matrix is
        not positive definite with this noise, or the kernel is a closure, the constructor's path runs on the
        concatenated data (noise-bump loop from self.noise, same warning and error)."""
        X_new = np.asarray(X_new)
        y_new = np.asarray(y_new)
        D = self._X.shape[0]
        if not np.issubdtype(X_new.dtype, np.number) or X_new.size % D != 0:
            raise ValueError("is.numeric(X_new), length(X_new) %% nrow(self$X) == 0 are not all TRUE")
        X_new = X_new.astype(np.float64)
        if X_new.ndim < 2:
            X_new = X_new.reshape(-1, D).T  # dim(X_new) <- c(D, length / D)  (column-major fill)
        elif X_new.ndim != 2 or X_new.shape[0] != D:
            raise ValueError("non-conformable arrays: nrow(X_new) = %d, nrow(self$X) = %d" % (X_new.shape[0], D))
        m = X_new.shape[1]
        if not (np.issubdtype(y_new.dtype, np.number) and y_new.ndim == 1 and len(y_new) == m):
            raise ValueError("is.numeric(y_new), is.vector(y_new), length(y_new) == ncol(X_new) are not all TRUE")
        if m == 0:
            return self
        X_all = np.concatenate([self._X, X_new], axis=1)
        y_all = np.concatenate([self._y, y_new.astype(np.float64)])
        if kernel_spec_of(self._k) is not None:
            lib = self._ctx.lib
            xp = _lib.points(X_new)
            yp = np.ascontiguousarray(y_new, dtype=np.float64)
            logp = C.c_double(0.0)
            info = C.c_long(0)
            _lib.check(lib.gprc_gpr_append(self._handle, _lib.dptr(xp), m, _lib.dptr(yp), C.byref(logp),
                                           C.byref(info)))
            if info.value == 0 and np.isfinite(logp.value):
                self._X, self._y = X_all, y_all
                self._logp = np.array([[logp.value]])
                self._alpha = None
                self._L = None
                return self
        fresh = GPR(X_all, y_all, noise=self._noise, k=self._k, ctx=self._ctx)
        self._ctx.lib.gprc_gpr_free(self._handle)
        self._handle, fresh._handle = fresh._handle, None
        self._X, self._y, self._noise, self._logp = fresh._X, fresh._y, fresh._noise, fresh._logp
        self._alpha = None
        self._L = None
        return self


def _fmt(x):
    return ("%.15g" % x)


def _fit_par(X, y, noise, name):
    from .fit import fit
    return fit(X, y, noise, [name])["par"]


class GPR_constant(GPR):  # R/GPRclass.R:284-292
    def __init__(self, X, y, noise, c=None, ctx=None):
        if c is None:
            c = _fit_par(X, y, noise, "constant")
        c = float(np.asarray(c).ravel()[0])
        if not c > 0:
            raise ValueError("is.numeric(c), c > 0 are not all TRUE")
        super().__init__(X, y, noise, cov_func(constant, c=c), ctx=ctx)


class GPR_linear(GPR):  # R/GPRclass.R:295-303
    def __init__(self, X, y, noise, sigma=None, ctx=None):
        if sigma is None:
            sigma = _fit_par(X, y, noise, "linear")
        sigma = np.atleast_1d(np.asarray(sigma, dtype=float))
        if len(sigma) != as_matrix(X).shape[0]:
            raise ValueError("length(sigma) == nrow(X) is not TRUE")
        super().__init__(X, y, noise, cov_func(linear, sigma=sigma if len(sigma) > 1 else float(sigma[0])), ctx=ctx)


class GPR_polynomial(GPR):  # R/GPRclass.R:306-315
    def __init__(self, X, y, noise, sigma=None, p=None, ctx=None):
        if sigma is None or p is None:
            par = _fit_par(X, y, noise, "polynomial")
            sigma = par[0] if sigma is None else sigma
            p = par[1] if p is None else p
        super().__init__(X, y, noise, cov_func(polynomial, sigma=float(sigma), p=float(p)), ctx=ctx)


class GPR_sqrexp(GPR):  # R/GPRclass.R:318-327
    def __init__(self, X, y, noise, l=None, ctx=None):
        if l is None:
            l = _fit_par(X, y, noise, "sqrexp")
        super().__init__(X, y, noise, cov_func(sqrexp, l=float(np.asarray(l).ravel()[0])), ctx=ctx)


class GPR_gammaexp(GPR):  # R/GPRclass.R:330-339 -- NB reads par[[1]] as gamma and par[[2]] as l (SURVEY.md A.6)
    def __init__(self, X, y, noise, gamma=None, l=None, ctx=None):
        if gamma is None or l is None:
            par = _fit_par(X, y, noise, "gammaexp")
            gamma = par[0] if gamma is None else gamma
            l = par[1] if l is None else l
        super().__init__(X, y, noise, cov_func(gammaexp, l=float(l), gamma=float(gamma)), ctx=ctx)


class GPR_rationalquadratic(GPR):  # R/GPRclass.R:342-351 -- par[[1]] as alpha, par[[2]] as l (A.6)
    def __init__(self, X, y, noise, alpha=None, l=None, ctx=None):
        if alpha is None or l is None:
            par = _fit_par(X, y, noise, "rationalquadratic")
            alpha = par[0] if alpha is None else alpha
            l = par[1] if l is None else l
        super().__init__(X, y, noise, cov_func(rationalquadratic, l=float(l), alpha=float(alpha)), ctx=ctx)


# R spelling: GPR.sqrexp$new(...)
GPR.constant = GPR_constant
GPR.linear = GPR_linear
GPR.polynomial = GPR_polynomial
GPR.sqrexp = GPR_sqrexp
GPR.gammaexp = GPR_gammaexp
GPR.rationalquadratic = GPR_rationalquadratic
