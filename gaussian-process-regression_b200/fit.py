"""fit(): hyper-parameter optimisation, host mirror of R/fit.R.  The optimiser loops stay on the host; ``dens`` and
``dens_deriv`` (R/fit.R:117-139) are evaluated by libgprc (gprc_logml / gprc_logml_grad).

Independent units -- kernel families (R/fit.R:113), polynomial degrees (R/fit.R:148) and, as an extension, several
start vectors -- are sharded across ranks when a torch.distributed process group is passed (SURVEY.md section 8e)."""
from __future__ import annotations

import ctypes as C
import math
import sys

import numpy as np

from . import _lib
from ._optim import OptimError, r_optim
from .kernels import BUILTIN, PARAM_NAMES, CovFunc, KernelSpec, as_matrix, cov_func

# R/fit.R:2-33: registry of kernels and optimiser start values, in the order of names(cov_dict)
cov_dict = {
    "sqrexp": dict(func=BUILTIN["sqrexp"], display="Squared Exponential", start=[1.0]),
    "gammaexp": dict(func=BUILTIN["gammaexp"], display="Gamma Exponential", start=[1.0, 1.0]),
    "constant": dict(func=BUILTIN["constant"], display="Constant", start=[1.0]),
    "linear": dict(func=BUILTIN["linear"], display="Linear", start=[1.0]),
    "polynomial": dict(func=BUILTIN["polynomial"], display="Polynomial", start=[1.0, 2.0]),
    "rationalquadratic": dict(func=BUILTIN["rationalquadratic"], display="Rational Quadratic", start=[1.0, 1.0]),
}
HAS_DERIV = ("sqrexp", "gammaexp", "rationalquadratic", "polynomial")  # R/fit.R:125


def _spec(name, v):
    v = list(np.atleast_1d(np.asarray(v, dtype=float)))
    return KernelSpec(name, **dict(zip(PARAM_NAMES[name], v)))  # positional, as do.call(func, append(list(x, y), v))


class Objective:
    """dens / dens_deriv bound to one data set; X and y are converted once."""

    def __init__(self, X, y, noise, ctx=None, minors="literal"):
        self.X = as_matrix(X)
        self.y = np.ascontiguousarray(np.asarray(y, dtype=np.float64))
        self.noise = float(noise)
        self.ctx = ctx or _lib.default_context()
        self.xp = _lib.points(self.X)
        self.minors = minors

    def dens(self, name, v):
        """log p(y | X, theta), R/fit.R:117-124.  Raises OptimError where the reference's stopifnot/chol would."""
        kc, keep = _spec(name, v).to_c()
        logp, minlog, info = C.c_double(0.0), C.c_double(0.0), C.c_long(0)
        _lib.check(self.ctx.lib.gprc_logml(self.ctx.handle, kc, _lib.dptr(self.xp), self.X.shape[0], self.X.shape[1],
                                           _lib.dptr(self.y), self.noise, C.byref(logp), C.byref(minlog),
                                           C.byref(info)))
        if info.value != 0 or not math.isfinite(logp.value):
            raise OptimError("not positive definite (leading minor %d)" % info.value)
        # R/fit.R:119: min over the leading minors of det(.) > 0, with det() = exp(log-modulus), which rounds to 0 below
        # log(2^-1075) = -745.13 (A.4): the same exp() decides here
        if self.minors == "literal" and not (math.exp(minlog.value) > 0.0):
            raise OptimError("min(sapply(..., det)) > 0 is not TRUE")
        return logp.value

    def dens_deriv(self, name, v, formula=_lib.GRAD_AS_CODED):
        """R/fit.R:126-139 (as coded by default: SURVEY.md A.5, A.6)."""
        kc, keep = _spec(name, v).to_c()
        nparam = len(cov_dict[name]["start"])
        grad = np.zeros(nparam)
        info = C.c_long(0)
        _lib.check(self.ctx.lib.gprc_logml_grad(self.ctx.handle, kc, _lib.dptr(self.xp), self.X.shape[0],
                                                self.X.shape[1], _lib.dptr(self.y), self.noise, formula,
                                                _lib.dptr(grad), nparam, C.byref(info)))
        if info.value != 0:
            raise OptimError("system is computationally singular")  # solve(K) of R/fit.R:136
        return grad

    def fit_family(self, name):
        """One pass of the loop body of R/fit.R:113-162 inside the library (gprc_fit_family, csrc/optim.hpp): X and y
        are uploaded once, the optimiser (Brent_fmin / vmmin / optim_until_error restated in C++) runs in the call and
        every dens / dens_deriv evaluation stays on the device.  Same trajectory as ``_fit_one`` on the host."""
        par, npar, value = np.zeros(2), C.c_int(0), C.c_double(0.0)
        evals = (C.c_long * 2)()
        _lib.check(self.ctx.lib.gprc_fit_family(self.ctx.handle, _lib.KERNEL_IDS[name], _lib.dptr(self.xp),
                                                self.X.shape[0], self.X.shape[1], _lib.dptr(self.y), self.noise,
                                                0 if self.minors == "literal" else 1, _lib.dptr(par), C.byref(npar),
                                                C.byref(value), evals))
        return dict(par=par[:npar.value].copy(), value=value.value, evaluations=(evals[0], evals[1]))

    def dens_batch(self, name, thetas):
        """Independent evaluations in one call (multi-start / grid): returns logp (nan where not PD)."""
        thetas = np.atleast_2d(np.asarray(thetas, dtype=float))
        specs = (_lib.GprcKernel * len(thetas))()
        keeps = []
        for i, v in enumerate(thetas):
            kc, keep = _spec(name, v).to_c()
            specs[i] = kc
            keeps.append(keep)
        logp = np.zeros(len(thetas))
        minlog = np.zeros(len(thetas))
        info = (C.c_long * len(thetas))()
        _lib.check(self.ctx.lib.gprc_logml_batch(self.ctx.handle, specs, len(thetas), _lib.dptr(self.xp),
                                                 self.X.shape[0], self.X.shape[1], _lib.dptr(self.y), self.noise,
                                                 _lib.dptr(logp), _lib.dptr(minlog), info))
        return logp, minlog, np.array(list(info))


def optim_until_error(start, f, **kw):
    """R/fit.R:47-69: objective errors score -10000; if optim() itself throws, the best recorded evaluation wins."""
    record = []
    errors = (OptimError, np.linalg.LinAlgError, FloatingPointError, ValueError, ZeroDivisionError)

    def f_new(p):
        try:
            out = f(p)
        except errors:
            return -10000.0
        if not out == -10000:
            record.append((np.array(p, dtype=float), out))
        return out

    gr = kw.pop("gr", None)
    try:
        return r_optim(start, f_new, gr=gr, **kw)
    except errors:
        if not record:
            try:
                value = f(np.asarray(start, float))
            except errors:
                value = -10000.0
            return dict(par=np.asarray(start, float), value=value)
        best = int(np.argmax([r[1] for r in record]))
        return dict(par=record[best][0], value=record[best][1])


def _fit_one(obj, cov, engine="host"):
    """One pass of the loop body of R/fit.R:113-162 for the covariance family ``cov``.  engine = "library" runs the
    optimiser inside libgprc (Objective.fit_family); "host" drives it from here, one ABI call per evaluation."""
    if engine == "library":
        r = obj.fit_family(cov)
        return dict(par=r["par"], value=r["value"])
    nparam = len(cov_dict[cov]["start"])
    f = lambda v: obj.dens(cov, v)
    kw = {}
    if cov in HAS_DERIV:
        kw["gr"] = lambda v: obj.dens_deriv(cov, v)
    if nparam == 1:
        kw.update(method="Brent", lower=0.0, upper=10.0)
    else:
        kw.update(method="BFGS")
    if cov == "polynomial":  # R/fit.R:145-156
        cands = [optim_until_error([cov_dict[cov]["start"][0]], lambda sig, i=i: f([float(np.atleast_1d(sig)[0]), float(i)]),
                                   method="Brent", lower=0.0, upper=5.0) for i in range(1, 11)]
        best = int(np.argmax([q["value"] for q in cands]))
        return dict(par=np.array([float(np.atleast_1d(cands[best]["par"])[0]), float(best + 1)]),
                    value=cands[best]["value"])
    return optim_until_error(cov_dict[cov]["start"], f, **kw)


def fit(X, y, noise, cov_names=None, ctx=None, minors="literal", group=None, verbose=True, engine="host"):
    """fit(X, y, noise, cov_names), R/fit.R:110-169 -> dict(par, cov, score, func).

    ``group``: optional torch.distributed process group; the covariance families are dealt round-robin to the ranks
    and the (par, value) pairs are all-gathered, after which every rank applies which.max (R/fit.R:164)."""
    cov_names = list(cov_dict) if cov_names is None else list(cov_names)
    for c in cov_names:
        if c not in cov_dict:
            raise KeyError(c)
    obj = Objective(X, y, noise, ctx=ctx, minors=minors)
    if group is None:
        results = [_fit_one(obj, cov, engine) for cov in cov_names]
    else:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        mine = {i: _fit_one(obj, cov, engine) for i, cov in enumerate(cov_names) if i % world == rank}
        payload = {i: (np.atleast_1d(r["par"]).tolist(), float(r["value"])) for i, r in mine.items()}
        gathered = [None] * world
        dist.all_gather_object(gathered, payload, group=group)
        merged = {}
        for part in gathered:
            merged.update(part)
        results = [dict(par=np.array(merged[i][0]), value=merged[i][1]) for i in range(len(cov_names))]
    params = [np.atleast_1d(r["par"]) for r in results]
    score = [float(r["value"]) for r in results]
    best = int(np.argmax(score))
    name, par = cov_names[best], params[best]
    if verbose:
        print("The optimal covariance function is %s, with parameters %s" % (name, ", ".join("%.15g" % p for p in par)),
              file=sys.stderr)  # message(), R/fit.R:166
    func = cov_func(cov_dict[name]["func"], *[float(p) for p in par])
    return dict(par=par, cov=name, score=score, func=func)


def multistart(X, y, noise, cov, starts, ctx=None, group=None):
    """Extension used by BASELINE config 3: evaluate / optimise from several start vectors, sharded across ranks.
    Returns the (start, par, value) of every start; each trajectory is the reference's optimiser for ``cov``."""
    obj = Objective(X, y, noise, ctx=ctx, minors="cholesky")
    starts = np.atleast_2d(np.asarray(starts, dtype=float))
    idx = list(range(len(starts)))
    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    out = {}
    for i in idx:
        if i % world != rank:
            continue
        kw = dict(method="BFGS", gr=lambda v: obj.dens_deriv(cov, v, _lib.GRAD_TEXTBOOK)) if starts.shape[1] > 1 \
            else dict(method="Brent", lower=0.0, upper=10.0)
        r = optim_until_error(starts[i], lambda v: obj.dens(cov, v), **kw)
        out[i] = (np.atleast_1d(r["par"]).tolist(), float(r["value"]))
    if group is not None:
        import torch.distributed as dist
        gathered = [None] * world
        dist.all_gather_object(gathered, out, group=group)
        out = {}
        for part in gathered:
            out.update(part)
    return [dict(start=starts[i], par=np.array(out[i][0]), value=out[i][1]) for i in idx]
