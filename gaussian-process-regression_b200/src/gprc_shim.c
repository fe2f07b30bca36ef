/*
 * gprc_shim.c -- the `.Call` shim between the R host code (R/GPRclass.R, R/GPCclass.R, R/fit.R of this package) and
 * libgprc's C ABI (include/gprc.h).  It is deliberately logic-free: unwrap SEXP arguments, call one library function,
 * wrap the results.  Rules it follows (SURVEY.md section 7, "R's .Call contract"):
 *   - R owns every SEXP buffer; nothing is retained across calls except external pointers to library handles;
 *   - library handles live in EXTPTRSXPs with C finalizers (R_RegisterCFinalizerEx, onexit = TRUE);
 *   - the library never longjmps: status codes come back first, resources are released, THEN Rf_error is raised.
 * R is not installed in the build image, so this file is compile-checked against tests/stubs/Rinternals.h only
 * (tests/test_abi_and_host.py); it needs R's real headers and `R CMD SHLIB` to produce gprc.so.
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <string.h>

#include "gprc.h"

static gprc_ctx* g_ctx = NULL;

/* A pending Ctrl-C is detected WITHOUT long-jumping through library frames: R_CheckUserInterrupt runs inside
 * R_ToplevelExec, which returns FALSE if it jumped.  The library polls this between chunks of a long predict and returns
 * -8; the entry point then releases what it holds and raises the interrupt from shim level (SURVEY.md section 8b). */
static void check_interrupt_body(void* unused) { (void)unused; R_CheckUserInterrupt(); }
static int interrupt_pending(void* unused) { (void)unused; return R_ToplevelExec(check_interrupt_body, NULL) == FALSE; }

static gprc_ctx* ctx(void) {
  if (!g_ctx) {
    int dev = 0;
    SEXP opt = Rf_GetOption1(Rf_install("gprc.device"));
    if (opt != R_NilValue) dev = Rf_asInteger(opt);
    if (gprc_ctx_create(&g_ctx, dev) != 0) Rf_error("gprc: %s", gprc_last_error());
    gprc_ctx_set_interrupt(g_ctx, interrupt_pending, NULL);
  }
  return g_ctx;
}

/* list(id=, c=, sigma=, p=, l=, gamma=, alpha=) -- the `gprc_kernel` attribute cov_func() attaches (NAMED, A.6) */
static void kernel_from_sexp(SEXP k, gprc_kernel* out) {
  memset(out, 0, sizeof *out);
  SEXP names = Rf_getAttrib(k, R_NamesSymbol);
  for (R_xlen_t i = 0; i < XLENGTH(k); ++i) {
    const char* nm = CHAR(STRING_ELT(names, i));
    SEXP v = VECTOR_ELT(k, i);
    if (!strcmp(nm, "id")) out->id = Rf_asInteger(v);
    else if (!strcmp(nm, "c")) out->c = Rf_asReal(v);
    else if (!strcmp(nm, "p")) out->p = Rf_asReal(v);
    else if (!strcmp(nm, "l")) out->l = Rf_asReal(v);
    else if (!strcmp(nm, "gamma")) out->gamma = Rf_asReal(v);
    else if (!strcmp(nm, "alpha")) out->alpha = Rf_asReal(v);
    else if (!strcmp(nm, "sigma")) {
      if (XLENGTH(v) > 1) { out->sigma_vec = REAL(v); out->sigma_len = (int)XLENGTH(v); }
      else out->sigma = Rf_asReal(v);
    }
  }
}

static void gpr_finalizer(SEXP p) {
  gprc_gpr* g = (gprc_gpr*)R_ExternalPtrAddr(p);
  if (g) { gprc_gpr_free(g); R_ClearExternalPtr(p); }
}
static void gpc_finalizer(SEXP p) {
  gprc_gpc* g = (gprc_gpc*)R_ExternalPtrAddr(p);
  if (g) { gprc_gpc_free(g); R_ClearExternalPtr(p); }
}

/* covariance_matrix(A, B, k), R/GPRclass.R:355-357 */
SEXP C_gprc_cov_matrix(SEXP k, SEXP A, SEXP B) {
  gprc_kernel kk; kernel_from_sexp(k, &kk);
  const int d = Rf_nrows(A); const long nA = Rf_ncols(A), nB = Rf_ncols(B);
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, (int)nA, (int)nB));
  int rc = gprc_cov_matrix(ctx(), &kk, REAL(A), d, nA, REAL(B), nB, REAL(out));
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  return out;
}

/* one attempt of the loop R/GPRclass.R:141-148; K is NULL for built-in kernels, else the precomputed matrix.
 * returns list(ptr, logp, info) */
SEXP C_gprc_gpr_fit(SEXP k, SEXP X, SEXP y, SEXP noise, SEXP K) {
  gprc_gpr* g = NULL; double logp = NA_REAL; long info = 0; int rc;
  const long n = XLENGTH(y);
  if (K == R_NilValue) {
    gprc_kernel kk; kernel_from_sexp(k, &kk);
    rc = gprc_gpr_fit(ctx(), &kk, REAL(X), Rf_nrows(X), n, REAL(y), Rf_asReal(noise), &g, &logp, &info);
  } else {
    rc = gprc_gpr_fit_precomputed(ctx(), REAL(K), n, REAL(y), Rf_asReal(noise), &g, &logp, &info);
  }
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 3));
  SEXP ptr = PROTECT(R_MakeExternalPtr(g, R_NilValue, R_NilValue));
  if (g) R_RegisterCFinalizerEx(ptr, gpr_finalizer, TRUE);
  SET_VECTOR_ELT(out, 0, ptr);
  SET_VECTOR_ELT(out, 1, Rf_ScalarReal(logp));
  SET_VECTOR_ELT(out, 2, Rf_ScalarReal((double)info));
  UNPROTECT(2);
  return out;
}

/* $predict(X_star, pointwise_var = TRUE): cbind(mean, var), R/GPRclass.R:160-165 */
SEXP C_gprc_gpr_predict(SEXP ptr, SEXP Xs, SEXP Ks, SEXP kss) {
  gprc_gpr* g = (gprc_gpr*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL (restored from saveRDS?); rebuild with GPR$new");
  const long m = (Ks == R_NilValue) ? Rf_ncols(Xs) : Rf_ncols(Ks);
  /* the library reads d x m (or n x m) doubles: a matrix with the wrong number of rows must never reach it */
  if (Ks == R_NilValue ? Rf_nrows(Xs) != gprc_gpr_dim(g) : Rf_nrows(Ks) != gprc_gpr_n(g) || Rf_length(kss) != m)
    Rf_error("non-conformable arrays");
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, (int)m, 2));
  int rc = (Ks == R_NilValue) ? gprc_gpr_predict(g, REAL(Xs), m, REAL(out), REAL(out) + m)
                              : gprc_gpr_predict_precomputed(g, REAL(Ks), REAL(kss), m, REAL(out), REAL(out) + m);
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  return out;
}

/* $predict(X_star, pointwise_var = FALSE): list(mean (m x 1), cov (m x m)), R/GPRclass.R:167-168 */
SEXP C_gprc_gpr_predict_cov(SEXP ptr, SEXP Xs) {
  gprc_gpr* g = (gprc_gpr*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL");
  const long m = Rf_ncols(Xs);
  if (Rf_nrows(Xs) != gprc_gpr_dim(g)) Rf_error("non-conformable arrays");
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 2));
  SEXP mean = PROTECT(Rf_allocMatrix(REALSXP, (int)m, 1));
  SEXP cov = PROTECT(Rf_allocMatrix(REALSXP, (int)m, (int)m));
  int rc = gprc_gpr_predict_cov(g, REAL(Xs), m, REAL(mean), REAL(cov));
  SET_VECTOR_ELT(out, 0, mean); SET_VECTOR_ELT(out, 1, cov);
  UNPROTECT(3);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  return out;
}

/* $add_points(X_new, y_new) of built-in kernels: list(logp, info); info > 0 leaves the model as it was */
SEXP C_gprc_gpr_append(SEXP ptr, SEXP Xnew, SEXP ynew) {
  gprc_gpr* g = (gprc_gpr*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL");
  const long k = Rf_ncols(Xnew);
  /* the library reads d x k and k doubles */
  if (Rf_nrows(Xnew) != gprc_gpr_dim(g) || XLENGTH(ynew) != k) Rf_error("non-conformable arrays");
  double logp = NA_REAL; long info = 0;
  int rc = gprc_gpr_append(g, REAL(Xnew), k, REAL(ynew), &logp, &info);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 2));
  SET_VECTOR_ELT(out, 0, Rf_ScalarReal(logp));
  SET_VECTOR_ELT(out, 1, Rf_ScalarReal((double)info));
  UNPROTECT(1);
  return out;
}

/* active bindings $L / $alpha (lazy download), R/GPRclass.R:258-273 */
SEXP C_gprc_gpr_get(SEXP ptr, SEXP what) {
  gprc_gpr* g = (gprc_gpr*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL");
  const int w = Rf_asInteger(what); const long n = gprc_gpr_n(g);
  SEXP out = PROTECT(w == GPRC_GET_ALPHA ? Rf_allocVector(REALSXP, n) : Rf_allocMatrix(REALSXP, (int)n, (int)n));
  int rc = gprc_gpr_get(g, w, REAL(out));
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  return out;
}

/* dens(v), R/fit.R:117-124: c(logp, min_leading_logdet, info) */
SEXP C_gprc_logml(SEXP k, SEXP X, SEXP y, SEXP noise) {
  gprc_kernel kk; kernel_from_sexp(k, &kk);
  double logp = NA_REAL, minlog = NA_REAL; long info = 0;
  int rc = gprc_logml(ctx(), &kk, REAL(X), Rf_nrows(X), XLENGTH(y), REAL(y), Rf_asReal(noise), &logp, &minlog, &info);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  SEXP out = PROTECT(Rf_allocVector(REALSXP, 3));
  REAL(out)[0] = logp; REAL(out)[1] = minlog; REAL(out)[2] = (double)info;
  UNPROTECT(1);
  return out;
}

/* dens_deriv(v), R/fit.R:126-139 */
SEXP C_gprc_logml_grad(SEXP k, SEXP X, SEXP y, SEXP noise, SEXP formula, SEXP nparam) {
  gprc_kernel kk; kernel_from_sexp(k, &kk);
  const int np = Rf_asInteger(nparam); long info = 0;
  SEXP out = PROTECT(Rf_allocVector(REALSXP, np));
  int rc = gprc_logml_grad(ctx(), &kk, REAL(X), Rf_nrows(X), XLENGTH(y), REAL(y), Rf_asReal(noise),
                           Rf_asInteger(formula), REAL(out), np, &info);
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  if (info) Rf_error("Lapack routine dgesv: system is exactly singular");  /* solve(K) of R/fit.R:136 */
  return out;
}

/* GPC$initialize Newton loop, R/GPCclass.R:73-103: list(ptr, iters, trace, sum_diagL, sum_log_diagL, status) */
SEXP C_gprc_gpc_fit(SEXP k, SEXP X, SEXP y, SEXP eps, SEXP guard, SEXP K) {
  gprc_gpc* g = NULL; int iters = 0, status = 0; double sd = NA_REAL, sl = NA_REAL; double trace[256]; int rc;
  const long n = XLENGTH(y);
  if (K == R_NilValue) {
    gprc_kernel kk; kernel_from_sexp(k, &kk);
    rc = gprc_gpc_fit(ctx(), &kk, REAL(X), Rf_nrows(X), n, REAL(y), Rf_asReal(eps), Rf_asLogical(guard), 0, &g,
                      &iters, trace, 256, &sd, &sl, &status);
  } else {
    rc = gprc_gpc_fit_precomputed(ctx(), REAL(K), n, REAL(y), Rf_asReal(eps), Rf_asLogical(guard), 0, &g, &iters,
                                  trace, 256, &sd, &sl, &status);
  }
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  SEXP out = PROTECT(Rf_allocVector(VECSXP, 6));
  SEXP ptr = PROTECT(R_MakeExternalPtr(g, R_NilValue, R_NilValue));
  if (g) R_RegisterCFinalizerEx(ptr, gpc_finalizer, TRUE);
  const int nt = iters < 256 ? iters : 256;
  SEXP tr = PROTECT(Rf_allocVector(REALSXP, nt));
  memcpy(REAL(tr), trace, sizeof(double) * nt);
  SET_VECTOR_ELT(out, 0, ptr); SET_VECTOR_ELT(out, 1, Rf_ScalarInteger(iters)); SET_VECTOR_ELT(out, 2, tr);
  SET_VECTOR_ELT(out, 3, Rf_ScalarReal(sd)); SET_VECTOR_ELT(out, 4, Rf_ScalarReal(sl));
  SET_VECTOR_ELT(out, 5, Rf_ScalarInteger(status));
  UNPROTECT(3);
  return out;
}

/* fs_bar / Vfs of $predict_class, R/GPCclass.R:110-115: m x 2 matrix */
SEXP C_gprc_gpc_predict_latent(SEXP ptr, SEXP Xs, SEXP Ks, SEXP kss) {
  gprc_gpc* g = (gprc_gpc*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL");
  const long m = (Ks == R_NilValue) ? Rf_ncols(Xs) : Rf_ncols(Ks);
  /* the library reads d x m (or n x m) doubles: a matrix with the wrong number of rows must never reach it */
  if (Ks == R_NilValue ? Rf_nrows(Xs) != gprc_gpc_dim(g) : Rf_nrows(Ks) != gprc_gpc_n(g) || Rf_length(kss) != m)
    Rf_error("non-conformable arrays");
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, (int)m, 2));
  int rc = (Ks == R_NilValue) ? gprc_gpc_predict_latent(g, REAL(Xs), m, REAL(out), REAL(out) + m)
                              : gprc_gpc_predict_latent_precomputed(g, REAL(Ks), REAL(kss), m, REAL(out), REAL(out) + m);
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  return out;
}

/* $predict_class complete on the device (latent prediction + QUADPACK dqagi per point), R/GPCclass.R:108-118.
 * Returns the probabilities; a non-zero QUADPACK code raises the message integrate() would raise. */
SEXP C_gprc_gpc_predict_class(SEXP ptr, SEXP Xs) {
  static const char* msg[] = {"", "maximum number of subdivisions reached", "roundoff error was detected",
                              "extremely bad integrand behaviour",
                              "roundoff error is detected in the extrapolation table",
                              "the integral is probably divergent", "the input is invalid"};
  gprc_gpc* g = (gprc_gpc*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL");
  const long m = Rf_ncols(Xs);
  if (Rf_nrows(Xs) != gprc_gpc_dim(g)) Rf_error("non-conformable arrays");
  SEXP out = PROTECT(Rf_allocVector(REALSXP, m));
  int* ier = (int*)R_alloc((size_t)m, sizeof(int));
  int rc = gprc_gpc_predict_class(g, REAL(Xs), m, REAL(out), ier);
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  for (long i = 0; i < m; ++i) {
    if (ier[i] < 0) Rf_error("non-finite function value");
    if (ier[i] > 0) Rf_error("%s", msg[ier[i] <= 6 ? ier[i] : 6]);
  }
  return out;
}

SEXP C_gprc_gpc_get(SEXP ptr, SEXP what) {
  gprc_gpc* g = (gprc_gpc*)R_ExternalPtrAddr(ptr);
  if (!g) Rf_error("gprc: model handle is NULL");
  const int w = Rf_asInteger(what); const long n = gprc_gpc_n(g);
  SEXP out = PROTECT(w == GPRC_GET_L ? Rf_allocMatrix(REALSXP, (int)n, (int)n) : Rf_allocVector(REALSXP, n));
  int rc = gprc_gpc_get(g, w, REAL(out));
  UNPROTECT(1);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  return out;
}

/* one pass of fit()'s loop body inside the library (gprc_fit_family, R/fit.R:113-162): c(value, par...) */
SEXP C_gprc_fit_family(SEXP id, SEXP X, SEXP y, SEXP noise, SEXP strict) {
  double par[2] = {0.0, 0.0}, value = NA_REAL; int npar = 0;
  int rc = gprc_fit_family(ctx(), Rf_asInteger(id), REAL(X), Rf_nrows(X), XLENGTH(y), REAL(y), Rf_asReal(noise),
                           Rf_asLogical(strict) ? 0 : 1, par, &npar, &value, NULL);
  if (rc) Rf_error("gprc: %s", gprc_last_error());
  SEXP out = PROTECT(Rf_allocVector(REALSXP, 1 + npar));
  REAL(out)[0] = value;
  for (int i = 0; i < npar; ++i) REAL(out)[1 + i] = par[i];
  UNPROTECT(1);
  return out;
}

/* gprc_ctx_set_option(option, value): predict path, INT8 digits / tile, ... (include/gprc.h GPRC_OPT_*) */
SEXP C_gprc_set_option(SEXP option, SEXP value) {
  if (gprc_ctx_set_option(ctx(), Rf_asInteger(option), Rf_asInteger(value)) != 0) Rf_error("gprc: %s", gprc_last_error());
  return R_NilValue;
}

static const R_CallMethodDef call_methods[] = {
    {"C_gprc_cov_matrix", (DL_FUNC)&C_gprc_cov_matrix, 3},
    {"C_gprc_gpr_fit", (DL_FUNC)&C_gprc_gpr_fit, 5},
    {"C_gprc_gpr_predict", (DL_FUNC)&C_gprc_gpr_predict, 4},
    {"C_gprc_gpr_predict_cov", (DL_FUNC)&C_gprc_gpr_predict_cov, 2},
    {"C_gprc_gpr_append", (DL_FUNC)&C_gprc_gpr_append, 3},
    {"C_gprc_gpr_get", (DL_FUNC)&C_gprc_gpr_get, 2},
    {"C_gprc_logml", (DL_FUNC)&C_gprc_logml, 4},
    {"C_gprc_logml_grad", (DL_FUNC)&C_gprc_logml_grad, 6},
    {"C_gprc_fit_family", (DL_FUNC)&C_gprc_fit_family, 5},
    {"C_gprc_set_option", (DL_FUNC)&C_gprc_set_option, 2},
    {"C_gprc_gpc_fit", (DL_FUNC)&C_gprc_gpc_fit, 6},
    {"C_gprc_gpc_predict_latent", (DL_FUNC)&C_gprc_gpc_predict_latent, 4},
    {"C_gprc_gpc_predict_class", (DL_FUNC)&C_gprc_gpc_predict_class, 2},
    {"C_gprc_gpc_get", (DL_FUNC)&C_gprc_gpc_get, 2},
    {NULL, NULL, 0}};

void R_init_gprc(DllInfo* dll) {
  R_registerRoutines(dll, NULL, call_methods, NULL, NULL);
  R_useDynamicSymbols(dll, FALSE);
}

void R_unload_gprc(DllInfo* dll) {
  (void)dll;
  if (g_ctx) { gprc_ctx_free(g_ctx); g_ctx = NULL; }
}
