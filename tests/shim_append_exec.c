/* shim_append_exec.c -- EXECUTES C_gprc_gpr_append of src/gprc_shim.c (the `.Call` behind GPR$add_points) against libgprc
 * on a GPU, with the miniature R runtime of tests/stubs/mini_r.c standing in for R:
 *   - two known answers of the reference's tests/testthat/test-gpr.R (constant and sqrexp), reached by fitting the first
 *     point and appending the second, tolerance 1.5e-8 as expect_equivalent;
 *   - the return shape list(logp, info) and the logp of a direct fit of both points;
 *   - info > 0 (constant kernel, noise 0: the Schur complement is exactly 0): the model predicts as before;
 *   - a matrix with the wrong number of rows: "non-conformable arrays" raised from shim level.
 *   gcc -std=c11 -Itests/stubs -Iinclude src/gprc_shim.c tests/stubs/mini_r.c tests/shim_append_exec.c -L<pkg> -lgprc -lm */
#include <math.h>
#include <setjmp.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "mini_r.h"
#include "gprc.h"

void R_init_gprc(DllInfo*);
void R_unload_gprc(DllInfo*);

typedef SEXP (*F3)(SEXP, SEXP, SEXP);
typedef SEXP (*F4)(SEXP, SEXP, SEXP, SEXP);
typedef SEXP (*F5)(SEXP, SEXP, SEXP, SEXP, SEXP);

static int failures = 0;
static void expect(int cond, const char* what) {
  printf("%-78s %s\n", what, cond ? "ok" : "FAIL");
  if (!cond) ++failures;
}
static int near(double a, double b, double tol) { return fabs(a - b) <= tol; }

static SEXP spec(int id, const char* p1, double v1) {
  const char* names[2] = {"id", p1};
  SEXP vals[2] = {Rf_ScalarInteger(id), Rf_ScalarReal(v1)};
  return mini_r_named_list(2, names, vals);
}
static void* must(const char* name, int nargs) {
  void* f = (void*)mini_r_lookup(name, nargs);
  if (!f) {
    printf("routine %s with %d arguments is not registered\n", name, nargs);
    exit(2);
  }
  return f;
}

/* GPR$new(x0, y0, noise, k)$add_points(x1, y1)$predict(xs) */
static void known_answer(F5 fit, F3 append, F4 predict, SEXP k, double x0, double x1, double y0, double y1, double noise,
                         double xs, double mean, double var, const char* what) {
  SEXP r = fit(k, mini_r_matrix(1, 1, &x0), mini_r_vector(1, &y0), Rf_ScalarReal(noise), R_NilValue);
  SEXP a = append(VECTOR_ELT(r, 0), mini_r_matrix(1, 1, &x1), mini_r_vector(1, &y1));
  SEXP p = predict(VECTOR_ELT(r, 0), mini_r_matrix(1, 1, &xs), R_NilValue, R_NilValue);
  /* the logp of fitting both points at once */
  const double X[2] = {x0, x1}, y[2] = {y0, y1};
  SEXP both = fit(k, mini_r_matrix(1, 2, X), mini_r_vector(2, y), Rf_ScalarReal(noise), R_NilValue);
  const double lp = Rf_asReal(VECTOR_ELT(a, 0)), lp2 = Rf_asReal(VECTOR_ELT(both, 1));
  char buf[160];
  snprintf(buf, sizeof buf, "%s: list(logp, info 0), mean %.12f var %.12f", what, REAL(p)[0], REAL(p)[1]);
  expect(Rf_length(a) == 2 && Rf_asReal(VECTOR_ELT(a, 1)) == 0.0 && near(REAL(p)[0], mean, 1.5e-8) &&
             near(REAL(p)[1], var, 1.5e-8),
         buf);
  snprintf(buf, sizeof buf, "%s: logp %.12f equals the fit of both points", what, lp);
  expect(near(lp, lp2, 1e-12 * fabs(lp2)), buf);
}

int main(void) {
  mini_r_init();
  R_init_gprc(NULL);
  F5 fit = (F5)must("C_gprc_gpr_fit", 5);
  F3 append = (F3)must("C_gprc_gpr_append", 3);
  F4 predict = (F4)must("C_gprc_gpr_predict", 4);
  expect(mini_r_lookup("C_gprc_gpr_append", 2) == NULL, "a call with the wrong number of arguments is not resolved");

  /* ---- tests/testthat/test-gpr.R:12-15 and 23-27, one point at a time ---- */
  const double e1 = exp(-1.0), e2 = exp(-2.0), e3 = exp(-3.0), e4 = exp(-4.0);
  known_answer(fit, append, predict, spec(GPRC_CONSTANT, "c", 1.0), 1, 2, 1, 3, 1.0, 3.0, 4.0 / 3, 1.0 / 3,
               "test-gpr.R:12-15 constant, appended");
  known_answer(fit, append, predict, spec(GPRC_SQREXP, "l", 1.0), 1, 2, 0, 1, 1.0, 0.0, (2 * e2 - e1) / (4 - e1),
               1 - (2 * e1 - 2 * e3 + 2 * e4) / (4 - e1), "test-gpr.R:23-27 sqrexp, appended");
  expect(mini_r_protect_depth() == 0, "PROTECT / UNPROTECT balanced after the append calls");

  /* ---- info > 0: constant kernel c = 1, noise 0; S = 1 - 1 * 1^-1 * 1 = 0 ---- */
  {
    const double x0 = 1.0, y0 = 2.0, x1 = 5.0, y1 = -1.0, xs[2] = {0.0, 3.0};
    SEXP r = fit(spec(GPRC_CONSTANT, "c", 1.0), mini_r_matrix(1, 1, &x0), mini_r_vector(1, &y0), Rf_ScalarReal(0.0),
                 R_NilValue);
    SEXP ptr = VECTOR_ELT(r, 0);
    SEXP before = predict(ptr, mini_r_matrix(1, 2, xs), R_NilValue, R_NilValue);
    double b[4];
    memcpy(b, REAL(before), sizeof b);
    SEXP a = append(ptr, mini_r_matrix(1, 1, &x1), mini_r_vector(1, &y1));
    SEXP after = predict(ptr, mini_r_matrix(1, 2, xs), R_NilValue, R_NilValue);
    expect(Rf_asReal(VECTOR_ELT(a, 1)) == 2.0, "not positive definite: info is the 1-based failing row (2)");
    expect(memcmp(b, REAL(after), sizeof b) == 0, "... and the model predicts bit for bit as before");
  }

  /* ---- X_new with the wrong number of rows: raised from the shim, before the library reads anything ---- */
  {
    const double x0 = 0.5, y0 = 1.0, bad[2] = {1.0, 2.0}, yb = 0.0;
    SEXP r = fit(spec(GPRC_SQREXP, "l", 1.0), mini_r_matrix(1, 1, &x0), mini_r_vector(1, &y0), Rf_ScalarReal(0.1),
                 R_NilValue);
    jmp_buf jb;
    mini_r_handler = &jb;
    int raised = 0;
    if (setjmp(jb) == 0) append(VECTOR_ELT(r, 0), mini_r_matrix(2, 1, bad), mini_r_vector(1, &yb));
    else raised = 1;
    mini_r_handler = NULL;
    expect(raised && strstr(mini_r_last_error, "non-conformable") != NULL, "nrow(X_new) != nrow(X): non-conformable arrays");
  }

  const int freed = mini_r_gc();
  expect(freed >= 5 && mini_r_gc() == 0, "finalizers ran once for every model handle");
  R_unload_gprc(NULL);
  printf(failures ? "%d FAILURES\n" : "ALL OK (%d)\n", failures);
  return failures ? 1 : 0;
}
