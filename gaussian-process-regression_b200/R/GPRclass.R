# Host side of GPR (reference: R/GPRclass.R:116-351 of the CPU package).  Argument checks, the noise-bump retry and
# the return shapes stay in R; everything numerical is one .Call.  The plot methods of the CPU package are unchanged
# and omitted here (they only call $predict).

#' @export
GPR <- R6::R6Class("GPR",
  private = list(.X = NULL, .k = NULL, .y = NULL, .noise = NULL, .logp = NULL, .ptr = NULL,
    readonly = function(name, value, missing_value) {
      if (!missing_value) stop(sprintf("`$%s` is read only", name), call. = FALSE)
    }),
  public = list(
    initialize = function(X, y, noise = 0, k = fit(X, y, noise, cov_names)$func, cov_names = names(cov_dict)) {
      stopifnot(is.numeric(X), is.vector(y), is.numeric(y))
      stopifnot(is.numeric(noise), length(noise) == 1, noise >= 0)
      if (!is.matrix(X)) dim(X) <- c(1, length(X))
      stopifnot(length(y) == ncol(X), is.function(k))
      storage.mode(X) <- "double"
      spec <- .gprc_spec(k)
      K <- if (is.null(spec)) covariance_matrix(X, X, k) else NULL   # closure kernels: built in R as before
      tried <- noise
      for (attempt in 1:10) {                                        # schedule: noise, noise + 0.01, ..., + 0.09
        res <- .Call(C_gprc_gpr_fit, spec, X, as.double(y), as.double(tried), K)
        if (res[[3]] == 0 && is.finite(res[[2]])) {
          if (attempt > 1)
            warning(sprintf("Noise got changed to %s to avoid errors in cholesky decomposition", tried))
          break
        }
        res <- NULL
        tried <- 0.01 * attempt + noise
      }
      if (is.null(res))
        stop("Inputs lead to non positive definite covariance matrix. Try using a larger noise or a smaller lengthscale.")
      private$.X <- X; private$.y <- y; private$.k <- k
      private$.ptr <- res[[1]]; private$.noise <- tried
      private$.logp <- matrix(res[[2]], 1, 1)
    },
    predict = function(X_star, pointwise_var = TRUE) {
      stopifnot(is.numeric(X_star), length(X_star) %% nrow(private$.X) == 0)
      if (is.null(dim(X_star))) dim(X_star) <- c(nrow(private$.X), length(X_star) / nrow(private$.X))
      # a matrix with the wrong number of rows passes the length check above; the reference then fails inside
      # covariance_matrix (R/GPRclass.R:356) -- fail here, before the library reads nrow(X) * m doubles
      if (nrow(X_star) != nrow(private$.X)) stop("non-conformable arrays")
      storage.mode(X_star) <- "double"
      spec <- .gprc_spec(private$.k)
      if (pointwise_var) {
        if (!is.null(spec)) return(.Call(C_gprc_gpr_predict, private$.ptr, X_star, NULL, NULL))
        Ks <- covariance_matrix(private$.X, X_star, private$.k)
        return(.Call(C_gprc_gpr_predict, private$.ptr, NULL, Ks, as.double(private$.k(X_star, X_star))))
      }
      if (!is.null(spec)) return(.Call(C_gprc_gpr_predict_cov, private$.ptr, X_star))
      Ks <- covariance_matrix(private$.X, X_star, private$.k)
      v <- .Call(C_gprc_gpr_get, private$.ptr, 2L) %*% Ks            # L^-1 K_star
      list(t(Ks) %*% self$alpha, covariance_matrix(X_star, X_star, private$.k) - t(v) %*% v)
    },
    # append training points in place: afterwards the model is GPR$new(cbind(X, X_new), c(y, y_new), noise, k) with
    # this model's noise and kernel.  Built-in kernels extend the Cholesky factor on the device; a matrix that is not
    # positive definite with this noise, or a closure kernel, takes the constructor's path (noise-bump loop included).
    add_points = function(X_new, y_new) {
      stopifnot(is.numeric(X_new), length(X_new) %% nrow(private$.X) == 0)
      if (is.null(dim(X_new))) dim(X_new) <- c(nrow(private$.X), length(X_new) / nrow(private$.X))
      if (nrow(X_new) != nrow(private$.X)) stop("non-conformable arrays")
      stopifnot(is.numeric(y_new), is.vector(y_new), length(y_new) == ncol(X_new))
      if (ncol(X_new) == 0) return(invisible(self))
      storage.mode(X_new) <- "double"
      X <- cbind(private$.X, X_new); y <- c(private$.y, y_new)
      if (!is.null(.gprc_spec(private$.k))) {
        res <- .Call(C_gprc_gpr_append, private$.ptr, X_new, as.double(y_new))   # list(logp, info)
        if (res[[2]] == 0 && is.finite(res[[1]])) {
          private$.X <- X; private$.y <- y; private$.logp <- matrix(res[[1]], 1, 1)
          return(invisible(self))
        }
      }
      fresh <- GPR$new(X, y, private$.noise, private$.k)$.__enclos_env__$private
      private$.X <- fresh$.X; private$.y <- fresh$.y; private$.ptr <- fresh$.ptr
      private$.noise <- fresh$.noise; private$.logp <- fresh$.logp
      invisible(self)
    }
  ),
  active = list(
    X = function(value) { private$readonly("X", value, missing(value)); private$.X },
    k = function(value) { private$readonly("k", value, missing(value)); private$.k },
    y = function(value) { private$readonly("y", value, missing(value)); private$.y },
    noise = function(value) { private$readonly("noise", value, missing(value)); private$.noise },
    logp = function(value) { private$readonly("logp", value, missing(value)); private$.logp },
    # the factor and alpha stay on the device; they are downloaded when somebody asks for them
    L = function(value) { private$readonly("L", value, missing(value)); .Call(C_gprc_gpr_get, private$.ptr, 0L) },
    alpha = function(value) { private$readonly("alpha", value, missing(value)); .Call(C_gprc_gpr_get, private$.ptr, 1L) }
  )
)

.gpr_subclass <- function(name, make_kernel) {
  R6::R6Class(paste0("GPR.", name), inherit = GPR,
    public = list(initialize = function(X, y, noise, ...) super$initialize(X, y, noise, make_kernel(X, y, noise, ...))))
}
.par_of <- function(X, y, noise, name) fit(X, y, noise, name)$par

#' @export
GPR.constant <- .gpr_subclass("constant", function(X, y, noise, c = .par_of(X, y, noise, "constant")) {
  stopifnot(is.numeric(c), c > 0); cov_func(constant, c = c) })
#' @export
GPR.linear <- .gpr_subclass("linear", function(X, y, noise, sigma = .par_of(X, y, noise, "linear")) {
  stopifnot(length(sigma) == NROW(if (is.matrix(X)) X else matrix(X, 1))); cov_func(linear, sigma = sigma) })
#' @export
GPR.polynomial <- .gpr_subclass("polynomial", function(X, y, noise, sigma, p) {
  if (missing(sigma) || missing(p)) { par <- .par_of(X, y, noise, "polynomial")
    if (missing(sigma)) sigma <- par[[1]]; if (missing(p)) p <- par[[2]] }
  stopifnot(length(sigma) == 1, length(p) == 1); cov_func(polynomial, sigma = sigma, p = p) })
#' @export
GPR.sqrexp <- .gpr_subclass("sqrexp", function(X, y, noise, l = .par_of(X, y, noise, "sqrexp")) {
  stopifnot(length(l) == 1); cov_func(sqrexp, l = l) })
#' @export
GPR.gammaexp <- .gpr_subclass("gammaexp", function(X, y, noise, gamma, l) {   # par[[1]] -> gamma, par[[2]] -> l (sic)
  if (missing(gamma) || missing(l)) { par <- .par_of(X, y, noise, "gammaexp")
    if (missing(gamma)) gamma <- par[[1]]; if (missing(l)) l <- par[[2]] }
  stopifnot(length(gamma) == 1, length(l) == 1); cov_func(gammaexp, l = l, gamma = gamma) })
#' @export
GPR.rationalquadratic <- .gpr_subclass("rationalquadratic", function(X, y, noise, alpha, l) {  # par[[1]] -> alpha (sic)
  if (missing(alpha) || missing(l)) { par <- .par_of(X, y, noise, "rationalquadratic")
    if (missing(alpha)) alpha <- par[[1]]; if (missing(l)) l <- par[[2]] }
  stopifnot(length(alpha) == 1, length(l) == 1); cov_func(rationalquadratic, l = l, alpha = alpha) })

# covariance_matrix(A, B, k): device build for tagged kernels, the CPU package's outer() gather otherwise
covariance_matrix <- function(A, B, covariance_function) {
  spec <- .gprc_spec(covariance_function)
  if (!is.null(spec)) {
    storage.mode(A) <- "double"; storage.mode(B) <- "double"
    return(.Call(C_gprc_cov_matrix, spec, A, B))
  }
  outer(seq_len(ncol(A)), seq_len(ncol(B)),
        function(i, j) covariance_function(A[, i, drop = FALSE], B[, j, drop = FALSE]))
}

#' @export
cov_func <- function(func, ...) {
  force(func)
  .gprc_tag(function(x, y) func(x, y, ...), func, list(...))
}
# constant / linear / polynomial / sqrexp / gammaexp / rationalquadratic (S3 generics with .matrix and .numeric
# methods), multivariate_normal and expand_range are kept verbatim from the CPU package: they are user-callable R
# functions, not part of the accelerated path.
