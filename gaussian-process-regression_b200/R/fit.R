# Host side of fit() (reference: R/fit.R of the CPU package).  cov_dict / cov_df, optim_until_error and the optimiser
# set-up are unchanged R code; only the two objective closures change: dens() and dens_deriv() become one .Call each.

.dens_device <- function(X, y, noise, name, strict = TRUE) {
  force(X); force(y); force(noise); force(name)
  function(v) {
    spec <- c(list(id = .gprc_ids[[name]]), setNames(as.list(as.double(v)), .gprc_formals(name)))
    r <- .Call(C_gprc_logml, spec, X, as.double(y), as.double(noise))   # c(logp, min leading-minor log det, info)
    # stopifnot(min(sapply(1:n, function(i) det(...[1:i, 1:i]))) > 0): det() = exp(log-modulus), 0 below log(2^-1075)
    if (r[3] != 0 || !is.finite(r[1]) || (strict && !(exp(r[2]) > 0)))
      stop("covariance matrix is not (numerically) positive definite")
    matrix(r[1], 1, 1)
  }
}

.dens_deriv_device <- function(X, y, noise, name, formula = 0L) {
  function(v) {
    spec <- c(list(id = .gprc_ids[[name]]), setNames(as.list(as.double(v)), .gprc_formals(name)))
    .Call(C_gprc_logml_grad, spec, X, as.double(y), as.double(noise), as.integer(formula), length(v))
  }
}

.gprc_formals <- function(name)
  setdiff(names(formals(get(paste0(name, ".matrix"), envir = asNamespace("gprc")))), c("x", "y"))

# options(gprc.fit_engine = "library"): the same optimiser trajectories, run inside libgprc (gprc_fit_family: Brent_fmin,
# vmmin and optim_until_error restated in C++, X and y uploaded once); default "R": optim() drives, one .Call per
# evaluation.  Both give the same par / value.
#' @export
fit <- function(X, y, noise, cov_names = as.list(cov_df$name)) {
  if (!is.matrix(X)) dim(X) <- c(1, length(X))
  storage.mode(X) <- "double"
  in_library <- identical(getOption("gprc.fit_engine", "R"), "library")
  results <- lapply(cov_names, function(cov) {
    if (in_library) {
      r <- .Call(C_gprc_fit_family, .gprc_ids[[cov]], X, as.double(y), as.double(noise), TRUE)
      return(list(par = r[-1], value = r[1]))
    }
    start <- cov_df[cov, ]$start[[1]]
    dens <- .dens_device(X, y, noise, cov)
    if (cov == "polynomial") {                       # degrees 1..10, Brent over sigma in [0, 5]
      runs <- lapply(1:10, function(p) optim_until_error(start[1], function(sig) dens(c(sig, p)), method = "Brent",
                                                         lower = 0, upper = 5, control = list(fnscale = -1)))
      best <- which.max(vapply(runs, function(q) as.numeric(q$value), numeric(1)))
      return(list(par = c(runs[[best]]$par, best), value = as.numeric(runs[[best]]$value)))
    }
    args <- list(start, dens, control = list(fnscale = -1))
    if (cov %in% c("sqrexp", "gammaexp", "rationalquadratic")) args$gr <- .dens_deriv_device(X, y, noise, cov)
    args <- c(args, if (length(start) == 1) list(method = "Brent", lower = 0, upper = 10) else list(method = "BFGS"))
    do.call(optim_until_error, args)
  })
  score <- vapply(results, function(r) as.numeric(r$value), numeric(1))
  win <- which.max(score)
  name <- cov_names[[win]]; par <- results[[win]]$par
  message(sprintf("The optimal covariance function is %s, with parameters %s", name, paste(par, collapse = ", ")))
  list(par = par, cov = name, score = score,
       func = do.call(cov_func, c(list(cov_df[name, ]$func[[1]]), as.list(par))))
}
