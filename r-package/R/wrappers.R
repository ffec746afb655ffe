# User-facing samplers.  Argument lists, defaults and the returned list are those of bmmmcmc 1.0
# (reference R/utils.R:23-107); the initial state is drawn here with R's RNG exactly as the reference
# does, then handed to the CUDA back end through the Rcpp host (src/host.cpp).
#
# Back-end settings that have no place in the reference's argument lists are R options:
#   options(bmm.seed = NULL)              Philox key; NULL draws it from R's RNG (set.seed() reproducible)
#   options(bmm.device = 0L)              CUDA device
#   options(bmm.stephens_fixed = FALSE)   TRUE: corrected Stephens relabelling (inverse permutation for the
#                                         column re-ordering, log p in the online cost, running-mean Q)
#                                         instead of the reference's (stephens.cpp:56,79,85,92)

.bmm_defaults <- function(nsamples, burnin, burnrelabel, alpha, clamp = TRUE) {
    if (is.null(burnin)) burnin <- round(0.1 * nsamples)
    if (clamp && burnrelabel > burnin) burnrelabel <- round(0.1 * burnin)
    list(burnin = burnin, burnrelabel = burnrelabel, alpha = if (is.null(alpha)) 0 else alpha)
}

.bmm_initial_weights <- function(K) {
    w <- exp(stats::runif(K))
    w / sum(w)
}

gibbs_dp <- function(data, nsamples, alpha = NULL, a = 1, b = 1, beta = 0.5, gamma = 0.5,
                     burnin = NULL, relabel = FALSE, burnrelabel = 50, maxK = 30, debug = FALSE) {
    d <- .bmm_defaults(nsamples, burnin, burnrelabel, alpha)
    collapsed_gibbs_dp_cpp(data, nsamples, d$alpha, beta, gamma, a, b, d$burnin, relabel,
                           d$burnrelabel, maxK, debug)
}

gibbs_collapsed <- function(data, nsamples, K, alpha = NULL, beta = 0.5, gamma = 0.5, a = 1, b = 1,
                            burnin = NULL, relabel = FALSE, burnrelabel = 50, debug = FALSE) {
    d <- .bmm_defaults(nsamples, burnin, burnrelabel, alpha)
    start <- sample(1:K, nrow(data), replace = TRUE)
    collapsed_gibbs_cpp(data, start, nsamples, K, d$alpha, beta, gamma, a, b, d$burnin, relabel,
                        d$burnrelabel, debug)
}

gibbs_full <- function(data, nsamples, K, alpha = NULL, beta = 0.5, gamma = 0.5, a = 1, b = 1,
                       burnin = NULL, relabel = FALSE, burnrelabel = 50, debug = FALSE) {
    d <- .bmm_defaults(nsamples, burnin, burnrelabel, alpha)
    w0 <- .bmm_initial_weights(K)
    theta0 <- matrix(stats::runif(K * ncol(data)), nrow = K, ncol = ncol(data))
    gibbs_cpp(data, w0, theta0, nsamples, K, d$alpha, beta, gamma, a, b, d$burnin, relabel,
              d$burnrelabel, debug)
}

# The reference wrapper does not clamp burnrelabel for this sampler (R/utils.R:95-107); kept.
gibbs_stickbreaking <- function(data, nsamples, maxK, alpha = NULL, beta = 0.5, gamma = 0.5, a = 1, b = 1,
                                burnin = NULL, relabel = FALSE, burnrelabel = 50, debug = FALSE) {
    d <- .bmm_defaults(nsamples, burnin, burnrelabel, alpha, clamp = FALSE)
    w0 <- .bmm_initial_weights(maxK)
    theta0 <- matrix(stats::runif(maxK * ncol(data)), nrow = maxK, ncol = ncol(data))
    gibbs_stickbreaking_cpp(data, w0, theta0, nsamples, maxK, d$alpha, beta, gamma, a, b, d$burnin,
                            relabel, d$burnrelabel, debug)
}

#' Posterior predictive distribution of new observations
#'
#' Not in the reference (its TODO file lists "Implement predictive distribution"): for every row of
#' \code{newdata}, the log of the posterior predictive probability averaged over the kept draws of an
#' uncollapsed sampler, and the cluster responsibilities averaged over the draws.
#'
#' @param obj The list returned by \code{gibbs_full} or \code{gibbs_stickbreaking}.
#' @param newdata An M x P 0/1 integer matrix.
#' @return A list with \code{log_pred} (length M) and \code{membership} (M x K).
#' @export
predict_gibbs <- function(obj, newdata) {
    if (is.null(obj$pi)) stop("predict_gibbs needs the pi history of gibbs_full / gibbs_stickbreaking")
    newdata <- as.matrix(newdata)
    storage.mode(newdata) <- "integer"
    predictive_cpp(newdata, obj$theta, obj$pi)
}

#' WAIC of a fitted model
#'
#' Not in the reference: the widely applicable information criterion (Watanabe 2010) of an uncollapsed fit, computed on
#' the GPU, in the layout of \code{loo::waic}, to compare fits at several K (lower \code{waic} is better).
#'
#' @param obj The list returned by \code{gibbs_full} or \code{gibbs_stickbreaking}.
#' @param data The N x P 0/1 matrix the model was fitted to.
#' @return A list with \code{estimates} (rows elpd_waic, p_waic, waic; columns Estimate, SE), \code{pointwise}
#'   (N x 3, the same three columns) and \code{loglik}, the observed-data log-likelihood of every kept draw.
#' @export
waic_gibbs <- function(obj, data) {
    if (is.null(obj$pi)) stop("waic_gibbs needs the pi history of gibbs_full / gibbs_stickbreaking")
    data <- as.matrix(data)
    storage.mode(data) <- "integer"
    r <- waic_cpp(data, obj$theta, obj$pi)
    dimnames(r$estimates) <- list(c("elpd_waic", "p_waic", "waic"), c("Estimate", "SE"))
    colnames(r$pointwise) <- c("elpd_waic", "p_waic", "waic")
    r
}

#' PSIS-LOO of a fitted model
#'
#' Not in the reference: Pareto-smoothed importance-sampling leave-one-out cross-validation (Vehtari, Gelman & Gabry
#' 2017) of an uncollapsed fit, computed on the GPU, in the layout of \code{loo::loo} (lower \code{looic} is better).
#' Observations with \code{pareto_k} above 0.7 have an unreliable estimate.  \code{mcse_elpd_loo} is not computed:
#' current \code{loo} estimates it from random gamma draws, which cannot be reproduced.
#'
#' @param obj The list returned by \code{gibbs_full} or \code{gibbs_stickbreaking}.
#' @param data The N x P 0/1 matrix the model was fitted to.
#' @param r_eff Relative efficiency of the draws, one value or one per observation (e.g. from \code{loo::relative_eff}).
#' @return A list with \code{estimates} (rows elpd_loo, p_loo, looic; columns Estimate, SE), \code{pointwise} (N x 4:
#'   elpd_loo, p_loo, looic, influence_pareto_k) and \code{diagnostics} (\code{pareto_k}, \code{n_eff}).
#' @export
loo_gibbs <- function(obj, data, r_eff = 1) {
    if (is.null(obj$pi)) stop("loo_gibbs needs the pi history of gibbs_full / gibbs_stickbreaking")
    data <- as.matrix(data)
    storage.mode(data) <- "integer"
    r <- loo_cpp(data, obj$theta, obj$pi, as.numeric(r_eff))
    dimnames(r$estimates) <- list(c("elpd_loo", "p_loo", "looic"), c("Estimate", "SE"))
    colnames(r$pointwise) <- c("elpd_loo", "p_loo", "looic", "influence_pareto_k")
    r
}

#' Log-likelihood matrix of a fitted model
#'
#' Not in the reference: the S x N matrix of log p(x_i | draw s) over the kept draws, computed on the GPU, as
#' \code{loo::loo()} and \code{loo::waic()} take it.
#'
#' @param obj The list returned by \code{gibbs_full} or \code{gibbs_stickbreaking}.
#' @param data The N x P 0/1 matrix the model was fitted to.
#' @return An S x N numeric matrix.
#' @export
log_lik_gibbs <- function(obj, data) {
    if (is.null(obj$pi)) stop("log_lik_gibbs needs the pi history of gibbs_full / gibbs_stickbreaking")
    data <- as.matrix(data)
    storage.mode(data) <- "integer"
    log_lik_cpp(data, obj$theta, obj$pi)
}
