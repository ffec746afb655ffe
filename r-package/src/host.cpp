// Rcpp host of the B200 back end: the four sampler entry points the R wrappers call, with the argument
// lists of the reference's .Call symbols (/root/reference/src/RcppExports.cpp:11-135), forwarding to the
// C ABI of include/bmm_capi.h.  This file only allocates the returned R objects (same names, shapes and
// storage modes as full_gibbs.cpp:233-248, stickbreaking.cpp:238-254, collapsed_gibbs.cpp:229-243,
// collapsed_gibbs_dp.cpp:285-299) and turns a non-zero return code into an R error.
//
// The build image has no R / Rcpp: tests/test_rhost.py compiles this file, unmodified, against the Rcpp stand-in of
// oracle/shim/ and checks on the GPU that every element of the returned lists equals the ctypes path's.  Everything
// below the C ABI is exercised through the same entry points by tests/test_gpu_parity.py.
#include <cmath>

#include <Rcpp.h>

#include "bmm_capi.h"

using namespace Rcpp;

namespace {

struct RunSpec {
    int sampler;           // BMM_SAMPLER_*
    bool has_pi;           // full / stick-breaking return `pi`
    int K;                 // K or maxK
};

// chains / seed / device are taken from R options so the exported signatures stay the reference's:
//   options(bmm.chains = 1L, bmm.seed = NULL, bmm.device = 0L, bmm.stephens_fixed = FALSE)
// bmm.stephens_fixed = TRUE selects BMM_FLAG_STEPHENS_FIXED (corrected relabelling, not the reference's).
// bmm.seed = NULL draws the Philox key from R's RNG, so set.seed() keeps runs reproducible.
unsigned long long philox_seed() {
    SEXP s = Rf_GetOption1(Rf_install("bmm.seed"));
    if (!Rf_isNull(s)) return (unsigned long long)Rf_asReal(s);
    const double hi = floor(R::unif_rand() * 4294967296.0), lo = floor(R::unif_rand() * 4294967296.0);
    return ((unsigned long long)hi << 32) | (unsigned long long)lo;
}

int int_option(const char *name, int dflt) {
    SEXP s = Rf_GetOption1(Rf_install(name));
    return Rf_isNull(s) ? dflt : Rf_asInteger(s);
}

List run(const RunSpec &spec, IntegerMatrix df, const double *init_pi, const double *init_theta, const int *init_z,
         int nsamples, double alpha, double beta, double gamma, double a, double b, int burnin, bool relabel,
         int burnrelabel, bool debug) {
    const int N = df.nrow(), P = df.ncol(), K = spec.K, S = nsamples - burnin;
    if (S <= 0) stop("burnin must be smaller than nsamples");
    bmm_args args = {};
    args.X = df.begin();            // IntegerMatrix storage is already N x P int32 column-major
    args.N = N; args.P = P; args.nsamples = nsamples; args.K = K;
    args.alpha = alpha; args.beta = beta; args.gamma = gamma; args.a = a; args.b = b;
    args.burnin = burnin; args.relabel = relabel; args.burnrelabel = burnrelabel; args.debug = debug;
    args.n_chains = 1; args.seed = philox_seed(); args.precision = BMM_FP64;
    args.device = int_option("bmm.device", 0);
    if (int_option("bmm.stephens_fixed", 0)) args.flags |= BMM_FLAG_STEPHENS_FIXED;
    bmm_init init = {init_pi, init_theta, init_z};

    NumericMatrix pi(spec.has_pi ? S : 0, spec.has_pi ? K : 0);
    NumericMatrix alpha_out(S, 1);                 // arma::vec wraps as an S x 1 matrix in the reference
    IntegerMatrix perms(S, K), z(S, N);
    NumericVector theta(Dimension(K, P, S));
    IntegerMatrix z_orig(relabel ? S : 0, relabel ? N : 0);
    NumericVector theta_orig = relabel ? NumericVector(Dimension(K, P, S)) : NumericVector(0);

    bmm_out out = {};
    out.pi = spec.has_pi ? pi.begin() : nullptr;
    out.alpha = alpha_out.begin();
    out.permutations = perms.begin();
    out.z = z.begin();
    out.theta = theta.begin();
    if (relabel) { out.z_original = z_orig.begin(); out.theta_original = theta_orig.begin(); }

    int rc;
    switch (spec.sampler) {
        case BMM_SAMPLER_FULL: rc = bmm_gibbs_full(&args, &init, &out); break;
        case BMM_SAMPLER_STICKBREAKING: rc = bmm_gibbs_stickbreaking(&args, &init, &out); break;
        case BMM_SAMPLER_COLLAPSED: rc = bmm_gibbs_collapsed(&args, &init, &out); break;
        default: rc = bmm_gibbs_dp(&args, &out); break;
    }
    if (rc != BMM_OK) stop(bmm_last_error());

    List ret;
    if (spec.has_pi) ret["pi"] = pi;
    ret["alpha"] = alpha_out;
    ret["permutations"] = perms;
    ret["z"] = z;
    ret["theta"] = theta;
    if (relabel) { ret["z_original"] = z_orig; ret["theta_original"] = theta_orig; }
    return ret;
}

}  // namespace

// [[Rcpp::export]]
List gibbs_cpp(IntegerMatrix df, NumericVector initialPi, NumericMatrix initialTheta, int nsamples, int K,
               double alpha, double beta, double gamma, double a, double b, int burnin, bool relabel,
               int burnrelabel, bool debug) {
    return run({BMM_SAMPLER_FULL, true, K}, df, initialPi.begin(), initialTheta.begin(), nullptr, nsamples, alpha,
               beta, gamma, a, b, burnin, relabel, burnrelabel, debug);
}

// [[Rcpp::export]]
List gibbs_stickbreaking_cpp(IntegerMatrix df, NumericVector initialPi, NumericMatrix initialTheta, int nsamples,
                             int maxK, double alpha, double beta, double gamma, double a, double b, int burnin,
                             bool relabel, int burnrelabel, bool debug) {
    return run({BMM_SAMPLER_STICKBREAKING, true, maxK}, df, initialPi.begin(), initialTheta.begin(), nullptr,
               nsamples, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug);
}

// [[Rcpp::export]]
List collapsed_gibbs_cpp(IntegerMatrix df, IntegerVector initialK, int nsamples, int K, double alpha, double beta,
                         double gamma, double a, double b, int burnin, bool relabel, int burnrelabel, bool debug) {
    return run({BMM_SAMPLER_COLLAPSED, false, K}, df, nullptr, nullptr, initialK.begin(), nsamples, alpha, beta,
               gamma, a, b, burnin, relabel, burnrelabel, debug);
}

// [[Rcpp::export]]
List collapsed_gibbs_dp_cpp(IntegerMatrix df, int nsamples, double alpha, double beta, double gamma, double a,
                            double b, int burnin, bool relabel, int burnrelabel, int maxK, bool debug) {
    return run({BMM_SAMPLER_DP, false, maxK}, df, nullptr, nullptr, nullptr, nsamples, alpha, beta, gamma, a, b,
               burnin, relabel, burnrelabel, debug);
}

// [[Rcpp::export]]
NumericMatrix my_stephens_batch(NumericVector p, bool debug) {
    IntegerVector dim = p.attr("dim");
    if (dim.size() != 3) stop("p must be an N x K x M array");
    NumericMatrix q(dim[0], dim[1]);
    if (bmm_stephens_batch(dim[0], dim[1], dim[2], p.begin(), q.begin(), nullptr) != BMM_OK) stop(bmm_last_error());
    return q;
}

// [[Rcpp::export]]
IntegerMatrix my_lpsolve(NumericMatrix cost) {
    const int K = cost.nrow();
    if (cost.ncol() != K) stop("cost must be square");
    IntegerMatrix sol(K, K);
    if (bmm_assign(K, 1, cost.begin(), sol.begin()) != BMM_OK) stop(bmm_last_error());
    return sol;
}

// rdirichlet_cpp (reference: src/full_gibbs.cpp:10-27, registered as _bmmmcmc_rdirichlet_cpp,
// src/RcppExports.cpp:56-64): one Dirichlet(alpha_m) draw as a column vector.  The Philox key comes from
// options(bmm.seed) or, when that is NULL, from R's RNG, so set.seed() keeps it reproducible.
// [[Rcpp::export]]
NumericMatrix rdirichlet_cpp(NumericVector alpha_m) {
    const int K = alpha_m.size();
    if (K < 1) stop("alpha_m must not be empty");
    NumericMatrix out(K, 1);                       // arma::vec wraps as a K x 1 matrix in the reference
    if (bmm_rdirichlet(K, alpha_m.begin(), philox_seed(), out.begin()) != BMM_OK) stop(bmm_last_error());
    return out;
}

// WAIC of a fitted model (no reference counterpart; the layout of loo::waic): estimates 3 x 2 (rows elpd_waic, p_waic, waic;
// columns Estimate, SE = sqrt(N var(pointwise))), pointwise N x 3 (same columns order as the estimate rows), loglik[S].
// theta: K x P x S array and pi: S x K matrix as gibbs_full / gibbs_stickbreaking return them; data: the N x P 0/1 matrix.
// [[Rcpp::export]]
List waic_cpp(IntegerMatrix data, NumericVector theta, NumericMatrix pi) {
    IntegerVector dim = theta.attr("dim");
    if (dim.size() != 3) stop("theta must be a K x P x S array");
    const int K = dim[0], P = dim[1], S = dim[2], N = data.nrow();
    if (data.ncol() != P || pi.nrow() != S || pi.ncol() != K) stop("data / theta / pi dimensions do not match");
    if (S < 2) stop("waic needs at least 2 draws");
    NumericVector loglik(S), lppd(N), pw(N);
    if (bmm_waic(data.begin(), N, P, K, S, 1, theta.begin(), pi.begin(), 0u, 0, loglik.begin(), lppd.begin(), pw.begin(),
                 nullptr, nullptr) != BMM_OK)
        stop(bmm_last_error());
    NumericMatrix pointwise(N, 3), estimates(3, 2);
    for (int i = 0; i < N; ++i) {
        pointwise(i, 0) = lppd[i] - pw[i];
        pointwise(i, 1) = pw[i];
        pointwise(i, 2) = -2.0 * (lppd[i] - pw[i]);
    }
    for (int j = 0; j < 3; ++j) {
        double sum = 0.0, ss = 0.0;
        for (int i = 0; i < N; ++i) sum += pointwise(i, j);
        const double mean = sum / N;
        for (int i = 0; i < N; ++i) ss += (pointwise(i, j) - mean) * (pointwise(i, j) - mean);
        estimates(j, 0) = sum;
        estimates(j, 1) = N > 1 ? std::sqrt(N * (ss / (N - 1))) : NAN;
    }
    return List::create(Named("estimates") = estimates, Named("pointwise") = pointwise, Named("loglik") = loglik);
}

// PSIS-LOO of a fitted model (no reference counterpart; the layout of loo::loo without mcse_elpd_loo, which current loo
// estimates by random gamma draws that cannot be reproduced): estimates 3 x 2 (rows elpd_loo, p_loo, looic; columns
// Estimate, SE = sqrt(N var(pointwise))), pointwise N x 4 (elpd_loo, p_loo, looic, influence_pareto_k), diagnostics =
// list(pareto_k, n_eff).  r_eff: one value, or one per observation (> 0).  theta, pi and data as waic_cpp.
// [[Rcpp::export]]
List loo_cpp(IntegerMatrix data, NumericVector theta, NumericMatrix pi, NumericVector r_eff) {
    IntegerVector dim = theta.attr("dim");
    if (dim.size() != 3) stop("theta must be a K x P x S array");
    const int K = dim[0], P = dim[1], S = dim[2], N = data.nrow();
    if (data.ncol() != P || pi.nrow() != S || pi.ncol() != K) stop("data / theta / pi dimensions do not match");
    if (S < 2) stop("loo needs at least 2 draws");
    if (r_eff.size() != 1 && r_eff.size() != N) stop("r_eff must have length 1 or one value per observation");
    NumericVector re(N), elpd(N), lpd(N), k(N), n_eff(N);
    for (int i = 0; i < N; ++i) {
        re[i] = r_eff[r_eff.size() == 1 ? 0 : i];
        if (!(re[i] > 0.0) || !std::isfinite(re[i])) stop("r_eff must be finite and > 0");
    }
    if (bmm_loo(data.begin(), N, P, K, S, 1, theta.begin(), pi.begin(), re.begin(), 0u, 0, elpd.begin(), lpd.begin(),
                k.begin(), n_eff.begin()) != BMM_OK)
        stop(bmm_last_error());
    NumericMatrix pointwise(N, 4), estimates(3, 2);
    for (int i = 0; i < N; ++i) {
        pointwise(i, 0) = elpd[i];
        pointwise(i, 1) = lpd[i] - elpd[i];
        pointwise(i, 2) = -2.0 * elpd[i];
        pointwise(i, 3) = k[i];
    }
    for (int j = 0; j < 3; ++j) {
        double sum = 0.0, ss = 0.0;
        for (int i = 0; i < N; ++i) sum += pointwise(i, j);
        const double mean = sum / N;
        for (int i = 0; i < N; ++i) ss += (pointwise(i, j) - mean) * (pointwise(i, j) - mean);
        estimates(j, 0) = sum;
        estimates(j, 1) = N > 1 ? std::sqrt(N * (ss / (N - 1))) : NAN;
    }
    return List::create(Named("estimates") = estimates, Named("pointwise") = pointwise,
                        Named("diagnostics") = List::create(Named("pareto_k") = k, Named("n_eff") = n_eff));
}

// The S x N log-likelihood matrix l[s, i] = log p(x_i | draw s) that loo::loo() takes.  theta, pi and data as waic_cpp.
// [[Rcpp::export]]
NumericMatrix log_lik_cpp(IntegerMatrix data, NumericVector theta, NumericMatrix pi) {
    IntegerVector dim = theta.attr("dim");
    if (dim.size() != 3) stop("theta must be a K x P x S array");
    const int K = dim[0], P = dim[1], S = dim[2], N = data.nrow();
    if (data.ncol() != P || pi.nrow() != S || pi.ncol() != K) stop("data / theta / pi dimensions do not match");
    if (S < 2) stop("log_lik needs at least 2 draws");
    NumericMatrix out(S, N);
    if (bmm_loglik_matrix(data.begin(), N, P, K, S, 1, theta.begin(), pi.begin(), 0u, 0, out.begin()) != BMM_OK)
        stop(bmm_last_error());
    return out;
}

// Posterior predictive distribution (no reference counterpart; the reference's TODO:6 lists it).  theta: K x P x S array
// and pi: S x K matrix as gibbs_full / gibbs_stickbreaking return them; newdata: M x P 0/1 integer matrix.
// [[Rcpp::export]]
List predictive_cpp(IntegerMatrix newdata, NumericVector theta, NumericMatrix pi) {
    IntegerVector dim = theta.attr("dim");
    if (dim.size() != 3) stop("theta must be a K x P x S array");
    const int K = dim[0], P = dim[1], S = dim[2], M = newdata.nrow();
    if (newdata.ncol() != P || pi.nrow() != S || pi.ncol() != K) stop("newdata / theta / pi dimensions do not match");
    NumericVector logpred(M);
    NumericMatrix member(M, K);
    if (bmm_predictive(newdata.begin(), M, P, K, S, theta.begin(), pi.begin(), logpred.begin(), member.begin()) != BMM_OK)
        stop(bmm_last_error());
    return List::create(Named("log_pred") = logpred, Named("membership") = member);
}
