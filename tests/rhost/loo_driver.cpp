// TEST INFRASTRUCTURE.  loo_gibbs's and log_lik_gibbs's Rcpp host functions (r-package/src/host.cpp::loo_cpp,
// log_lik_cpp), compiled unmodified against the Rcpp stand-in (oracle/shim/) and linked with libbmm_b200.so, driven the
// way R's generated RcppExports.cpp would drive them: Rcpp matrices in, the returned objects out.  tests/test_gpu_loo.py
// compares them with the ctypes path.
#include <cstring>
#include <string>

#include "../../r-package/src/host.cpp"

namespace {
thread_local std::string g_err;

const SEXPREC *find(const List &l, const char *name) {
    for (size_t i = 0; i < l.p->names.size(); ++i)
        if (l.p->names[i] == name) return l.p->elts[i].get();
    return nullptr;
}

bool copy_out(const SEXPREC *s, double *dst, long long n) {
    if (!s) return false;
    const std::vector<double> &v = s->real;
    if ((long long)v.size() != n) return false;
    std::memcpy(dst, v.data(), v.size() * sizeof(double));
    return true;
}

void inputs(const int *X, int N, int P, int K, int S, const double *theta, const double *pi, IntegerMatrix &x,
            NumericVector &th, NumericMatrix &pm) {
    std::memcpy(x.begin(), X, sizeof(int) * (size_t)N * P);
    std::memcpy(th.begin(), theta, sizeof(double) * (size_t)K * P * S);
    std::memcpy(pm.begin(), pi, sizeof(double) * (size_t)S * K);
}
}  // namespace

extern "C" {

const char *rhost_loo_last_error(void) { return g_err.c_str(); }

// loo_gibbs with r_eff = N values: estimates[3 x 2 cm], pointwise[N x 4 cm], pareto_k[N], n_eff[N]
int rhost_loo(const int *X, int N, int P, int K, int S, const double *theta, const double *pi, const double *r_eff,
              double *estimates, double *pointwise, double *pareto_k, double *n_eff) {
    try {
        IntegerMatrix x(N, P);
        NumericVector th(Dimension(K, P, S)), re(N);
        NumericMatrix pm(S, K);
        inputs(X, N, P, K, S, theta, pi, x, th, pm);
        std::memcpy(re.begin(), r_eff, sizeof(double) * (size_t)N);
        List r = loo_cpp(x, th, pm, re);
        const SEXPREC *dg = find(r, "diagnostics");
        if (!copy_out(find(r, "estimates"), estimates, 6) || !copy_out(find(r, "pointwise"), pointwise, (long long)N * 4) ||
            !dg || dg->names.size() != 2 || dg->names[0] != "pareto_k" || dg->names[1] != "n_eff" ||
            !copy_out(dg->elts[0].get(), pareto_k, N) || !copy_out(dg->elts[1].get(), n_eff, N))
            throw std::runtime_error("loo_cpp returned an unexpected list");
        return 0;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

// log_lik_gibbs: out[S x N cm]
int rhost_loglik(const int *X, int N, int P, int K, int S, const double *theta, const double *pi, double *out) {
    try {
        IntegerMatrix x(N, P);
        NumericVector th(Dimension(K, P, S));
        NumericMatrix pm(S, K);
        inputs(X, N, P, K, S, theta, pi, x, th, pm);
        NumericMatrix m = log_lik_cpp(x, th, pm);
        if (m.nrow() != S || m.ncol() != N) throw std::runtime_error("log_lik_cpp returned a matrix of the wrong shape");
        std::memcpy(out, m.begin(), sizeof(double) * (size_t)S * N);
        return 0;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

}  // extern "C"
