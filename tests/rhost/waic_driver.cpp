// TEST INFRASTRUCTURE.  waic_gibbs's Rcpp host function (r-package/src/host.cpp::waic_cpp), compiled unmodified against
// the Rcpp stand-in (oracle/shim/) and linked with libbmm_b200.so, driven the way R's generated RcppExports.cpp would
// drive it: Rcpp matrices in, the returned list out.  tests/test_gpu_waic.py compares the list with the ctypes path.
#include <cstring>
#include <string>

#include "../../r-package/src/host.cpp"

namespace {
thread_local std::string g_err;

bool copy_out(const List &l, const char *name, double *dst, long long cap) {
    for (size_t i = 0; i < l.p->names.size(); ++i)
        if (l.p->names[i] == name) {
            const std::vector<double> &v = sexp_traits<double>::vec(*l.p->elts[i]);
            if ((long long)v.size() > cap) return false;
            std::memcpy(dst, v.data(), v.size() * sizeof(double));
            return true;
        }
    return false;
}
}  // namespace

extern "C" {

const char *rhost_waic_last_error(void) { return g_err.c_str(); }

// waic_gibbs: estimates[3 x 2 cm], pointwise[N x 3 cm], loglik[S]
int rhost_waic(const int *X, int N, int P, int K, int S, const double *theta, const double *pi, double *estimates,
               double *pointwise, double *loglik) {
    try {
        IntegerMatrix x(N, P);
        std::memcpy(x.begin(), X, sizeof(int) * (size_t)N * P);
        NumericVector th(Dimension(K, P, S));
        std::memcpy(th.begin(), theta, sizeof(double) * (size_t)K * P * S);
        NumericMatrix pm(S, K);
        std::memcpy(pm.begin(), pi, sizeof(double) * (size_t)S * K);
        List r = waic_cpp(x, th, pm);
        if (!copy_out(r, "estimates", estimates, 6) || !copy_out(r, "pointwise", pointwise, (long long)N * 3) ||
            !copy_out(r, "loglik", loglik, S))
            throw std::runtime_error("waic_cpp returned an unexpected list");
        return 0;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

}  // extern "C"
