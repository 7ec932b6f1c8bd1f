// TEST INFRASTRUCTURE (tests/test_host_nb_math.py): compiles the FP64 device arithmetic of
// digdriver_b200/csrc/nb_math.cuh for the HOST with g++ (-ffp-contract=off), so the CPU-only test tier can
// check the very same source against the reference-generated golden vectors before it ever runs on a GPU.
// Nothing in the product imports or links this file.
#include <cmath>
#include <cstdint>
#include <cstring>

#define DIG_NB_MATH_HOST_CHECK
#define __device__
using std::isinf;
using std::isnan;
using std::fma;
static inline double __longlong_as_double(long long v)
{
    double d;
    std::memcpy(&d, &v, sizeof d);
    return d;
}
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __ddiv_rn(double a, double b) { return a / b; }

#include "../digdriver_b200/csrc/nb_math.cuh"

extern "C" {

void hc_nb_midp(const double *k, const double *a, const double *p, int64_t n, double *out)
{
    for (int64_t i = 0; i < n; ++i) out[i] = dig_nb::nb_midp(k[i], a[i], p[i]);
}

void hc_nb_exact(const double *k, const double *a, const double *p, int64_t n, double *out)
{
    for (int64_t i = 0; i < n; ++i) out[i] = dig_nb::nb_exact(k[i], a[i], p[i]);
}

void hc_nb_variant(int mode, const double *k, const double *a, const double *p, const double *mu, int64_t n, double *out)
{
    for (int64_t i = 0; i < n; ++i) out[i] = dig_nb::nb_variant(mode, k[i], a[i], p[i], mu ? mu[i] : 0.0, mu != nullptr);
}

void hc_loglik(int kind, const double *x, const double *a, const double *b, int64_t n, double *out)
{
    for (int64_t i = 0; i < n; ++i)
        out[i] = kind == 0 ? dig_nb::ll_nb_dev(x[i], a[i], b[i])
                           : kind == 1 ? dig_nb::ll_pois_dev(x[i], a[i]) : dig_nb::ll_gamma_dev(x[i], a[i], b[i]);
}

void hc_llr(int model, const double *alpha, const double *theta, const double *pi3, const double *obs3,
            const double *mrfold, const double *t_syn, int64_t n, double *out)
{
    for (int64_t g = 0; g < n; ++g) {
        double r[4];
        dig_nb::llr_row(model, alpha[g], theta[g], pi3 + g * 3, obs3 + g * 3, mrfold[g], t_syn ? t_syn[g] : 0.0, r);
        for (int j = 0; j < 4; ++j) out[j * n + g] = r[j];
    }
}

void hc_fisher2(const double *a, const double *b, int64_t n, double *out)
{
    for (int64_t i = 0; i < n; ++i) out[i] = dig_nb::fisher2(a[i], b[i]);
}

void hc_chi2_sf(int df, const double *x, int64_t n, double *out)
{
    for (int64_t i = 0; i < n; ++i) out[i] = dig_nb::chi2_sf(x[i], df);
}
}
