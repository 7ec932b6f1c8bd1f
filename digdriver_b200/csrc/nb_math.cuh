// FP64 negative-binomial mid-p arithmetic shared by nbtest.cu and genetest.cu (see nbtest.cu for the method).
#pragma once
#ifndef DIG_NB_MATH_HOST_CHECK      /* tools/host_nb_check.cpp compiles this header with g++ */
#include "dig_common.cuh"
#endif

namespace dig_nb {

__device__ const double c_sfe[31] = {
    0.0, 0.1534264097200273452913848, 0.0810614667953272582196702, 0.0548141210519176538961390,
    0.0413406959554092940938221, 0.03316287351993628748511048, 0.02767792568499833914878929,
    0.02374616365629749597132920, 0.02079067210376509311152277, 0.01848845053267318523077934,
    0.01664469118982119216319487, 0.01513497322191737887351255, 0.01387612882307074799874573,
    0.01281046524292022692424986, 0.01189670994589177009505572, 0.01110455975820691732662991,
    0.010411265261972096497478567, 0.009799416126158803298389475, 0.009255462182712732917728637,
    0.008768700134139385462952823, 0.008330563433362871256469318, 0.007934114564314020547248100,
    0.007573675487951840794972024, 0.007244554301320383179543912, 0.006942840107209529865664152,
    0.006665247032707682442354394, 0.006408994188004207068439631, 0.006171712263039457647532867,
    0.005951370112758847735624416, 0.005746216513010115682023589, 0.005554733551962801371038690};

constexpr double LN_SQRT_2PI = 0.918938533204672741780329736406;
constexpr double LN_2PI = 1.837877066409345483560659472811;

// log(n!) - log(sqrt(2 pi n) (n/e)^n)
__device__ inline double stirlerr(double n)
{
    if (n <= 15.0) {
        const double nn = n + n;
        if (nn == floor(nn)) return c_sfe[(int)nn];
        return lgamma(n + 1.0) - (n + 0.5) * log(n) + n - LN_SQRT_2PI;
    }
    const double S0 = 1.0 / 12.0, S1 = 1.0 / 360.0, S2 = 1.0 / 1260.0, S3 = 1.0 / 1680.0, S4 = 1.0 / 1188.0;
    const double nn = n * n;
    if (n > 500.0) return (S0 - S1 / nn) / n;
    if (n > 80.0) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35.0) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

// deviance term x log(x/np) + np - x without cancellation when x ~ np
__device__ inline double bd0(double x, double np)
{
    if (fabs(x - np) < 0.1 * (x + np)) {
        double v = (x - np) / (x + np);
        double s = (x - np) * v;
        if (fabs(s) < 2.2250738585072014e-308) return s;
        double ej = 2.0 * x * v;
        v = v * v;
        for (int j = 1; j < 1000; ++j) {
            ej *= v;
            const double s1 = s + ej / (double)((j << 1) + 1);
            if (s1 == s) return s1;
            s = s1;
        }
    }
    return x * log(x / np) + np - x;
}

// log of the binomial-type kernel of Loader's algorithm (x, n real)
__device__ inline double log_dbinom_raw(double x, double n, double p, double q)
{
    if (x == 0.0) {
        if (n == 0.0) return 0.0;
        return p < 0.1 ? -bd0(n, n * q) - n * p : n * log(q);
    }
    if (x == n) return q < 0.1 ? -bd0(n, n * p) - n * q : n * log(p);
    const double lc = stirlerr(n) - stirlerr(x) - stirlerr(n - x) - bd0(x, n * p) - bd0(n - x, n * q);
    // log(1 - x/n): once x/n is near 1 (k << alpha in the NB density) the rounding of x/n is all that is left of
    // 1 - x/n, so take it as (n - x)/n, where n - x is exact
    const double r = x / n;
    const double lf = LN_2PI + log(x) + (r < 0.5 ? log1p(-r) : log((n - x) / n));
    return lc - 0.5 * lf;
}

// log of Gamma(k+a)/(Gamma(a) Gamma(k+1)) p^a q^k for real k >= 0, a > 0, 0 < p,q < 1
__device__ inline double log_nb_density(double k, double a, double p, double q)
{
    if (k == 0.0) return p > 0.5 ? a * log1p(-q) : a * log(p);
    if (k < 1e-10 * a)
        return a * log(p) + k * (log(a) + log(q)) - lgamma(k + 1.0) + log1p(k * (k - 1.0) / (2.0 * a));
    return log_dbinom_raw(a, k + a, p, q) + log(a / (a + k));
}

// Continued fraction of I_x(a,b) (the form of Numerical Recipes' betacf: 1 / (1 + d_1 / (1 + d_2 / (1 + ...)))); converges
// fast for x < (a+1)/(a+b+2).  Evaluated by the forward (Wallis) recurrence on numerators and denominators that carry
// a common scale instead of modified Lentz: with d_n = N_n / D_n the step
//     A_n = D_n A_{n-1} + N_n A_{n-2},  B_n likewise,  and (A_{n-1}, B_{n-1}) scaled by D_n as well
// needs NO division (Lentz spends six per iteration, each a chain of ~30 dependent FP64 instructions; the gene-test kernel
// is bound by the latency of exactly that chain).  Same truncation rule as before: stop when two successive convergents
// agree to 1e-15 (|A_n B_{n-1} - A_{n-1} B_n| <= eps |A_{n-1} B_n|, the `del` of Lentz), checked after each odd step.
// y is 1 - x as the caller holds it (the NB's p and q = 1 - p), so it carries no cancellation of its own.
__device__ inline double beta_cf(double a, double b, double x, double y)
{
    const double EPS = 1e-15, BIG = 0x1p+200, SMALL = 0x1p-200;    // growth per iteration < 2^110 (a + 2m up to ~2^27 squared, twice): products stay finite
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    // convergents after the leading term d_1 = -qab x / qap:  (R, S) = A_1, B_1 and (P, Q) = A_2, B_2, both times qap.
    // Q = (a+1) - (a+b) x cancels near the side switch; as a y + 1 - b x with the larger product exact inside the
    // outer fma it keeps its digits (qap - qab * x lost ~1e-5 relative at alpha = 1e12)
    const double ay = a * y, bx = b * x;
    double R = qap, S = qap, P = qap, Q = ay >= bx ? fma(a, y, fma(-b, x, 1.0)) : fma(-b, x, fma(a, y, 1.0));
    for (int m = 1; m < 2000000; ++m) {
        const double dm = (double)m, m2 = 2.0 * dm;
        // even step: d = m (b - m) x / ((a + 2m - 1)(a + 2m))
        double N = dm * (b - dm) * x, D = (qam + m2) * (a + m2);
        double An = D * P + N * R, Bn = D * Q + N * S;
        R = D * P;
        S = D * Q;
        P = An;
        Q = Bn;
        // odd step: d = -(a + m)(a + b + m) x / ((a + 2m)(a + 2m + 1))
        N = -(a + dm) * (qab + dm) * x;
        D = (a + m2) * (qap + m2);
        An = D * P + N * R;
        Bn = D * Q + N * S;
        R = D * P;
        S = D * Q;
        P = An;
        Q = Bn;
        if (fabs(P * S - R * Q) <= EPS * fabs(R * Q)) break;
        const double mag = fabs(Q) > fabs(P) ? fabs(Q) : fabs(P);
        if (mag > BIG) {
            P *= SMALL; Q *= SMALL; R *= SMALL; S *= SMALL;
        } else if (mag < SMALL) {
            P *= BIG; Q *= BIG; R *= BIG; S *= BIG;
        }
    }
    return P / Q;
}

// P(X <= kk) / pmf(kk), the p side of the switch: q (kk+alpha)/alpha CF(alpha, kk+1, p).  While m << alpha every odd
// step of that fraction has 1 + d ~ q + (m - kk)/alpha, so the recurrence cancels about log10(1/q) digits per step when
// p is near 1 (3.5e-8 relative lost at alpha = 3e8, q = 3e-8; 1e-5 at alpha = 1e12, q = 3e-11).  For integer kk with
// q < 1e-4 (the site and codon regime) or kk < 1e-10 alpha, the finite sum is taken downward from kk instead: on this
// side of the switch its ratios j / ((j-1+alpha) q) stay below 1 and shrink, so it stops as soon as the geometric bound
// on the rest is below 1e-17 of the sum.  The sum has at most kk terms, so it is taken only for kk < 2e6 (beta_cf's own
// iteration cap); a larger kk keeps the fraction, and no thread loops on a j that j -= 1 cannot move.
__device__ inline double nb_lower_over_pmf(double kk, double alpha, double p, double q)
{
    if ((q < 1e-4 || kk < 1e-10 * alpha) && kk < 2e6 && kk == floor(kk)) {
        double t = 1.0, s = 1.0;
        for (double j = kk; j > 0.0; j -= 1.0) {
            const double r = j / ((j - 1.0 + alpha) * q);
            t *= r;
            s += t;
            if (r < 1.0 && t * r < 1e-17 * s * (1.0 - r)) break;
        }
        return s;
    }
    return q * (kk + alpha) / alpha * beta_cf(alpha, kk + 1.0, p, q);
}

__device__ inline double nb_midp(double k, double alpha, double p)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (isnan(k) || isnan(alpha) || isnan(p)) return nan;
    if (!(alpha > 0.0) || isinf(alpha) || k < 0.0 || isinf(k) || p < 0.0 || p > 1.0) return nan;
    const double q = 1.0 - p;
    const bool isint = (k == floor(k));
    if (q <= 0.0) return k == 0.0 ? 0.5 : 0.0;   // p == 1: all mass at 0
    if (p <= 0.0) return 1.0;
    // k = 0 (most sites / positions): pmf = p^alpha and sf = betainc(1, alpha, q) = 1 - (1 - q)^alpha in closed form
    if (k == 0.0) return 1.0 - 0.5 * exp(alpha * (p > 0.5 ? log1p(-q) : log(p)));
    const double lg = log_nb_density(k, alpha, p, q);
    const double a = k + 1.0;
    double sf;
    if (q < (a + 1.0) / (a + alpha + 2.0)) {
        const double cf = beta_cf(a, alpha, q, p);
        sf = exp(lg + log(q * (k + alpha) / a * cf));
    } else {
        sf = 1.0 - exp(lg + log(nb_lower_over_pmf(k, alpha, p, q)));
    }
    return (isint ? 0.5 * exp(lg) : 0.0) + sf;
}

// nb_pvalue_exact (nb_model.py:298-314): lower tail I_p(alpha, k+1) when k is below the mean alpha (1-p)/p,
// otherwise upper tail I_{1-p}(k, alpha) with the pmf as fallback when that underflows to 0.  Both tails come from
// the same density + continued-fraction pieces as nb_midp, choosing per tail the form that has no cancellation.
__device__ inline double nb_tail_upper_from(double kk, double alpha, double p, double q)     // P(X > kk) = I_q(kk+1, alpha)
{
    const double lg = log_nb_density(kk, alpha, p, q);
    const double a = kk + 1.0;
    if (q < (a + 1.0) / (a + alpha + 2.0)) return exp(lg + log(q * (kk + alpha) / a * beta_cf(a, alpha, q, p)));
    return 1.0 - exp(lg + log(nb_lower_over_pmf(kk, alpha, p, q)));
}

__device__ inline double nb_tail_lower_to(double kk, double alpha, double p, double q)       // P(X <= kk) = I_p(alpha, kk+1)
{
    const double lg = log_nb_density(kk, alpha, p, q);
    const double a = kk + 1.0;
    if (q < (a + 1.0) / (a + alpha + 2.0)) return 1.0 - exp(lg + log(q * (kk + alpha) / a * beta_cf(a, alpha, q, p)));
    return exp(lg + log(nb_lower_over_pmf(kk, alpha, p, q)));
}

// General regularized incomplete beta I_x(a, b) (lgamma prefactor + the same continued fraction); only used by
// nb_variant for the rare non-integer 0 < k < 1, where the density-relative forms above do not apply.
__device__ inline double ibeta_general(double a, double b, double x)
{
    if (x <= 0.0) return 0.0;
    if (x >= 1.0) return 1.0;
    const double lf = lgamma(a + b) - lgamma(a) - lgamma(b) + a * log(x) + b * log1p(-x);
    const double y = 1.0 - x;
    if (x < (a + 1.0) / (a + b + 2.0)) return exp(lf + log(beta_cf(a, b, x, y) / a));
    return 1.0 - exp(lf + log(beta_cf(b, a, y, x) / b));
}

// The other tail conventions of nb_model.py, selected by `mode` (include/dig_b200.h DIG_NB_*):
//   GREATER    :243-256  k == 0 -> 1, else betainc(k, alpha, 1-p), pmf(k) when that underflows to 0
//   LESS       :280-283  betainc(alpha, k+1, p)   (the reference computes this value and forgets to return it)
//   LESS_MIDP  :285-296  0.5 pmf(k) + (k > 0 ? betainc(alpha, k, p) : 0)
//   EXACT      :298-314  lower tail when k < mu, else GREATER without the k == 0 shortcut
//   MIDP       :316-337  k < mu ? LESS_MIDP : 0.5 pmf(k) + betainc(k+1, alpha, 1-p)
// mu is the caller's expectation; a falsy value (absent or 0) means alpha (1-p)/p as in `if not mu`.
enum { NB_GREATER = 0, NB_GREATER_MIDP = 1, NB_LESS = 2, NB_LESS_MIDP = 3, NB_EXACT = 4, NB_MIDP = 5 };

__device__ inline double nb_upper_incl(double k, double alpha, double p, double q)   // betainc(k, alpha, q), k > 0
{
    if (q <= 0.0) return 0.0;
    if (p <= 0.0) return 1.0;
    if (k < 1.0) return ibeta_general(k, alpha, q);
    return nb_tail_upper_from(k - 1.0, alpha, p, q);
}

__device__ inline double nb_lower_excl(double k, double alpha, double p, double q)   // betainc(alpha, k, p), k > 0
{
    if (q <= 0.0) return 1.0;
    if (p <= 0.0) return 0.0;
    if (k < 1.0) return ibeta_general(alpha, k, p);
    return nb_tail_lower_to(k - 1.0, alpha, p, q);
}

__device__ inline double nb_exact(double k, double alpha, double p)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (isnan(k) || isnan(alpha) || isnan(p)) return nan;
    if (!(alpha > 0.0) || isinf(alpha) || k < 0.0 || isinf(k) || p < 0.0 || p > 1.0) return nan;
    const double q = 1.0 - p;
    const double mean = alpha * q / p;                       // +inf when p == 0
    if (k < mean) {
        if (p <= 0.0) return 0.0;                            // betainc(alpha, k+1, 0)
        if (k == 0.0) return exp(alpha * log(p));            // I_p(alpha, 1) = p^alpha
        return nb_tail_lower_to(k, alpha, p, q);
    }
    // only reached with q < 1
    if (k == 0.0) return 1.0;                                // betainc(0, alpha, q) = 1 (q > 0), else pmf(0; p = 1) = 1
    if (q <= 0.0) return 0.0;                                // betainc(k, alpha, 0) = 0 and pmf(k > 0; p = 1) = 0
    const double up = nb_upper_incl(k, alpha, p, q);          // ibeta_general for a non-integer 0 < k < 1
    if (up == 0.0) return exp(log_nb_density(k, alpha, p, q));
    return up;
}

__device__ inline double nb_pmf(double k, double alpha, double p, double q)          // scipy.stats.nbinom.pmf
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (p <= 0.0) return nan;                                  // outside nbinom's parameter domain
    if (k != floor(k)) return 0.0;
    if (q <= 0.0) return k == 0.0 ? 1.0 : 0.0;
    return exp(log_nb_density(k, alpha, p, q));
}

__device__ inline double nb_variant(int mode, double k, double alpha, double p, double mu, bool has_mu)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (mode == NB_GREATER_MIDP) return nb_midp(k, alpha, p);
    if (isnan(k) || isnan(alpha) || isnan(p)) return nan;
    if (!(alpha > 0.0) || isinf(alpha) || k < 0.0 || isinf(k) || p < 0.0 || p > 1.0) return nan;
    const double q = 1.0 - p;
    if (mode == NB_GREATER || mode == NB_EXACT || mode == NB_MIDP) {
        bool lower = false;
        if (mode != NB_GREATER) {
            const double m = (has_mu && mu != 0.0) ? mu : alpha * q / p;     // +inf (or NaN -> upper) when p == 0
            lower = k < m;
        }
        if (mode == NB_GREATER || (mode == NB_EXACT && !lower)) {
            if (k == 0.0) return 1.0;
            const double up = nb_upper_incl(k, alpha, p, q);
            return up == 0.0 ? nb_pmf(k, alpha, p, q) : up;
        }
        if (mode == NB_EXACT) {                                // lower tail betainc(alpha, k+1, p)
            if (p <= 0.0) return 0.0;
            if (q <= 0.0) return 1.0;
            if (k == 0.0) return exp(alpha * log(p));
            return nb_tail_lower_to(k, alpha, p, q);
        }
        if (!lower) return nb_midp(k, alpha, p);               // MIDP, upper side
        const double half = 0.5 * nb_pmf(k, alpha, p, q);      // MIDP, lower side == LESS_MIDP
        return k > 0.0 ? half + nb_lower_excl(k, alpha, p, q) : half;
    }
    if (mode == NB_LESS) {
        if (p <= 0.0) return 0.0;
        if (q <= 0.0) return 1.0;
        if (k == 0.0) return exp(alpha * log(p));
        return nb_tail_lower_to(k, alpha, p, q);
    }
    if (mode == NB_LESS_MIDP) {
        const double half = 0.5 * nb_pmf(k, alpha, p, q);
        return k > 0.0 ? half + nb_lower_excl(k, alpha, p, q) : half;
    }
    return nan;
}

// Log-likelihood terms of the selection tests (transfer_tools.py:1254-1262), in SciPy's own formulas:
//   kind 0  _ll_nb(k, alpha, theta)      nbinom.logpmf(k, alpha, 1 / (1 + theta))
//   kind 1  _ll_pois(k, lam)             poisson.logpmf = xlogy(k, lam) - gammaln(k + 1) - lam
//   kind 2  _ll_gamma(lam, alpha, theta) gamma.logpdf(lam, alpha, scale=theta)
//                                        = xlogy(alpha - 1, lam/theta) - lam/theta - gammaln(alpha) - log(theta)
__device__ inline double xlogy(double x, double y) { return (x == 0.0 && !isnan(y)) ? 0.0 : x * log(y); }

__device__ inline double ll_pois_dev(double k, double lam)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (isnan(k) || isnan(lam) || lam < 0.0) return nan;
    if (k < 0.0 || k != floor(k)) return -INFINITY;
    return xlogy(k, lam) - lgamma(k + 1.0) - lam;
}

__device__ inline double ll_gamma_dev(double x, double a, double theta)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (isnan(x) || isnan(a) || isnan(theta) || !(a > 0.0) || !(theta > 0.0)) return nan;
    const double y = x / theta;
    if (y < 0.0) return -INFINITY;
    return xlogy(a - 1.0, y) - y - lgamma(a) - log(theta);
}

__device__ inline double ll_nb_dev(double k, double alpha, double theta)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const double p = __ddiv_rn(1.0, __dadd_rn(1.0, theta));
    const double q = 1.0 - p;
    if (isnan(p) || isnan(k) || isnan(alpha) || !(alpha > 0.0) || p <= 0.0 || p > 1.0) return nan;
    if (k < 0.0 || k != floor(k)) return -INFINITY;
    if (q <= 0.0) return k == 0.0 ? 0.0 : -INFINITY;
    return log_nb_density(k, alpha, p, q);
}

// chi2.sf(x, df) for df = 1, 2 (the likelihood-ratio tests)
__device__ inline double chi2_sf(double x, int df)
{
    if (isnan(x)) return x;
    if (x <= 0.0) return 1.0;
    return df == 1 ? erfc(sqrt(0.5 * x)) : exp(-0.5 * x);
}

// One row of _llr_test_nb (model 0; P / O = SYN, MIS, TRUNC) or _llr_test_gamma_poiss (model 1; SYN, MIS, NONS and the
// gamma prior term of T_SYN) -- transfer_tools.py:1172-1252, sums in the reference's order, no FMA contraction.
__device__ inline void llr_row(int model, double a, double t, const double *P, const double *O, double mrf, double t_syn,
                               double *out4)
{
    double l0[3], l1[3];
    for (int c = 0; c < 3; ++c) {
        if (model == 0) {
            l0[c] = ll_nb_dev(O[c], a, __dmul_rn(__dmul_rn(t, P[c]), mrf));
            l1[c] = ll_nb_dev(O[c], a, __ddiv_rn(O[c], a));
        } else {
            l0[c] = ll_pois_dev(O[c], __dmul_rn(__dmul_rn(__dmul_rn(a, t), P[c]), mrf));
            l1[c] = ll_pois_dev(O[c], O[c]);
        }
    }
    double ll[5];
    ll[0] = __dadd_rn(__dadd_rn(l0[0], l0[1]), l0[2]);
    ll[1] = __dadd_rn(__dadd_rn(l1[0], l0[1]), l0[2]);
    ll[2] = __dadd_rn(__dadd_rn(l0[0], l1[1]), l0[2]);
    ll[3] = __dadd_rn(__dadd_rn(l0[0], l0[1]), l1[2]);
    ll[4] = __dadd_rn(__dadd_rn(l0[0], l1[1]), l1[2]);
    if (model != 0) {
        const double lg = ll_gamma_dev(t_syn, a, __dmul_rn(__dmul_rn(t, P[0]), mrf));
        for (int j = 0; j < 5; ++j) ll[j] = __dadd_rn(ll[j], lg);
    }
    out4[0] = chi2_sf(-2.0 * (ll[0] - ll[1]), 1);
    out4[1] = chi2_sf(-2.0 * (ll[0] - ll[2]), 1);
    out4[2] = chi2_sf(-2.0 * (ll[0] - ll[3]), 1);
    out4[3] = chi2_sf(-2.0 * (ll[0] - ll[4]), 2);
}

// chi2.sf(-2 (ln p1 + ln p2), df=4) = exp(-y) (1 + y), y = -(ln p1 + ln p2)  (transfer_tools.py:860-861)
__device__ inline double fisher2(double a, double b)
{
    if (isnan(a) || isnan(b)) return __longlong_as_double(0x7ff8000000000000LL);
    const double y = -(log(a) + log(b));     // log(0) = -inf -> y = +inf -> 0
    if (isnan(y)) return y;
    if (y <= 0.0) return 1.0;
    if (isinf(y)) return 0.0;
    return exp(-y) * (1.0 + y);
}

}  // namespace dig_nb
