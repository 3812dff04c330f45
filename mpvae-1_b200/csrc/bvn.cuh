// Standard bivariate normal CDF in fp64: Phi2(h, k; rho) = P(X <= h, Y <= k), corr(X, Y) = rho.
//
// Genz's BVND (A. Genz, "Numerical computation of rectangular bivariate and trivariate normal and t probabilities",
// Statistics and Computing 14 (2004) 251-260), after Drezner & Wesolowsky (1990): for |rho| < 0.925 the integral of the
// bivariate density over the correlation, from 0 to rho, by Gauss-Legendre rules of 6, 12 or 20 nodes chosen by |rho|;
// for |rho| >= 0.925 the complementary integral from rho to +-1, whose singular part is taken out in closed form.  About
// 1e-15 absolute over the whole (h, k, rho) range, up to |rho| = 1 - 1e-15 (1 - rho^2 is formed as (1 - rho)(1 + rho)).
//
// __host__ __device__ like probit_math.cuh, so tests/host/bvn_host.cpp builds the same code with g++.
#pragma once
#include <math.h>

#include "probit_math.cuh"

namespace mpv {

// Positive half of the n-point Gauss-Legendre rule on [-1, 1] (nodes decreasing), n = 2 * H.  The rule on [0, 2] used
// below has the nodes 1 - x_i and 1 + x_i, each with weight w_i.
template <int H>
MPV_HD void gauss_legendre_half(double* x, double* w) {
    if (H == 3) {
        const double xs[3] = {0.9324695142031519, 0.6612093864662645, 0.2386191860831969};
        const double ws[3] = {0.17132449237917027, 0.3607615730481387, 0.46791393457269104};
        for (int i = 0; i < 3; ++i) { x[i] = xs[i]; w[i] = ws[i]; }
    } else if (H == 6) {
        const double xs[6] = {0.9815606342467192, 0.9041172563704748, 0.7699026741943047, 0.5873179542866175,
                              0.3678314989981802, 0.1252334085114689};
        const double ws[6] = {0.04717533638651141, 0.10693932599531907, 0.16007832854334642, 0.20316742672306573,
                              0.2334925365383546, 0.2491470458134027};
        for (int i = 0; i < 6; ++i) { x[i] = xs[i]; w[i] = ws[i]; }
    } else {
        const double xs[10] = {0.993128599185095, 0.9639719272779138, 0.912234428251326, 0.8391169718222188,
                               0.7463319064601508, 0.636053680726515, 0.5108670019508271, 0.37370608871541955,
                               0.22778585114164507, 0.07652652113349734};
        const double ws[10] = {0.017614007139150893, 0.040601429800386446, 0.06267204833410879, 0.08327674157670471,
                               0.1019301198172407, 0.1181945319615186, 0.1316886384491769, 0.1420961093183824,
                               0.14917298647260424, 0.15275338713072628};
        for (int i = 0; i < 10; ++i) { x[i] = xs[i]; w[i] = ws[i]; }
    }
}

MPV_HD double phi_cdf(double x) { return 0.5 * erfc(-x * 0.70710678118654752440); }

// sum over the 2H nodes t of exp((sn hk - hs) / (1 - sn^2)) w, sn = sin(asr t): the |rho| < 0.925 integrand
template <int H>
MPV_HD double bvn_near(double hk, double hs, double asr) {
    double x[H], w[H];
    gauss_legendre_half<H>(x, w);
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < H; ++i) {
#pragma unroll
        for (int side = -1; side <= 1; side += 2) {
            const double sn = sin(asr * (1.0 + side * x[i]));
            s += w[i] * exp((sn * hk - hs) / (1.0 - sn * sn));
        }
    }
    return s;
}

// P(X > dh, Y > dk): Genz's BVND verbatim (branches and constants), with the node tables above
MPV_HD double bvn_upper(double dh, double dk, double r) {
    const double tp = 6.283185307179586476925;
    double h = dh, k = dk, hk = h * k, bvn = 0.0;
    const double ar = fabs(r);
    if (ar < 0.925) {
        const double hs = (h * h + k * k) / 2.0;
        const double asr = asin(r) / 2.0;
        if (ar < 0.3) bvn = bvn_near<3>(hk, hs, asr);
        else if (ar < 0.75) bvn = bvn_near<6>(hk, hs, asr);
        else bvn = bvn_near<10>(hk, hs, asr);
        return bvn * asr / tp + phi_cdf(-h) * phi_cdf(-k);
    }
    if (r < 0.0) { k = -k; hk = -hk; }
    if (ar < 1.0) {
        const double as = (1.0 - ar) * (1.0 + ar);
        double a = sqrt(as);
        const double bs = (h - k) * (h - k);
        const double c = (4.0 - hk) / 8.0, d = (12.0 - hk) / 16.0;
        bvn = a * exp(-(bs / as + hk) / 2.0) * (1.0 - c * (bs - as) * (1.0 - d * bs / 5.0) / 3.0 + c * d * as * as / 5.0);
        if (hk > -160.0) {
            const double b = sqrt(bs);
            bvn -= exp(-hk / 2.0) * sqrt(tp) * phi_cdf(-b / a) * b * (1.0 - c * bs * (1.0 - d * bs / 5.0) / 3.0);
        }
        a /= 2.0;
        double x[10], w[10];
        gauss_legendre_half<10>(x, w);
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 10; ++i) {
#pragma unroll
            for (int side = -1; side <= 1; side += 2) {
                const double t = a * (1.0 + side * x[i]);
                const double xs = t * t;
                const double rs = sqrt(1.0 - xs);
                s += w[i] * exp(-(bs / xs + hk) / 2.0) *
                     (exp(-hk * (1.0 - rs) / (2.0 * (1.0 + rs))) / rs - (1.0 + c * xs * (1.0 + d * xs)));
            }
        }
        bvn = -(bvn + a * s) / tp;
    }
    if (r > 0.0) return bvn + phi_cdf(-fmax(h, k));
    if (h >= k) return -bvn;
    const double l = h < 0.0 ? phi_cdf(k) - phi_cdf(h) : phi_cdf(-h) - phi_cdf(-k);
    return l - bvn;
}

// Phi2(h, k; rho), clipped to [0, 1]
MPV_HD double bvn_cdf(double h, double k, double rho) {
    const double p = bvn_upper(-h, -k, rho);
    return fmin(1.0, fmax(0.0, p));
}

}  // namespace mpv
