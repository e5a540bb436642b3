// Per-point exchange-correlation math shared by the energy/potential kernels (functionals.cu) and the stress
// kernels (stress.cu).
#pragma once
#include "common.cuh"

constexpr double kCX = -0.7385587663820223;        // -(3/4)(3/pi)^(1/3)
constexpr double kRS13 = 0.6203504908994001;       // (3/(4 pi))^(1/3)

struct PZ {
    double e, v;   // eps_c * n and d(eps_c n)/dn
};
__device__ __forceinline__ PZ pz_correlation(double n, double c13) {
    // functionals.py:1515-1521 ; potential: tests/tools_for_tests.py:125-131
    const double A = 0.0311, B = -0.048, C = 0.002, D = -0.0116;
    const double ga = -0.1423, b1 = 1.0529, b2 = 0.3334;
    const double rs = kRS13 / c13;
    PZ r;
    if (rs < 1.0) {
        const double lr = log(rs);
        r.e = n * (A * lr + B + C * rs * lr + D * rs);
        r.v = lr * (A + (2.0 / 3.0) * C * rs) + (B - A / 3.0) + rs / 3.0 * (2.0 * D - C);
    } else {
        const double sr = sqrt(rs);
        const double dn = 1.0 + b1 * sr + b2 * rs;
        r.e = n * ga / dn;
        r.v = ga * (1.0 + (7.0 / 6.0) * b1 * sr + (4.0 / 3.0) * b2 * rs) / (dn * dn);
    }
    return r;
}


// PBE exchange (do_x) and/or correlation (do_c), functionals.py:1597-1635 with the reference's +1e-30 guards:
// energy density f, df/dn and df/dsigma at density n, sigma = |grad n|^2, c13 = cbrt(n)
// (tests/tools_for_tests.py:155-207)
__device__ __forceinline__ void pbe_point(double n, double sig, double c13, bool do_x, bool do_c, double& f, double& f_rho,
                                          double& f_sig) {
    f = 0.0; f_rho = 0.0; f_sig = 0.0;
    if (do_x) {
        const double cs = 0.026121172985233605;       // (1/4)(3 pi^2)^(-2/3)
        const double kap = 0.804, mu = 0.2195164512208958;
        const double ex = kCX * n * c13;
        const double r83 = n * n * c13 * c13;
        const double s2 = cs * sig / r83;
        const double q = 1.0 + mu / kap * s2;
        const double Fx = 1.0 + kap - kap / q, dF = mu / (q * q);
        f += Fx * ex;
        f_rho += Fx * (4.0 / 3.0) * kCX * c13 + ex * dF * (-8.0 / 3.0) * s2 / n;
        f_sig += ex * dF * cs / r83;
    }
    if (do_c) {
        const double A1 = 0.0310907, a1 = 0.2137, b1 = 7.5957, b2 = 3.5876, b3 = 1.6382, b4 = 0.49294;
        const double be = 0.066725, ga = 0.0310906908696549;   // (1 - ln 2) / pi^2
        const double ct = 0.0634682060977037;                  // (1/16)(pi/3)^(1/3)
        const double rs = kRS13 / c13;
        const double sr = sqrt(rs);
        const double Q = 2.0 * A1 * (b1 * sr + b2 * rs + b3 * rs * sr + b4 * rs * rs);
        const double lg = log(1.0 + 1.0 / Q);
        const double eps = -2.0 * A1 * (1.0 + a1 * rs) * lg;
        const double dQ = A1 * (b1 / sr + 2.0 * b2 + 3.0 * b3 * sr + 4.0 * b4 * rs);
        const double deps = (-2.0 * A1 * a1 * lg + 2.0 * A1 * (1.0 + a1 * rs) * dQ / (Q * (Q + 1.0))) * (-rs / (3.0 * n));
        const double ee = exp(-eps / ga);
        const double Aa = be / ga / (ee - 1.0 + 1e-30);
        const double dAa = Aa * Aa / be * ee * deps;
        const double r73 = n * n * c13 + 1e-30;
        const double t2 = ct * sig / r73;
        const double dt2_rho = -ct * sig * (7.0 / 3.0) * n * c13 / (r73 * r73);
        const double dt2_sig = ct / r73;
        const double X = Aa * t2;
        const double num = 1.0 + X, dnm = 1.0 + X + X * X;
        const double Rr = num / dnm;
        const double dR = -X * (2.0 + X) / (dnm * dnm);
        const double inner = 1.0 + be / ga * t2 * Rr;
        const double H = ga * log(inner);
        const double dH_rho = be / inner * (Rr * dt2_rho + t2 * dR * (Aa * dt2_rho + t2 * dAa));
        const double dH_sig = be / inner * (Rr + t2 * dR * Aa) * dt2_sig;
        f += n * (eps + H);
        f_rho += eps + H + n * (deps + dH_rho);
        f_sig += n * dH_sig;
    }
}

// ---- semilocal kinetic functionals e(n, sigma, L), sigma = |grad n|^2, L = lap n ----------------------------------------
//   e = C_TF n^(5/3) F(p, q),  p = s^2 = kSlC sigma / n^(8/3),  q = kSlC L / n^(5/3)   (functional_tools.py:122-135)
//   LuoKarasievTrickey (PAD_SEMILOCAL_LKT, p0 = a):          F = 1 / cosh(a s) + (5/3) p
//   PauliGaussian      (PAD_SEMILOCAL_PG, p0 = mu, p1 = beta): F = (5/3) p + exp(-mu p) + beta q^2
//   e_n = C_TF n^(2/3) ((5/3) F - (8/3) p F_p - (5/3) q F_q),  e_sigma = C_TF kSlC F_p / n,  e_L = C_TF kSlC F_q
// No guard on n: as in pbe_point, n <= 0 gives whatever these formulas give (cbrt of a negative density, a 0/0 at n = 0),
// as the reference's torch expressions do; the densities the solvers produce are positive.
constexpr double kSlC = 0.026121172985233605;      // (1/4)(3 pi^2)^(-2/3)

// tanh(x) / x for x >= 0 (the sigma-derivative of 1/cosh(a s) carries tanh(a s) / s): its Taylor series below x = 1/16
// (truncation error < 1e-14 relative), so sigma = 0 is no 0/0
__device__ __forceinline__ double tanh_over_x_series(double x) {
    const double x2 = x * x;
    return 1.0 + x2 * (-1.0 / 3.0 + x2 * (2.0 / 15.0 + x2 * (-17.0 / 315.0 + x2 * (62.0 / 2835.0))));
}

__device__ __forceinline__ void semilocal_kinetic_point(double n, double sig, double lap, int variant, double p0, double p1,
                                                        double& e, double& e_n, double& e_sig, double& e_lap) {
    const double c13 = cbrt(n), n23 = c13 * c13, n53 = n * n23;
    const double p = kSlC * sig / (n * n * n23);
    double F, Fp, qFq = 0.0;
    e_lap = 0.0;
    if (variant == 0) {
        const double s = sqrt(p), x = p0 * s;
        const double sech = 1.0 / cosh(x);
        const double tox = x < 0.0625 ? tanh_over_x_series(x) : tanh(x) / x;
        F = sech + (5.0 / 3.0) * p;
        Fp = 5.0 / 3.0 - 0.5 * p0 * p0 * sech * tox;
    } else {
        const double q = kSlC * lap / n53, g = exp(-p0 * p);
        F = (5.0 / 3.0) * p + g + p1 * q * q;
        Fp = 5.0 / 3.0 - p0 * g;
        qFq = 2.0 * p1 * q * q;
        e_lap = kCTF * kSlC * 2.0 * p1 * q;
    }
    e = kCTF * n53 * F;
    e_n = kCTF * n23 * ((5.0 / 3.0) * F - (8.0 / 3.0) * p * Fp - (5.0 / 3.0) * qFq);
    e_sig = kCTF * kSlC * Fp / n;
}
