// lto_orbit.h -- the halo-orbit lookups of the trajectory-stacking initial guess (CRTBP_Multishoot_direct_demo.jl:117-157,
// interpInitialStates / find_τ of HelperFunctions.jl:18-48), compiled for the host (the fit, tests) and the device (lto_guess.cu).
//
// An orbit table is 6 x n (column-major: state k of node i at X[i*6 + k]) on the uniform grid LinRange(0, 1, n), n >= 3.  Each row
// is interpolated by a natural cubic spline, the interpolant of solvers._orbit_states (scipy's CubicSpline(bc_type="natural")):
//   orbit_fit    solves scipy's tridiagonal system for the knot slopes with LAPACK gtsv's elimination (no pivoting is ever needed:
//                the matrix is diagonally dominant) and stores scipy's piecewise-cubic coefficients, coef[(i*6 + k)*4 + 0..3] =
//                c0..c3 of interval i, y = c3 + c2 s + c1 s^2 + c0 s^3 with s = tau - x_i;
//   orbit_eval   evaluates them in scipy's PPoly order, with no fused multiply-adds on the device;
//   orbit_wrap   tau wrapped as _orbit_states does (while tau > 1: tau -= 1; while tau < 0: tau += 1 -- tau = 1 stays 1);
//   find_τ       scans tau_k = k * 0.001 (np.linspace(0, 1, 1001)) for the first smallest distance (lto_guess.cu).
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define LTO_ORBIT_FN __host__ __device__ inline
#else
#define LTO_ORBIT_FN inline
#endif

#define LTO_ORBIT_NTAU 1001          // find_τ's candidates tau_k = k / 1000, k = 0 .. 1000

LTO_ORBIT_FN double orb_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
LTO_ORBIT_FN double orb_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// knot i of np.linspace(0, 1, n): i * (1 / (n - 1)), the last one exactly 1
LTO_ORBIT_FN double orbit_knot(int i, int n) { return i == n - 1 ? 1.0 : orb_mul((double)i, 1.0 / (double)(n - 1)); }

// candidate k of np.linspace(0, 1, 1001)
LTO_ORBIT_FN double orbit_tau_candidate(int k) { return k == LTO_ORBIT_NTAU - 1 ? 1.0 : orb_mul((double)k, 1.0 / (double)(LTO_ORBIT_NTAU - 1)); }

LTO_ORBIT_FN double orbit_wrap(double tau) {
    while (tau > 1) tau -= 1;
    while (tau < 0) tau += 1;
    return tau;
}

// interval i with x_i <= tau < x_{i+1}; the last one for tau >= x_{n-2} (scipy's find_interval, extrapolating at the ends)
LTO_ORBIT_FN int orbit_interval(double tau, int n) {
    int i = (int)(tau * (double)(n - 1));
    if (!(i >= 0)) i = 0;
    if (i > n - 2) i = n - 2;
    while (i > 0 && tau < orbit_knot(i, n)) --i;
    while (i < n - 2 && tau >= orbit_knot(i + 1, n)) ++i;
    return i;
}

// component k of the spline at tau (tau already wrapped)
LTO_ORBIT_FN double orbit_eval(const double* coef, int n, double tau, int k) {
    const int i = orbit_interval(tau, n);
    const double s = tau - orbit_knot(i, n);
    const double* c = coef + ((long long)i * 6 + k) * 4;
    double res = c[3];
    res = orb_add(res, orb_mul(c[2], s));
    double z = orb_mul(s, s);
    res = orb_add(res, orb_mul(c[1], z));
    z = orb_mul(z, s);
    return orb_add(res, orb_mul(c[0], z));
}

// find_τ's distance norm(f(tau_k) - x) of a candidate state (6 doubles) to x
LTO_ORBIT_FN double orbit_distance(const double* cand, const double* x) {
    double acc = 0.0;
    for (int k = 0; k < 6; ++k) { const double e = cand[k] - x[k]; acc = orb_add(acc, orb_mul(e, e)); }
    return sqrt(acc);
}

// np.argmin's order of (distance, index): the first NaN wins, otherwise the smaller distance, ties to the lower index
LTO_ORBIT_FN bool orbit_before(double da, int ka, double db, int kb) {
    const bool na = !(da == da), nb = !(db == db);
    if (na || nb) return na && (!nb || ka < kb);
    return da < db || (da == db && ka < kb);
}

// Fit (host): X 6 x n, coef (n-1) * 24 doubles, work 4 n doubles.
LTO_ORBIT_FN void orbit_fit(const double* X, int n, double* coef, double* work) {
    double* d = work; double* du = work + n; double* b = work + 2 * n; double* s = work + 3 * n;
    for (int k = 0; k < 6; ++k) {
        auto y = [&](int i) { return X[(long long)i * 6 + k]; };
        auto dx = [&](int i) { return orbit_knot(i + 1, n) - orbit_knot(i, n); };
        auto slope = [&](int i) { return (y(i + 1) - y(i)) / dx(i); };
        // rows: 0 and n-1 the natural end conditions (second derivative 0), 1..n-2 continuity of the second derivative
        d[0] = 2 * dx(0); du[0] = dx(0); b[0] = 3 * (y(1) - y(0));
        for (int r = 1; r < n - 1; ++r) {
            d[r] = 2 * (dx(r - 1) + dx(r)); du[r] = dx(r - 1);
            b[r] = 3 * (dx(r) * slope(r - 1) + dx(r - 1) * slope(r));
        }
        d[n - 1] = 2 * dx(n - 2); du[n - 1] = 0.0; b[n - 1] = 3 * (y(n - 1) - y(n - 2));
        // gtsv: the subdiagonal element of row r + 1 is dx(r + 1) (row n - 1: dx(n - 2))
        for (int r = 0; r < n - 1; ++r) {
            const double sub = r + 1 < n - 1 ? dx(r + 1) : dx(n - 2);
            const double fact = sub / d[r];
            d[r + 1] = d[r + 1] - fact * du[r];
            b[r + 1] = b[r + 1] - fact * b[r];
        }
        s[n - 1] = b[n - 1] / d[n - 1];
        for (int r = n - 2; r >= 0; --r) s[r] = (b[r] - du[r] * s[r + 1]) / d[r];
        // CubicHermiteSpline's coefficients
        for (int i = 0; i < n - 1; ++i) {
            const double h = dx(i), m = slope(i);
            const double t = (s[i] + s[i + 1] - 2 * m) / h;
            double* c = coef + ((long long)i * 6 + k) * 4;
            c[0] = t / h;
            c[1] = (m - s[i]) / h - t;
            c[2] = s[i];
            c[3] = y(i);
        }
    }
}
