// lto_prop_generic.cuh -- one-thread-per-propagation integrators (state [+ sensitivities]).
//
// These are the general kernels' bodies: every mode (FIXED / ADAPTIVE), every system
// (direct 6/7, indirect 12/14), with or without the variational equations.  The
// throughput kernels (lto_direct_cw.cu, ...) specialise the hot configurations; this
// file is the always-available path for the rest and the cross-check for them.
// The bodies are __host__ __device__ so that the arithmetic can be unit-tested on a
// machine without a GPU (tests/ build them into a test-only library); the product
// library only ever instantiates them inside __global__ kernels.
#pragma once
#include "lto_math.cuh"
#include "lto_tableau.h"

namespace lto {

enum { LTO_OK = 0, LTO_ST_NAN = 1, LTO_ST_HMIN = 2, LTO_ST_MAXSTEPS = 3, LTO_ST_BADP = 4 };

LTO_HD double linrange_at(double a, double b, int len, int j) {
    // Julia Base.lerpi: element j (0-based) of LinRange(a, b, len)
    const double t = (double)j / (double)(len - 1);
    return (1.0 - t) * a + t * b;
}

// One RKF7(8) step on an NT-vector.  k: [13][NT] scratch.  ynew = y + h*K*chi,
// gam = (41/840) h K psi  (GeneralCode/ode.jl:931-940).  Returns rhs status.
template <int NT, class RHS>
LTO_HD int rkf78_step(RHS& rhs, const double* y, double h, double* ynew, double* gam, double* k, double* ytmp) {
    int st = rhs(y, k);
#pragma unroll
    for (int j = 1; j < 13; ++j) {
#pragma unroll 1
        for (int c = 0; c < NT; ++c) {
            double acc = 0.0;
#pragma unroll
            for (int i = 0; i < j; ++i)
                if (lto_tab::Bf(j, i) != 0.0) acc = fma(lto_tab::Bf(j, i), k[i * NT + c], acc);
            ytmp[c] = fma(h, acc, y[c]);
        }
        st |= rhs(ytmp, k + j * NT);
    }
#pragma unroll 1
    for (int c = 0; c < NT; ++c) {
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < 13; ++i)
            if (lto_tab::CHIf(i) != 0.0) acc = fma(lto_tab::CHIf(i), k[i * NT + c], acc);
        ynew[c] = fma(h, acc, y[c]);
        const double e = (k[0 * NT + c] + k[10 * NT + c]) - (k[11 * NT + c] + k[12 * NT + c]);
        gam[c] = (h * lto_tab::ERRC) * e;
    }
    return st;
}

// ---------------------------------------------------------------------------
// RHS functors on the augmented vector  y = [x | col_0 | col_1 | ...]
// ---------------------------------------------------------------------------
template <int NS, bool SENS>
struct EPRhs {
    static constexpr int NCOL = SENS ? NS + 3 : 0;
    static constexpr int NT = NS * (1 + NCOL);
    const EPConst& c;
    double u[3], omega, mdot, bm[3];
    LTO_HD EPRhs(const EPConst& c_, const double* u_, double omega_) : c(c_), omega(omega_) {
        u[0] = u_[0]; u[1] = u_[1]; u[2] = u_[2];
        const double un = sqrt(fma(u[0], u[0], fma(u[1], u[1], u[2] * u[2])));
        mdot = -omega * un * c.cmdot;                       // CRTBP_prop_EP_deriv.jl:42
        for (int i = 0; i < 3; ++i) {
            const double uh = (un > 0.0) ? u[i] / un : 1.0; // one-sided slope at |u| = 0 (forward FD of the reference)
            bm[i] = -omega * c.cmdot * uh;
        }
    }
    LTO_HD int operator()(const double* y, double* dy) const {
        EPStage st;
        ep_stage<NS>(y, u, omega, mdot, c, dy, st);
        if (SENS) {
#pragma unroll 1
            for (int col = 0; col < NCOL; ++col) {
                const int bvc = col - NS;
                ep_col<NS>(st, omega, y + NS * (1 + col), bvc, bvc >= 0 ? bm[bvc] : 0.0, dy + NS * (1 + col));
            }
        }
        return 0;
    }
};

template <int ND, bool SENS>
struct SCRhs {
    static constexpr int NCOL = SENS ? ND : 0;
    static constexpr int NT = ND * (1 + NCOL);
    const SCConst& c;
    double thrustLimit, rho;
    LTO_HD SCRhs(const SCConst& c_, double tl, double rho_) : c(c_), thrustLimit(tl), rho(rho_) {}
    LTO_HD int operator()(const double* y, double* dy) const {
        SCStage st;
        if (sc_stage<ND>(y, c, thrustLimit, rho, dy, st)) return LTO_ST_BADP;
        if (SENS) {
#pragma unroll 1
            for (int col = 0; col < NCOL; ++col) sc_col<ND>(st, c.omega, y + ND * (1 + col), dy + ND * (1 + col));
        }
        return 0;
    }
};

// ---------------------------------------------------------------------------
// Drivers
// ---------------------------------------------------------------------------
// FIXED grid: ode7_8 (ode.jl:773-953) on tspan = LinRange(t0, t1, nsteps).  maxErr over
// the first NX components only (the reference integrates the bare state).
template <int NT, int NX, class RHS>
LTO_HD int drive_fixed(RHS& rhs, double* y, double t0, double t1, int nsteps, double* maxErr,
                       double* k, double* ytmp, double* ynew, double* gam) {
    double me = 0.0;
    int st = 0;
    for (int ind = 1; ind < nsteps; ++ind) {
        const double h = linrange_at(t0, t1, nsteps, ind) - linrange_at(t0, t1, nsteps, ind - 1);   // ode.jl:904
        st |= rkf78_step<NT>(rhs, y, h, ynew, gam, k, ytmp);
        double delta = 0.0;
        for (int c = 0; c < NX; ++c) delta = fmax(delta, fabs(gam[c]));                            // ode.jl:943
        if (delta > me) me = delta;                                                                // ode.jl:946-948
        for (int c = 0; c < NT; ++c) y[c] = ynew[c];
    }
    *maxErr = me;
    return st;
}

// Span rule of the adaptive controllers.  Their loop conditions (t < tfinal, h >= hmin) are false for a NaN end point and for a
// reversed span, so without this the leg would come back as x0 with status OK, never integrated: a non-finite end point is
// LTO_ST_NAN, tfinal < t0 is LTO_ST_HMIN (the leg does not reach its end time).  tfinal == t0 stays OK (x0, no attempts).
LTO_HD bool finite_time(double t) { return fabs(t) <= 1.7976931348623157e308; }   // false for +-inf and NaN
LTO_HD int span_status(double t0, double tfinal) {
    if (!(finite_time(t0) && finite_time(tfinal))) return LTO_ST_NAN;
    return (tfinal < t0) ? LTO_ST_HMIN : LTO_OK;
}

// ode78 controller (ode.jl:477-534).  NE = number of leading components the norms span.
template <int NT, class RHS>
LTO_HD int drive_ode78(RHS& rhs, double* y, double t0, double tfinal, double tol, int ne, int max_attempts,
                       int* nacc, int* natt, double* k, double* ytmp, double* ynew, double* gam) {
    const int ss = span_status(t0, tfinal);
    if (ss) { *nacc = 0; *natt = 0; return ss; }
    const double hmax = (tfinal - t0) / 2.5;
    double t = t0;
    const double hmin = (tfinal - t) / 1e7;
    double h = (tfinal - t) / 50.0;
    int na = 0, nt = 0, status = 0;
    while ((t < tfinal) && (h >= hmin)) {
        if (t + h > tfinal) h = tfinal - t;
        if (nt >= max_attempts) { status = LTO_ST_MAXSTEPS; break; }
        ++nt;
        const int rs = rkf78_step<NT>(rhs, y, h, ynew, gam, k, ytmp);
        if (rs) { status = rs; break; }
        double delta = 0.0, xn = 0.0;
        for (int c = 0; c < ne; ++c) { delta = fmax(delta, fabs(gam[c])); xn = fmax(xn, fabs(y[c])); }
        if (!(delta == delta)) { status = LTO_ST_NAN; break; }
        const double tau = tol * fmax(xn, 1.0);
        if (delta <= tau) {
            t += h;
            for (int c = 0; c < NT; ++c) y[c] = ynew[c];
            ++na;
        }
        if (delta == 0.0) delta = 1e-16;
        h = fmin(hmax, 0.8 * h * pow(tau / delta, 0.125));
    }
    if (status == 0 && t < tfinal) status = LTO_ST_HMIN;
    *nacc = na; *natt = nt;
    return status;
}

LTO_HD double inv_eighth_root(double e) { return sqrt(sqrt(sqrt(1.0 / e))); }

// Sharp-law safeguard of the STATE-ONLY controller (indirect path, p = 1: umag = aL (1 + tanh((|lv| - 1) / 2 rho)) / 2,
// CRTBP_stateCostate_deriv.jl:41-43).  Where a step crosses the switch |lv| = 1 the dominant error is quadrature-like (a sharp
// function of time integrated into v), and Fehlberg's 7(8) estimate is blind to exactly that (k1 = k12 and k11 = k13 for a pure
// quadrature).  With the sensitivities in the norm (ForwardDiff semantics) the 1/rho growth of Phi tightens the steps by itself
// and the pair behaves like DOP853 (measured on the converged rho = 1e-4 demo trajectory: 1e-10 .. 1e-8 both); the state-only
// controller instead runs at  tol * clamp(10 rho, 1e-3, 1):  rho = 1e-4 -> 1e-8 (was 5e-6), 1e-3 -> 1e-12 (was 8e-10).
LTO_HD double state_tol_scale(double p, double rho) { return (p == 1.0) ? fmin(1.0, fmax(10.0 * rho, 1e-3)) : 1.0; }

template <int NE>
LTO_HD double scaled_rms(const double* e, const double* a, const double* b, double atol, double rtol, int ne) {
    double s = 0.0;
    for (int c = 0; c < ne; ++c) {
        const double sc = fma(rtol, fmax(fabs(a[c]), fabs(b[c])), atol);
        const double q = e[c] / sc;
        s = fma(q, q, s);
    }
    return sqrt(s / (double)ne);
}

// OrdinaryDiffEq-style controller used for the indirect path (DESIGN.md "indirect controller"):
// scaled RMS error, accept iff <= 1, q = clamp(0.9*E^(-1/8), 0.2, 5), Hairer initial step.
template <int NT, class RHS>
//
// `robust` (the state-only norm, i.e. every call without sensitivities in the norm): the embedded Fehlberg estimate
// (41/840) h (k1 + k11 - k12 - k13) is the SUM of two differences, (k1 - k12) and (k11 - k13), which can cancel; with nothing but
// the 12 state components in the norm that let segments through with 300x the requested error (measured on config 4: up to 1e-9
// at 1e-13 where the control direction turns quickly, |lv| -> 0).  The state-only controller therefore takes, per component,
// max(|sum|, |k1 - k12|, |k11 - k13|) -- an upper bound of the same estimate that cannot cancel (same q formula).  With the
// sensitivities in the norm (ForwardDiff semantics, 156 components) the plain estimate is kept: it is accurate to 5e-13 there.
LTO_HD int drive_rk8(RHS& rhs, double* y, double t0, double tfinal, double atol, double rtol, int ne, int max_attempts,
                     int* nacc, int* natt, double* k, double* ytmp, double* ynew, double* gam, bool robust = false) {
    const double span = tfinal - t0;
    int na = 0, nt = 0, status = 0;
    *nacc = 0; *natt = 0;
    const int ss = span_status(t0, tfinal);          // same span rule as drive_ode78
    if (ss) return ss;
    // initial step: f0 -> k[0..NT), euler probe -> k[NT..2NT)
    int rs = rhs(y, k);
    if (rs) return rs;
    const double d0 = scaled_rms<0>(y, y, y, atol, rtol, ne);
    const double d1 = scaled_rms<0>(k, y, y, atol, rtol, ne);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * (d0 / d1);
    h0 = fmin(h0, span);
    for (int c = 0; c < NT; ++c) ytmp[c] = fma(h0, k[c], y[c]);
    rs = rhs(ytmp, k + NT);
    if (rs) return rs;
    for (int c = 0; c < ne; ++c) gam[c] = k[NT + c] - k[c];
    const double d2 = scaled_rms<0>(gam, y, y, atol, rtol, ne) / h0;
    const double dm = fmax(d1, d2);
    const double h1 = (dm <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : inv_eighth_root(dm / 0.01);
    double h = fmin(fmin(100.0 * h0, h1), span);
    const double hmin = span * 1e-12;
    double t = t0;
    bool last_rejected = false;
    while (t < tfinal) {
        if (h < hmin) { status = LTO_ST_HMIN; break; }
        if (nt >= max_attempts) { status = LTO_ST_MAXSTEPS; break; }
        bool last = false;
        if (t + h >= tfinal) { h = tfinal - t; last = true; }
        ++nt;
        rs = rkf78_step<NT>(rhs, y, h, ynew, gam, k, ytmp);
        if (rs) { status = rs; break; }
        if (robust) {
            const double ce = h * lto_tab::ERRC;
            for (int c = 0; c < ne; ++c) {
                const double ga = ce * (k[0 * NT + c] - k[11 * NT + c]), gb = ce * (k[10 * NT + c] - k[12 * NT + c]);
                gam[c] = fmax(fabs(gam[c]), fmax(fabs(ga), fabs(gb)));          // NaN in gam[c] must survive: fmax drops it
                if (!(ga + gb == ga + gb)) gam[c] = ga + gb;
            }
        }
        const double eest = scaled_rms<0>(gam, y, ynew, atol, rtol, ne);
        if (!(eest == eest)) { status = LTO_ST_NAN; break; }
        double q = (eest == 0.0) ? 5.0 : 0.9 * inv_eighth_root(eest);
        q = fmin(5.0, fmax(0.2, q));
        if (eest <= 1.0) {
            ++na;
            for (int c = 0; c < NT; ++c) y[c] = ynew[c];
            if (last) { t = tfinal; break; }
            t += h;
            if (last_rejected) q = fmin(q, 1.0);
            last_rejected = false;
        } else {
            last_rejected = true;
            q = fmin(q, 1.0);
        }
        h = h * q;
    }
    *nacc = na; *natt = nt;
    return status;
}

// ---------------------------------------------------------------------------
// One leg of a direct segment (multiShoot_CRTBP_direct.jl:82-98).
//   backward != 0: flip the velocity of x0, omega = -1, same positive time grid,
//   and flip the velocity of the result back (:92,:98).  The sensitivity block is
//   returned already in the defect's frame:  out = R S [R | I]  (SURVEY A.3), so the
//   caller only has to subtract.
// S (if SENS): NS x (NS+3) column-major.
// ---------------------------------------------------------------------------
struct DirectCfg { int mode; int nsteps; double tol; int err_norm; int max_attempts; };

template <int NS, bool SENS>
LTO_HD int ep_leg(const double* x0, const double* u, int backward, double t0, double t1, const DirectCfg& cfg,
                  const EPConst& c, double* xend, double* S, double* maxErr, int* natt) {
    typedef EPRhs<NS, SENS> R;
    constexpr int NT = R::NT;
    double y[NT], ynew[NT], gam[NT], ytmp[NT], k[13 * NT];
    const double omega = backward ? -1.0 : 1.0;
    for (int i = 0; i < NS; ++i) y[i] = x0[i];
    if (backward) { y[3] = -y[3]; y[4] = -y[4]; y[5] = -y[5]; }
    if (SENS) {
        for (int i = NS; i < NT; ++i) y[i] = 0.0;
        for (int j = 0; j < NS; ++j) y[NS * (1 + j) + j] = 1.0;
    }
    R rhs(c, u, omega);
    int st, na = 0, nt = 0;
    if (cfg.mode == 0) {
        st = drive_fixed<NT, NS>(rhs, y, t0, t1, cfg.nsteps, maxErr, k, ytmp, ynew, gam);
        nt = cfg.nsteps - 1;
    } else {
        *maxErr = 0.0;
        st = drive_ode78<NT>(rhs, y, t0, t1, cfg.tol, (SENS && cfg.err_norm) ? NT : NS, cfg.max_attempts, &na, &nt,
                             k, ytmp, ynew, gam);
    }
    *natt = nt;
    for (int i = 0; i < NS; ++i) xend[i] = y[i];
    if (backward) { xend[3] = -xend[3]; xend[4] = -xend[4]; xend[5] = -xend[5]; }
    if (SENS) {
        for (int j = 0; j < NS + 3; ++j)
            for (int i = 0; i < NS; ++i) {
                double v = y[NS * (1 + j) + i];
                if (backward) {
                    const bool fi = (i >= 3 && i < 6), fj = (j >= 3 && j < 6);
                    if (fi != fj) v = -v;          // R S R on state columns, R S on control columns
                }
                S[j * NS + i] = v;
            }
    }
    for (int i = 0; i < NS; ++i) if (!(xend[i] == xend[i])) st = st ? st : LTO_ST_NAN;
    return st;
}

// ---------------------------------------------------------------------------
// One indirect segment t0 -> t1 (multiShoot_CRTBP_indirect.jl:75-79 / :103-111).
// Phi (if SENS): ND x ND column-major.
// ---------------------------------------------------------------------------
struct IndirectCfg { double atol, rtol; int controller; int err_norm; int max_attempts; };

template <int ND, bool SENS>
LTO_HD int sc_seg(const double* x0, double t0, double t1, const IndirectCfg& cfg, const SCConst& c,
                  double thrustLimit, double rho, double* xend, double* Phi, int* nacc, int* natt) {
    typedef SCRhs<ND, SENS> R;
    constexpr int NT = R::NT;
    double y[NT], ynew[NT], gam[NT], ytmp[NT], k[13 * NT];
    for (int i = 0; i < ND; ++i) y[i] = x0[i];
    if (SENS) {
        for (int i = ND; i < NT; ++i) y[i] = 0.0;
        for (int j = 0; j < ND; ++j) y[ND * (1 + j) + j] = 1.0;
    }
    R rhs(c, thrustLimit, rho);
    const int ne = (SENS && cfg.err_norm) ? NT : ND;
    int st;
    const double ts = (ne == ND) ? state_tol_scale(c.p, rho) : 1.0;
    if (cfg.controller == 0) st = drive_rk8<NT>(rhs, y, t0, t1, cfg.atol * ts, cfg.rtol * ts, ne, cfg.max_attempts, nacc, natt, k, ytmp, ynew, gam, ne == ND);
    else                     st = drive_ode78<NT>(rhs, y, t0, t1, cfg.rtol, ne, cfg.max_attempts, nacc, natt, k, ytmp, ynew, gam);
    for (int i = 0; i < ND; ++i) xend[i] = y[i];
    if (SENS) for (int i = 0; i < ND * ND; ++i) Phi[i] = y[ND + i];
    for (int i = 0; i < ND; ++i) if (!(xend[i] == xend[i])) st = st ? st : LTO_ST_NAN;
    return st;
}

}  // namespace lto
