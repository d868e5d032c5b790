// lto_switch.h -- the switch times of the p = 1 control law (CRTBP_stateCostate_deriv.jl:36-53) on one integration step, compiled for
// the host (tests) and the device (K4's switch pass, lto_indirect_cw.cu).
//
// Switching function S(t) = |lv(t)| - 1: the thrust is "on" where S > 0 and "off" where S <= 0 (zero counts as off).  n = |lv| is
// formed as sc_stage forms it (sqrt of the fma sum), so a node state is on the same side here and in the kernel.  S is smooth where the
// throttle is sharp: lv' = -lr - C^T lv and lr' = -U(r) lv, so the thrust reaches lv only through U(r), two integrations away.
//
//   sw_end    lv, lv' and lv'' = U(r) lv - C^T lv' of a 12-dim state [r v lr lv] (U: grav_eval's gravity gradient, omega as sc_stage)
//   sw_eval   the quintic Hermite interpolant of lv on a step [t, t + h] in theta in [0, 1] from both ends' (lv, h lv', h^2 lv'')
//   sw_scan   S on the interpolant at theta = k/8, k = 0..8 (the ends from the exact end states, so a step's last sample is the next
//             step's first), every bracket with a sign change refined by Newton on the polynomial safeguarded by bisection; writes at
//             most `cap` (time, direction) pairs after the `count` already found and returns the new count (it counts past `cap`).
//             Direction +1: off -> on (a burn starts), -1: on -> off.  A touch with no sign change between samples is not a switch.
#pragma once
#include <math.h>
#include <stdint.h>
#include "lto_math.cuh"

#if defined(__CUDACC__)
#define LTO_SW_FN __host__ __device__ inline
#else
#define LTO_SW_FN inline
#endif

#define LTO_SW_SAMPLES 8             // samples per step: theta = k / 8
#define LTO_SW_MAX_IT 64             // iteration cap of one root's refinement

struct SwEnd { double lv[3], ld[3], la[3]; };   // lv, lv', lv'' at one end of a step (per unit time, not scaled by h)

// n = |lv| as sc_stage forms it; the side of S = n - 1: on (1) where n > 1
LTO_SW_FN double sw_norm(double l0, double l1, double l2) { return sqrt(fma(l0, l0, fma(l1, l1, l2 * l2))); }
LTO_SW_FN int sw_side(double l0, double l1, double l2) { return sw_norm(l0, l1, l2) > 1.0 ? 1 : 0; }

// x = [r v lr lv] (12): lv' = -lr - C^T lv (CRTBP_stateCostate_deriv.jl:86-88), lv'' = -lr' - C^T lv' = U lv - C^T lv'
LTO_SW_FN void sw_end(double r0, double r1, double r2, double lr0, double lr1, double lr2, double lv0, double lv1, double lv2, double mu,
                      double m1, double omega, SwEnd& e) {
    lto::Grav g;
    lto::grav_eval(r0, r1, r2, mu, m1, g);
    const double w2 = 2.0 * omega;
    e.lv[0] = lv0; e.lv[1] = lv1; e.lv[2] = lv2;
    e.ld[0] = fma(w2, lv1, -lr0);
    e.ld[1] = fma(-w2, lv0, -lr1);
    e.ld[2] = -lr2;
    double Ul[3];
    lto::sym3_mul(g.U, e.lv, Ul);
    e.la[0] = fma(w2, e.ld[1], Ul[0]);
    e.la[1] = fma(-w2, e.ld[0], Ul[1]);
    e.la[2] = Ul[2];
}

// Coefficients c[q][0..5] of p_q(theta) = sum_k c_k theta^k with p(0) = lv0, p'(0) = h lv0', p''(0) = h^2 lv0'' and the same at theta = 1
LTO_SW_FN void sw_fit(const SwEnd& e0, const SwEnd& e1, double h, double (&c)[3][6]) {
    const double h2 = h * h;
    for (int q = 0; q < 3; ++q) {
        const double dp = e1.lv[q] - e0.lv[q];
        const double d0 = h * e0.ld[q], d1 = h * e1.ld[q];
        const double a0 = h2 * e0.la[q], a1 = h2 * e1.la[q];
        c[q][0] = e0.lv[q];
        c[q][1] = d0;
        c[q][2] = 0.5 * a0;
        c[q][3] = fma(10.0, dp, fma(-6.0, d0, fma(-4.0, d1, 0.5 * (a1 - 3.0 * a0))));
        c[q][4] = fma(-15.0, dp, fma(8.0, d0, fma(7.0, d1, 0.5 * (3.0 * a0 - 2.0 * a1))));
        c[q][5] = fma(6.0, dp, fma(-3.0, d0, fma(-3.0, d1, 0.5 * (a1 - a0))));
    }
}

// p(theta) and dp/dtheta by Horner
LTO_SW_FN void sw_eval(const double (&c)[3][6], double th, double (&p)[3], double (&dp)[3]) {
    for (int q = 0; q < 3; ++q) {
        double v = c[q][5], d = 5.0 * c[q][5];
        v = fma(v, th, c[q][4]); d = fma(d, th, 4.0 * c[q][4]);
        v = fma(v, th, c[q][3]); d = fma(d, th, 3.0 * c[q][3]);
        v = fma(v, th, c[q][2]); d = fma(d, th, 2.0 * c[q][2]);
        v = fma(v, th, c[q][1]); d = fma(d, th, c[q][1]);
        v = fma(v, th, c[q][0]);
        p[q] = v; dp[q] = d;
    }
}

// The root of S in (a, b), side(a) = sa, side(b) = !sa: Newton on n(theta) - 1, a step that leaves the bracket replaced by bisection;
// stops when the bracket or the Newton step is within a few ulp of theta, or after LTO_SW_MAX_IT iterations.
LTO_SW_FN double sw_refine(const double (&c)[3][6], double a, double b, int sa) {
    double th = 0.5 * (a + b);
    for (int it = 0; it < LTO_SW_MAX_IT; ++it) {
        double p[3], dp[3];
        sw_eval(c, th, p, dp);
        const double n = sw_norm(p[0], p[1], p[2]);
        if ((n > 1.0 ? 1 : 0) == sa) a = th; else b = th;
        const double tol = 4.0 * 2.220446049250313e-16 * fmax(fabs(a), fabs(b));
        if (!(b - a > tol)) break;
        const double dn = fma(p[0], dp[0], fma(p[1], dp[1], p[2] * dp[2])) / n;
        double tn = th - (n - 1.0) / dn;
        if (!(tn > a && tn < b)) tn = 0.5 * (a + b);
        const double step = fabs(tn - th);
        th = tn;
        if (!(step > tol)) break;
    }
    return th;
}

// The switches of one step [t, t + h] from its end values; see the top of the file.
LTO_SW_FN int sw_scan(const SwEnd& e0, const SwEnd& e1, double t, double h, int count, int cap, double* t_out, int32_t* dir_out) {
    double c[3][6];
    sw_fit(e0, e1, h, c);
    int s_prev = sw_side(e0.lv[0], e0.lv[1], e0.lv[2]);
    for (int k = 1; k <= LTO_SW_SAMPLES; ++k) {
        const double th1 = (double)k * (1.0 / LTO_SW_SAMPLES);
        int s;
        if (k == LTO_SW_SAMPLES) {
            s = sw_side(e1.lv[0], e1.lv[1], e1.lv[2]);
        } else {
            double p[3], dp[3];
            sw_eval(c, th1, p, dp);
            s = sw_side(p[0], p[1], p[2]);
        }
        if (s != s_prev) {
            const double th = sw_refine(c, (double)(k - 1) * (1.0 / LTO_SW_SAMPLES), th1, s_prev);
            if (count < cap) { t_out[count] = fma(th, h, t); dir_out[count] = s ? 1 : -1; }
            ++count;
        }
        s_prev = s;
    }
    return count;
}
