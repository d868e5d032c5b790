// lto_direct_cw.cu -- throughput kernel for the direct method, FIXED grid (K1):
// defectCalc + jacobianCalc of multiShoot_CRTBP_direct.jl:66-143 for a whole batch in one
// launch, with the variational equations in place of the reference's 2(n+3) finite-
// difference re-propagations.
//
// Mapping ("column-warp" layout, DESIGN.md section 4):
//   CTA  = 32 legs (16 segments: lane 2k = forward leg, lane 2k+1 = backward leg of one segment)
//   warp = one column of the augmented system:  warp XW carries the state x itself,
//          every other warp carries one column of S = [Phi | Gamma]  (n + 3 columns)
//   lane = leg.  Nothing is ever exchanged between lanes except the final defect.
// A state warp evaluates the nonlinear dynamics once per RK stage and leg and publishes
// the stage's linearisation (U_xx, k/m, -k u/m^2) through shared memory; the column warps
// apply it to their column.  The state does not depend on S, so a state warp runs AHEAD of
// the column warps through a 2-slot ring of step records guarded by mbarriers (full: the
// state warp's 32 lanes arrive; empty: every column thread arrives) -- no CTA-wide barrier.
// One RK step of the state is a long dependent chain (ncu, profiles/: ~4 cycles/instruction,
// never waiting), so a CTA keeps TWO tiles in flight, each with its own state warp; the
// column warps alternate between them step by step, which hides the state chain behind
// two column phases and fills the FP64 pipe.
// Stage storage: Nystrom form -- only the 3 acceleration components of each stage are
// kept (registers), positions are rebuilt with G = B*B (lto_tableau.h).  Stage 11 is
// needed by the error estimate only (ode.jl:892), which the reference takes over the
// state alone (ode.jl:940-943), so column warps skip it.
#include "lto_internal.h"
#include "lto_cw_common.cuh"
#include <algorithm>

namespace lto {

namespace cw {

constexpr int NTILE = 2;   // tiles in flight per CTA (one state warp each)
constexpr int NSLOT = 2;   // ring depth of step records per tile
// warps 2 and 3 are the state warps: with warp w on SM sub-partition w % 4 the FP64 load is
// [3 col | 3 col | state + 2 col | state + 2 col] (nstate 7), i.e. balanced
constexpr int XW0 = 2;

template <int NS>
struct Cfg {
    static constexpr int NCOL = NS + 3;
    static constexpr int NW = NTILE + NCOL;
    static constexpr int NTHREADS = 32 * NW;
    static constexpr int SVAL = (NS == 7) ? 10 : 6;          // U[6] (+ k/m, am[3]) per stage and leg, lane-contiguous (128-bit accesses)
    static constexpr int OFF_H = 13 * SVAL;                  // h (lane-strided, as bm)
    static constexpr int OFF_BM = OFF_H + 1;                 // bm[3] (nstate 7)
    static constexpr int STEP_DOUBLES = OFF_BM + ((NS == 7) ? 3 : 0);
    static constexpr size_t REC_BYTES = (size_t)NTILE * NSLOT * STEP_DOUBLES * 32 * sizeof(double);
    static constexpr int NV = 2 * (NS + 3);
    static constexpr size_t OUT_TILE_BYTES = (size_t)16 * NS * NV * sizeof(double);      // one tile's Jacobian blocks, in the output's own layout
    static constexpr size_t OUT_BYTES = (size_t)NTILE * OUT_TILE_BYTES;
    static constexpr size_t BAR_OFF = REC_BYTES + OUT_BYTES;
    static constexpr size_t FLAG_OFF = BAR_OFF + (size_t)NTILE * NSLOT * 2 * sizeof(unsigned long long);
    static constexpr size_t PARK_OFF = (FLAG_OFF + (size_t)NTILE * NSLOT * sizeof(int) + 15) & ~(size_t)15;   // after the ADAPTIVE "last step" flags
    static constexpr int NPARK = (NS == 7) ? 7 : 6;                                    // sr[3] sv[3] (sm) of one column thread
    static constexpr size_t SMEM = PARK_OFF + (size_t)NTILE * NCOL * NPARK * 32 * sizeof(double);   // column state of every tile, lane-strided
};

// ---------------------------------------------------------------------------
// -DLTO_K1_PROF: per-warp clock64() spans of K1 / K2, written to k1_prof[block][warp][K1P_N] when the warp retires
// (tools/k1_phase_clocks.py reads them through lto_k1_prof_read).  Without the switch every method is empty.
// ---------------------------------------------------------------------------
enum { K1P_WORK, K1P_BAR, K1P_PACE, K1P_STORE, K1P_TOTAL, K1P_STEPS, K1P_N };
#ifdef LTO_K1_PROF
constexpr int K1P_MAX_BLOCKS = 1024, K1P_MAX_WARPS = 16;
__device__ unsigned long long k1_prof[K1P_MAX_BLOCKS * K1P_MAX_WARPS * K1P_N];
struct K1Prof {
    long long c[K1P_N], t, t_begin;
    __device__ __forceinline__ void start() {
        for (int i = 0; i < K1P_N; ++i) c[i] = 0;
        t = t_begin = clock64();
    }
    __device__ __forceinline__ void mark() { t = clock64(); }
    __device__ __forceinline__ void add(int i) { const long long n = clock64(); c[i] += n - t; t = n; }
    __device__ __forceinline__ void step() { ++c[K1P_STEPS]; }
    __device__ __forceinline__ void flush(int warp, int lane) {
        c[K1P_TOTAL] = clock64() - t_begin;
        if (lane == 0 && blockIdx.x < K1P_MAX_BLOCKS)
            for (int i = 0; i < K1P_N; ++i) k1_prof[((size_t)blockIdx.x * K1P_MAX_WARPS + warp) * K1P_N + i] = (unsigned long long)c[i];
    }
};
#else
struct K1Prof {
    __device__ __forceinline__ void start() {}
    __device__ __forceinline__ void mark() {}
    __device__ __forceinline__ void add(int) {}
    __device__ __forceinline__ void step() {}
    __device__ __forceinline__ void flush(int, int) {}
};
#endif

using namespace cwc;

// ---------------------------------------------------------------------------
// State warp: one RK step of x = [r v (m)] in Nystrom form; publishes h into `rec` (lane-strided)
// and the stage linearisations of this step into `stg` (lane-contiguous), and accumulates maxErr.
// ---------------------------------------------------------------------------
template <int NS, bool PUB = true>
__device__ __forceinline__ double x_step(double (&r)[3], double (&v)[3], double& m, const double (&u)[3], double omega,
                                         double mdot, double h, const EPConst& c, double* __restrict__ rec, double* __restrict__ stg,
                                         double& maxErr) {
    constexpr int SVAL = Cfg<NS>::SVAL;
    const double h2 = h * h;
    const double w2 = 2.0 * omega;
    const double kom6 = c.kthr / c.default_mass;
    double a[13][3];
    double ev[3] = {0.0, 0.0, 0.0}, ea[3] = {0.0, 0.0, 0.0};
    if (PUB) rec[Cfg<NS>::OFF_H * 32] = h;
#pragma unroll
    for (int j = 0; j < 13; ++j) {
        double R[3], V[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            double accv = 0.0, accr = 0.0;
#pragma unroll
            for (int l = 0; l < j; ++l) {
                if (lto_tab::Bf(j, l) != 0.0) accv = fma(lto_tab::Bf(j, l), a[l][q], accv);
                if (lto_tab::Gf(j, l) != 0.0) accr = fma(lto_tab::Gf(j, l), a[l][q], accr);
            }
            V[q] = (j == 0) ? v[q] : fma(h, accv, v[q]);
            R[q] = (j == 0) ? r[q] : fma(h2, accr, fma(h * lto_tab::Cf(j), v[q], r[q]));
        }
        // ---- gravity: 1/r_b^3 (CRTBP_prop_EP_deriv.jl:24-29) and the gradient U_xx
        const double dx1 = R[0] + c.mu, dx2 = dx1 - 1.0;
        const double yz = fma(R[1], R[1], R[2] * R[2]);
        const double i1 = fast_rsqrt(fma(dx1, dx1, yz));
        const double i2 = fast_rsqrt(fma(dx2, dx2, yz));
        const double i1s = i1 * i1, i2s = i2 * i2;
        const double a31 = c.m1 * i1s * i1, a32 = c.mu * i2s * i2;
        const double gg1 = 1.0 - (a31 + a32);                       // 1 + g
        double kom = kom6, im = 0.0;
        if (NS == 7) { im = fast_rcp(fma(h * lto_tab::Cf(j), mdot, m)); kom = c.kthr * im; }
        // ---- acceleration (CRTBP_prop_EP_deriv.jl:48-50), thrust u*k/m (:32-38)
        a[j][0] = fma(u[0], kom, fma(-a31, dx1, fma(-a32, dx2, fma(w2, V[1], R[0]))));
        a[j][1] = fma(u[1], kom, fma(gg1, R[1], -w2 * V[0]));
        a[j][2] = fma(u[2], kom, (gg1 - 1.0) * R[2]);
        if (PUB && j != 10) {
            const double a51 = 3.0 * i1s * a31, a52 = 3.0 * i2s * a32;
            const double s5 = a51 + a52;
            const double p1 = a51 * dx1, p2 = a52 * dx2;
            const double t = p1 + p2;
            const double s5y = s5 * R[1];
            double2* w = reinterpret_cast<double2*>(stg + j * SVAL * 32);
            w[0] = make_double2(fma(p1, dx1, fma(p2, dx2, gg1)), fma(s5y, R[1], gg1));
            w[1] = make_double2(fma(s5 * R[2], R[2], gg1 - 1.0), t * R[1]);
            w[2] = make_double2(t * R[2], s5y * R[2]);
            if (NS == 7) {
                const double k2 = -kom * im;
                w[3] = make_double2(kom, k2 * u[0]);
                w[4] = make_double2(k2 * u[1], k2 * u[2]);
            }
        }
        if (lto_tab::PSIf(j) != 0.0) {
#pragma unroll
            for (int q = 0; q < 3; ++q) { ev[q] = fma(lto_tab::PSIf(j), V[q], ev[q]); ea[q] = fma(lto_tab::PSIf(j), a[j][q], ea[q]); }
        }
    }
    double delta = 0.0;
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        double sv = 0.0, sr = 0.0;
#pragma unroll
        for (int l = 0; l < 13; ++l) {
            if (lto_tab::CHIf(l) != 0.0) sv = fma(lto_tab::CHIf(l), a[l][q], sv);
            if (lto_tab::CHIBf(l) != 0.0) sr = fma(lto_tab::CHIBf(l), a[l][q], sr);
        }
        r[q] = fma(h2, sr, fma(h, v[q], r[q]));
        v[q] = fma(h, sv, v[q]);
        delta = fmax(delta, fmax(fabs(ev[q]), fabs(ea[q])));
    }
    if (NS == 7) m = fma(h, mdot, m);
    delta *= fabs(h * lto_tab::ERRC);                       // ode.jl:940-943 (mass row is identically 0)
    maxErr = fmax(maxErr, delta);                           // ode.jl:946-948
    return delta;
}

// ---------------------------------------------------------------------------
// Column warp: one RK step of one column s = [s_r s_v (s_m)] of S = [Phi | Gamma].
// ONE instruction stream serves every column (the instruction cache is shared by the
// whole SM): what distinguishes the columns is data --
//   Phi column of r or v : s_m == 0,            no forcing      (bm = 0, gc < 0)
//   Phi column of m      : s_m == 1,            no forcing      (bm = 0, gc < 0, sm = 1)
//   Gamma column gc      : s_m = bm*(t - t0),   forcing (k/m) e_gc on s_v, bm on s_m
// MASS = (NS == 7): rows/columns of the mass exist.  `rec`: h (lane-strided), `stg`: this lane's stage records.
// ---------------------------------------------------------------------------
template <int NS>
__device__ __forceinline__ void col_step(double (&sr)[3], double (&sv)[3], double& sm, double bm, int gc,
                                         double omega, double kom6, const double* __restrict__ rec, const double* __restrict__ stg) {
    constexpr int SVAL = Cfg<NS>::SVAL;
    constexpr bool MASS = (NS == 7);
    const double h = rec[Cfg<NS>::OFF_H * 32];
    const double h2 = h * h;
    const double w2 = 2.0 * omega;
    double a[13][3];
#pragma unroll
    for (int j = 0; j < 13; ++j) {
        if (j == 10) continue;
        double R[3], V[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            double accv = 0.0, accr = 0.0;
#pragma unroll
            for (int l = 0; l < j; ++l) {
                if (lto_tab::Bf(j, l) != 0.0) accv = fma(lto_tab::Bf(j, l), a[l][q], accv);
                if (lto_tab::Gf(j, l) != 0.0) accr = fma(lto_tab::Gf(j, l), a[l][q], accr);
            }
            V[q] = (j == 0) ? sv[q] : fma(h, accv, sv[q]);
            R[q] = (j == 0) ? sr[q] : fma(h2, accr, fma(h * lto_tab::Cf(j), sv[q], sr[q]));
        }
        const double2* w = reinterpret_cast<const double2*>(stg + j * SVAL * 32);
        const double2 w0 = w[0], w1 = w[1], w2v = w[2];
        const double U[6] = {w0.x, w0.y, w1.x, w1.y, w2v.x, w2v.y};
        double2 w3 = make_double2(kom6, 0.0), w4 = make_double2(0.0, 0.0);
        if (MASS) { w3 = w[3]; w4 = w[4]; }
        const double kom = w3.x;
        // forcing (k/m) e_gc: selected, not multiplied by a unit vector (w2 = +-2, so w2 * V is exact and the sums are unchanged)
        double acc[3];
        acc[0] = fma(w2, V[1], gc == 0 ? kom : 0.0);
        acc[1] = fma(-w2, V[0], gc == 1 ? kom : 0.0);
        acc[2] = gc == 2 ? kom : 0.0;
        if (MASS) {
            const double smj = fma(h * lto_tab::Cf(j), bm, sm);
            const double am[3] = {w3.y, w4.x, w4.y};
#pragma unroll
            for (int q = 0; q < 3; ++q) acc[q] = fma(am[q], smj, acc[q]);
        }
        sym3_mul_acc(U, R, acc);
#pragma unroll
        for (int q = 0; q < 3; ++q) a[j][q] = acc[q];
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        double dv = 0.0, dr = 0.0;
#pragma unroll
        for (int l = 0; l < 13; ++l) {
            if (lto_tab::CHIf(l) != 0.0) dv = fma(lto_tab::CHIf(l), a[l][q], dv);
            if (lto_tab::CHIBf(l) != 0.0) dr = fma(lto_tab::CHIBf(l), a[l][q], dr);
        }
        sr[q] = fma(h2, dr, fma(h, sv[q], sr[q]));
        sv[q] = fma(h, dv, sv[q]);
    }
    if (MASS) sm = fma(h, bm, sm);
}

// One column thread's state for one tile in flight.  Between its steps it is parked in shared memory (lane-strided), so a
// column thread holds one tile's state in registers, not NTILE.
struct ColState { double sr[3], sv[3], sm; };

template <int NS>
__device__ __forceinline__ void col_init(ColState& c, int col) {
#pragma unroll
    for (int q = 0; q < 3; ++q) { c.sr[q] = (col == q) ? 1.0 : 0.0; c.sv[q] = (col == q + 3) ? 1.0 : 0.0; }
    c.sm = (NS == 7 && col == 6) ? 1.0 : 0.0;                // S(0) = [I | 0]
}

template <int NS>
__device__ __forceinline__ void col_park(double* __restrict__ p, const ColState& c) {
#pragma unroll
    for (int q = 0; q < 3; ++q) { p[q * 32] = c.sr[q]; p[(3 + q) * 32] = c.sv[q]; }
    if (NS == 7) p[6 * 32] = c.sm;
}

template <int NS>
__device__ __forceinline__ void col_unpark(const double* __restrict__ p, ColState& c) {
#pragma unroll
    for (int q = 0; q < 3; ++q) { c.sr[q] = p[q * 32]; c.sv[q] = p[(3 + q) * 32]; }
    c.sm = (NS == 7) ? p[6 * 32] : 0.0;
}

// Store this column of the segment's Jacobian block, in the defect's frame:
//   forward leg  +S        -> columns [X_a | u_a]
//   backward leg -(R S R)  -> columns [X_b]      -(R S) -> [u_b]      (SURVEY A.3)
template <int NS>
__device__ __forceinline__ void col_store(double* __restrict__ stage, const ColState& c, int col, int lane) {
    constexpr int NV = 2 * (NS + 3);
    const int back = lane & 1, gc = col - NS;
    const int ocol = (gc >= 0) ? (2 * NS + (back ? 3 : 0) + gc) : ((back ? NS : 0) + col);
    double* J = stage + (lane >> 1) * (NS * NV) + ocol * NS;
    const double rj = (col >= 3 && col < 6) ? -1.0 : 1.0;
    const double sp = back ? -rj : 1.0;       // sign of the r / m rows
    const double sq = back ? rj : 1.0;        // sign of the v rows
    J[0] = sp * c.sr[0]; J[1] = sp * c.sr[1]; J[2] = sp * c.sr[2];
    J[3] = sq * c.sv[0]; J[4] = sq * c.sv[1]; J[5] = sq * c.sv[2];
    if (NS == 7) J[6] = sp * c.sm;
}

// This column thread's parked state of tile t.
template <int NS>
__device__ __forceinline__ double* col_park_at(double* parks, int t, int col, int lane) {
    return parks + (size_t)(t * Cfg<NS>::NCOL + col) * Cfg<NS>::NPARK * 32 + lane;
}

// One column step of tile t: wait for the state warp's record, step the parked column, release the record.
// ADAPT: returns whether this was the tile's last step (K2's per-slot flag).
template <int NS, bool ADAPT>
__device__ __forceinline__ bool col_tile_step(int t, unsigned g, int col, int gc, int lane, double omega, double kom6, double* recs, double* parks,
                                              unsigned bars, volatile int* lastf, K1Prof& pf) {
    typedef Cfg<NS> C;
    const unsigned slot = g & (NSLOT - 1), par = (g / NSLOT) & 1;
    const double* slotp = recs + (size_t)(t * NSLOT + slot) * C::STEP_DOUBLES * 32;
    const double* rec = slotp + lane;
    const unsigned full = bars + (unsigned)((t * NSLOT + slot) * 16), empty = full + 8;
    mbar_wait(full, par);
    pf.add(K1P_BAR);
    double* park = col_park_at<NS>(parks, t, col, lane);
    ColState cs;
    col_unpark<NS>(park, cs);
    const double bm = (NS == 7 && gc >= 0) ? rec[(C::OFF_BM + gc) * 32] : 0.0;   // the state warp republishes bm with every step
    const bool last = ADAPT && lastf[t * NSLOT + slot] != 0;
    col_step<NS>(cs.sr, cs.sv, cs.sm, bm, gc, omega, kom6, rec, slotp + lane * C::SVAL);
    mbar_arrive(empty);
    col_park<NS>(park, cs);
    pf.add(K1P_WORK);
    pf.step();
    return last;
}

// Both tiles of the pair are through: their 16 Jacobian blocks each are one contiguous run of the output.  Stage them in shared memory in
// the output's own layout and let the TMA engine write each run (one bulk store, fully coalesced, also when `jac` is NVLink peer memory of
// another GPU).
template <int NS>
__device__ __forceinline__ void col_tiles_store(const DirectArgs& a, long long pair, int col, int lane, double* outs, double* parks) {
    typedef Cfg<NS> C;
    const bool leader = (col == 0 && lane == 0);
#pragma unroll 1
    for (int t = 0; t < NTILE; ++t) {
        const long long seg0 = (pair * NTILE + t) * 16;
        double* stage = outs + (size_t)t * (C::OUT_TILE_BYTES / sizeof(double));
        // the previous store from THIS buffer has been read out: it is the oldest of the NTILE stores in flight (one per tile and
        // pair, issued in tile order), so the younger ones -- the other tile's, issued a moment ago -- need not be waited for.
        // Matters when `jac` is peer memory behind a saturated NVLink port (8 GPUs delivering to one): a store then takes tens
        // of microseconds to leave, and waiting for all of them stalled the CTA once per tile.
        if (leader) bulk_store_wait_read_but<NTILE - 1>();
        asm volatile("bar.sync 2, %0;" ::"n"(32 * C::NCOL) : "memory");
        ColState cs;
        col_unpark<NS>(col_park_at<NS>(parks, t, col, lane), cs);
        col_store<NS>(stage, cs, col, lane);
        fence_proxy_async();
        asm volatile("bar.sync 2, %0;" ::"n"(32 * C::NCOL) : "memory");
        if (leader && seg0 < a.n_seg) {
            const long long nseg = (a.n_seg - seg0 < 16) ? (a.n_seg - seg0) : 16;
            bulk_store(a.jac + seg0 * (long long)(NS * C::NV), smem_u32(stage), (unsigned)(nseg * NS * C::NV * sizeof(double)));
        }
    }
}

template <int NS>
__device__ __forceinline__ void column_warp(const DirectArgs& a, long long n_tiles, int warp, int col, int lane, double* recs, double* outs, double* parks,
                                            unsigned bars) {
    typedef Cfg<NS> C;
    const int nstep = a.cfg.nsteps - 1;
    const double omega = (lane & 1) ? -1.0 : 1.0;
    const double kom6 = a.c.kthr / a.c.default_mass;
    const int gc = col - NS;                             // >= 0: control component of a Gamma column
    K1Prof pf;
    pf.start();
    unsigned g = 0;                                      // step counter of each tile stream (same for both)
    for (long long pair = blockIdx.x; pair * NTILE < n_tiles; pair += gridDim.x) {
#pragma unroll 1
        for (int t = 0; t < NTILE; ++t) { ColState c; col_init<NS>(c, col); col_park<NS>(col_park_at<NS>(parks, t, col, lane), c); }
        for (int k = 0; k < nstep; ++k, ++g) {
            pf.mark();
#ifndef LTO_K1_NO_PACE
            // the column warps walk the step body together (shared instruction fetches): without this the column warp that shares its
            // sub-partition with a state warp and no second column warp (nstate 6) runs ahead and the instruction-cache hit rate drops
            // (78 % against 95 %).  Measured: nstate 6 0.707 -> 0.611 ms, nstate 7 unchanged (0.682 ms); a second barrier between the two
            // tiles of a step is no better for 6 and costs 8 % for 7.
            asm volatile("bar.sync 3, %0;" ::"n"(32 * C::NCOL) : "memory");
#endif
            pf.add(K1P_PACE);
            // one copy of the step body for both tiles: half the instruction footprint, and only one tile's column state live
#pragma unroll 1
            for (int t = 0; t < NTILE; ++t) col_tile_step<NS, false>(t, g, col, gc, lane, omega, kom6, recs, parks, bars, nullptr, pf);
        }
        pf.mark();
        col_tiles_store<NS>(a, pair, col, lane, outs, parks);
        pf.add(K1P_STORE);
    }
    if (col == 0 && lane == 0) bulk_store_wait_all();        // the last bulk stores must have completed before the CTA retires
    pf.flush(warp, lane);
}

template <int NS>
__device__ __forceinline__ void state_warp(const DirectArgs& a, long long n_tiles, int warp, int t, int lane, double* recs, unsigned bars) {
    typedef Cfg<NS> C;
    const int nsteps = a.cfg.nsteps, nstep = nsteps - 1;
    const int back = lane & 1;
    const double omega = back ? -1.0 : 1.0;
    double r[3], v[3], m = a.c.default_mass, u[3], bm[3] = {0.0, 0.0, 0.0}, mdot = 0.0, t0 = 0.0, t1 = 1.0, maxErr = 0.0;
    K1Prof pf;
    pf.start();
    unsigned g = 0;
    for (long long pair = blockIdx.x; pair * NTILE < n_tiles; pair += gridDim.x) {
        // ---- load this tile's legs (multiShoot_CRTBP_direct.jl:82-95)
        const long long seg = (pair * NTILE + t) * 16 + (lane >> 1);
        {
            const long long sc = seg < a.n_seg ? seg : a.n_seg - 1;     // ragged tail: recompute a valid segment, never store it
            const long long ia = lto_node_a(sc, a.npt);
            const double* X = (back ? a.Xb : a.Xa) + ia * NS;
            const double* U = (back ? a.ub : a.ua) + ia * 3;
            r[0] = X[0]; r[1] = X[1]; r[2] = X[2];
            v[0] = X[3]; v[1] = X[4]; v[2] = X[5];
            if (back) { v[0] = -v[0]; v[1] = -v[1]; v[2] = -v[2]; }     // :92
            if (NS == 7) m = X[6];
            u[0] = U[0]; u[1] = U[1]; u[2] = U[2];
            const double ta = a.ta[ia], tb = a.tb[ia];
            t0 = ta; t1 = ta + (tb - ta) / 2.0;                         // :70
            const double un = sqrt(fma(u[0], u[0], fma(u[1], u[1], u[2] * u[2])));
            mdot = -omega * un * a.c.cmdot;                             // CRTBP_prop_EP_deriv.jl:42
            if (NS == 7) {
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const double uh = (un > 0.0) ? u[q] / un : 1.0;     // one-sided slope at |u| = 0
                    bm[q] = -omega * a.c.cmdot * uh;
                }
            }
            maxErr = 0.0;
        }
        for (int k = 0; k < nstep; ++k, ++g) {
            const unsigned slot = g & (NSLOT - 1), use = g / NSLOT;
            double* slotp = recs + (size_t)(t * NSLOT + slot) * C::STEP_DOUBLES * 32;
            double* rec = slotp + lane;
            const unsigned full = bars + (unsigned)((t * NSLOT + slot) * 16), empty = full + 8;
            pf.mark();
            if (use > 0) mbar_wait(empty, (use - 1) & 1);               // every column thread is done with this slot
            pf.add(K1P_BAR);
            const double h = linrange_at(t0, t1, nsteps, k + 1) - linrange_at(t0, t1, nsteps, k);   // ode.jl:904
            if (NS == 7) {
#pragma unroll
                for (int q = 0; q < 3; ++q) rec[(C::OFF_BM + q) * 32] = bm[q];
            }
            x_step<NS>(r, v, m, u, omega, mdot, h, a.c, rec, slotp + lane * C::SVAL, maxErr);
            mbar_arrive(full);
            pf.add(K1P_WORK);
            pf.step();
        }
        // ---- defect = forward end - R * backward end (:98-101), errors (:104)
        const unsigned fullmask = 0xffffffffu;
        double xe[NS];
        xe[0] = r[0]; xe[1] = r[1]; xe[2] = r[2];
        xe[3] = back ? -v[0] : v[0]; xe[4] = back ? -v[1] : v[1]; xe[5] = back ? -v[2] : v[2];
        if (NS == 7) xe[6] = m;
        bool bad = false;
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            const double other = __shfl_xor_sync(fullmask, xe[q], 1);
            const double d = xe[q] - other;
            bad |= !(d == d);
            if (!back && seg < a.n_seg) a.defect[seg * NS + q] = d;
        }
        const double me_o = __shfl_xor_sync(fullmask, maxErr, 1);
        if (!back && seg < a.n_seg) {
            if (a.errors) a.errors[seg] = fmax(maxErr, me_o);
            if (a.status) a.status[seg] = bad ? LTO_ST_NAN : LTO_OK;
        }
    }
    pf.flush(warp, lane);
}


// ---------------------------------------------------------------------------
// K2: the same layout with the reference's ode78 controller (GeneralCode/ode.jl:477-534) in the state warps, norms over
// the state (LTO_NORM_STATE): the step sequence of a leg depends on x alone, so the state warp still runs ahead of the
// columns.  It retries rejected attempts by itself and publishes ACCEPTED steps only -- the column warps never see a
// rejection.  Legs of a tile take different numbers of steps: a finished leg publishes zero-length steps (h = 0, zero
// linearisation: the column is left unchanged) until the slowest leg of the tile is through; a per-slot flag tells the
// column warps which step is the tile's last.
// ---------------------------------------------------------------------------
// h = 0 and a zero linearisation: a column step leaves the column unchanged
template <int NS>
__device__ __forceinline__ void zero_step_record(double* rec, double* stg) {
    constexpr int SVAL = Cfg<NS>::SVAL;
#pragma unroll
    for (int j = 0; j < 13; ++j) {
        double2* w = reinterpret_cast<double2*>(stg + j * SVAL * 32);
#pragma unroll
        for (int p = 0; p < SVAL / 2; ++p) w[p] = make_double2(0.0, 0.0);
    }
    rec[Cfg<NS>::OFF_H * 32] = 0.0;
}

template <int NS>
__device__ __forceinline__ void state_warp_adapt(const DirectArgs& a, long long n_tiles, int t, int lane, double* recs, unsigned bars, volatile int* lastf) {
    typedef Cfg<NS> C;
    const int back = lane & 1;
    const double omega = back ? -1.0 : 1.0;
    const unsigned fullmask = 0xffffffffu;
    double r[3], v[3], m = a.c.default_mass, u[3], bm[3] = {0.0, 0.0, 0.0}, mdot = 0.0, dummy = 0.0;
    unsigned g = 0;
    for (long long pair = blockIdx.x; pair * NTILE < n_tiles; pair += gridDim.x) {
        const long long seg = (pair * NTILE + t) * 16 + (lane >> 1);
        const long long sc = seg < a.n_seg ? seg : a.n_seg - 1;
        const long long ia = lto_node_a(sc, a.npt);
        const double* X = (back ? a.Xb : a.Xa) + ia * NS;
        const double* U = (back ? a.ub : a.ua) + ia * 3;
        r[0] = X[0]; r[1] = X[1]; r[2] = X[2];
        v[0] = X[3]; v[1] = X[4]; v[2] = X[5];
        if (back) { v[0] = -v[0]; v[1] = -v[1]; v[2] = -v[2]; }
        if (NS == 7) m = X[6];
        u[0] = U[0]; u[1] = U[1]; u[2] = U[2];
        const double ta = a.ta[ia], tb = a.tb[ia];
        const double t0 = ta, tfinal = ta + (tb - ta) / 2.0;
        const double un = sqrt(fma(u[0], u[0], fma(u[1], u[1], u[2] * u[2])));
        mdot = -omega * un * a.c.cmdot;
        if (NS == 7) {
#pragma unroll
            for (int q = 0; q < 3; ++q) { const double uh = (un > 0.0) ? u[q] / un : 1.0; bm[q] = -omega * a.c.cmdot * uh; }
        }
        // ---- drive_ode78 (lto_prop_generic.cuh) / ode78 (ode.jl:477-534)
        const double hmax = (tfinal - t0) / 2.5, hmin = (tfinal - t0) / 1e7;
        double tt = t0, h = (tfinal - t0) / 50.0;
        int status = 0, nt = 0;
        bool done = !((tt < tfinal) && (h >= hmin));
        while (true) {
            const unsigned slot = g & (NSLOT - 1), use = g / NSLOT;
            double* slotp = recs + (size_t)(t * NSLOT + slot) * C::STEP_DOUBLES * 32;
            double* rec = slotp + lane;
            double* stg = slotp + lane * C::SVAL;
            const unsigned full = bars + (unsigned)((t * NSLOT + slot) * 16), empty = full + 8;
            if (use > 0) mbar_wait(empty, (use - 1) & 1);
            if (NS == 7) {
#pragma unroll
                for (int q = 0; q < 3; ++q) rec[(C::OFF_BM + q) * 32] = bm[q];
            }
            bool pending = !done;
            if (done) {                                                      // zero-length step: leaves the column unchanged
                zero_step_record<NS>(rec, stg);
            }
            while (__any_sync(fullmask, pending)) {
                if (pending) {
                    if (tt + h > tfinal) h = tfinal - tt;
                    if (nt >= a.cfg.max_attempts) { status = LTO_ST_MAXSTEPS; done = true; pending = false; }
                }
                if (pending) {
                    ++nt;
                    double r2[3] = {r[0], r[1], r[2]}, v2[3] = {v[0], v[1], v[2]}, m2 = m;
                    const double xn = fmax(fmax(fmax(fabs(r[0]), fabs(r[1])), fmax(fabs(r[2]), fabs(v[0]))), fmax(fmax(fabs(v[1]), fabs(v[2])), NS == 7 ? fabs(m) : 0.0));
                    double delta = x_step<NS>(r2, v2, m2, u, omega, mdot, h, a.c, rec, stg, dummy);
                    if (!(delta == delta)) { status = LTO_ST_NAN; done = true; pending = false; }
                    else {
                        const double tau = a.cfg.tol * fmax(xn, 1.0);
                        if (delta <= tau) {                                  // accepted: this record goes out
                            tt += h;
                            r[0] = r2[0]; r[1] = r2[1]; r[2] = r2[2]; v[0] = v2[0]; v[1] = v2[1]; v[2] = v2[2]; m = m2;
                            pending = false;
                        }
                        if (delta == 0.0) delta = 1e-16;
                        h = fmin(hmax, 0.8 * h * pow(tau / delta, 0.125));
                        if (!((tt < tfinal) && (h >= hmin))) { done = true; if (pending) { status = LTO_ST_HMIN; pending = false; } }
                    }
                }
            }
            if (status != 0) zero_step_record<NS>(rec, stg);               // a failed leg must not hand a rejected attempt to the columns
            const bool all_done = __all_sync(fullmask, done);
            if (lane == 0) lastf[t * NSLOT + slot] = all_done ? 1 : 0;
            mbar_arrive(full);
            ++g;
            if (all_done) break;
        }
        if (status == 0 && tt < tfinal) status = LTO_ST_HMIN;
        double xe[NS];
        xe[0] = r[0]; xe[1] = r[1]; xe[2] = r[2];
        xe[3] = back ? -v[0] : v[0]; xe[4] = back ? -v[1] : v[1]; xe[5] = back ? -v[2] : v[2];
        if (NS == 7) xe[6] = m;
        bool bad = false;
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            const double other = __shfl_xor_sync(fullmask, xe[q], 1);
            const double d = xe[q] - other;
            bad |= !(d == d);
            if (!back && seg < a.n_seg) a.defect[seg * NS + q] = d;
        }
        const int st_o = __shfl_xor_sync(fullmask, status, 1);
        if (!back && seg < a.n_seg) {
            if (a.errors) a.errors[seg] = 0.0;
            if (a.status) a.status[seg] = status ? status : (st_o ? st_o : (bad ? LTO_ST_NAN : LTO_OK));
        }
    }
}

template <int NS>
__device__ __forceinline__ void column_warp_adapt(const DirectArgs& a, long long n_tiles, int warp, int col, int lane, double* recs, double* outs,
                                                  double* parks, unsigned bars, volatile int* lastf) {
    const double omega = (lane & 1) ? -1.0 : 1.0;
    const double kom6 = a.c.kthr / a.c.default_mass;
    const int gc = col - NS;
    K1Prof pf;
    pf.start();
    unsigned g[NTILE];
#pragma unroll
    for (int t = 0; t < NTILE; ++t) g[t] = 0;
    for (long long pair = blockIdx.x; pair * NTILE < n_tiles; pair += gridDim.x) {
#pragma unroll 1
        for (int t = 0; t < NTILE; ++t) { ColState c; col_init<NS>(c, col); col_park<NS>(col_park_at<NS>(parks, t, col, lane), c); }
        unsigned alive = (1u << NTILE) - 1u;
        while (alive) {
            pf.mark();
#ifndef LTO_K1_NO_PACE
            asm volatile("bar.sync 3, %0;" ::"n"(32 * Cfg<NS>::NCOL) : "memory");     // keep the column warps on the same instructions (see column_warp)
#endif
            pf.add(K1P_PACE);
#pragma unroll
            for (int t = 0; t < NTILE; ++t) {
                if (!(alive & (1u << t))) continue;
                if (col_tile_step<NS, true>(t, g[t], col, gc, lane, omega, kom6, recs, parks, bars, lastf, pf)) alive &= ~(1u << t);
                ++g[t];
            }
        }
        pf.mark();
        col_tiles_store<NS>(a, pair, col, lane, outs, parks);
        pf.add(K1P_STORE);
    }
    if (col == 0 && lane == 0) bulk_store_wait_all();
    pf.flush(warp, lane);
}

template <int NS, bool ADAPT>
__global__ void __launch_bounds__(Cfg<NS>::NTHREADS, 1) k_direct_cw(DirectArgs a, long long n_tiles) {
    typedef Cfg<NS> C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* recs = reinterpret_cast<double*>(smem_raw);
    double* outs = reinterpret_cast<double*>(smem_raw + C::REC_BYTES);
    double* parks = reinterpret_cast<double*>(smem_raw + C::PARK_OFF);
    const unsigned bars = smem_u32(smem_raw + C::BAR_OFF);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < NTILE * NSLOT; ++i) {
            mbar_init(bars + i * 16, 32);                    // full : the state warp's lanes
            mbar_init(bars + i * 16 + 8, 32 * C::NCOL);      // empty: every column thread
        }
    }
    __syncthreads();
    volatile int* lastf = reinterpret_cast<volatile int*>(smem_raw + C::FLAG_OFF);
    if (warp >= XW0 && warp < XW0 + NTILE) {
        if (ADAPT) state_warp_adapt<NS>(a, n_tiles, warp - XW0, lane, recs, bars, lastf);
        else state_warp<NS>(a, n_tiles, warp, warp - XW0, lane, recs, bars);
    } else {
        const int col = warp < XW0 ? warp : warp - NTILE;
        if (ADAPT) column_warp_adapt<NS>(a, n_tiles, warp, col, lane, recs, outs, parks, bars, lastf);
        else column_warp<NS>(a, n_tiles, warp, col, lane, recs, outs, parks, bars);
    }
}

// ---------------------------------------------------------------------------
// K4 (direct): defect-only -- the line searches (:415-425), the t_f partials (:511-512) and the
// per-iteration check (:585) of multiShoot_CRTBP_direct.jl.  One thread per leg, the same x_step as the
// state warps above without publishing anything: 39 stage doubles in registers, no shared memory.
// ---------------------------------------------------------------------------
template <int NS>
__global__ void __launch_bounds__(128) k_direct_state(DirectArgs a) {
    const int nsteps = a.cfg.nsteps, nstep = nsteps - 1;
    const int lane = threadIdx.x & 31, back = lane & 1;
    const double omega = back ? -1.0 : 1.0;
    const long long n_pairs32 = (a.n_seg + 15) / 16;                       // warps' worth of legs
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarp = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = warp0; w < n_pairs32; w += nwarp) {
        const long long seg = w * 16 + (lane >> 1);
        const long long sc = seg < a.n_seg ? seg : a.n_seg - 1;
        const long long ia = lto_node_a(sc, a.npt);
        const double* X = (back ? a.Xb : a.Xa) + ia * NS;
        const double* U = (back ? a.ub : a.ua) + ia * 3;
        double r[3] = {X[0], X[1], X[2]}, v[3] = {X[3], X[4], X[5]}, m = a.c.default_mass, u[3] = {U[0], U[1], U[2]}, maxErr = 0.0;
        if (back) { v[0] = -v[0]; v[1] = -v[1]; v[2] = -v[2]; }           // :92
        if (NS == 7) m = X[6];
        const double ta = a.ta[ia], tb = a.tb[ia];
        const double t0 = ta, t1 = ta + (tb - ta) / 2.0;                   // :70
        const double un = sqrt(fma(u[0], u[0], fma(u[1], u[1], u[2] * u[2])));
        const double mdot = -omega * un * a.c.cmdot;                       // CRTBP_prop_EP_deriv.jl:42
        for (int k = 0; k < nstep; ++k) {
            const double h = linrange_at(t0, t1, nsteps, k + 1) - linrange_at(t0, t1, nsteps, k);   // ode.jl:904
            x_step<NS, false>(r, v, m, u, omega, mdot, h, a.c, nullptr, nullptr, maxErr);
        }
        const unsigned fullmask = 0xffffffffu;
        double xe[NS];
        xe[0] = r[0]; xe[1] = r[1]; xe[2] = r[2];
        xe[3] = back ? -v[0] : v[0]; xe[4] = back ? -v[1] : v[1]; xe[5] = back ? -v[2] : v[2];
        if (NS == 7) xe[6] = m;
        bool bad = false;
#pragma unroll
        for (int q = 0; q < NS; ++q) {
            const double other = __shfl_xor_sync(fullmask, xe[q], 1);
            const double d = xe[q] - other;
            bad |= !(d == d);
            if (!back && seg < a.n_seg) a.defect[seg * NS + q] = d;       // :101
        }
        const double me_o = __shfl_xor_sync(fullmask, maxErr, 1);
        if (!back && seg < a.n_seg) {
            if (a.errors) a.errors[seg] = fmax(maxErr, me_o);              // :104
            if (a.status) a.status[seg] = bad ? LTO_ST_NAN : LTO_OK;
        }
    }
}

}  // namespace cw

template <int NS>
static cudaError_t launch_state(const DirectArgs& a, cudaStream_t st) {
    int dev = 0, n_sm = 0;
    cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e;
    const long long n_warps = (a.n_seg + 15) / 16;
    const long long blocks = (n_warps + 3) / 4;
    const int grid = (int)std::min<long long>(blocks, (long long)n_sm * 16);
    cw::k_direct_state<NS><<<grid, 128, 0, st>>>(a);
    return cudaGetLastError();
}

template <int NS, bool ADAPT>
static cudaError_t launch_cw(const DirectArgs& a, cudaStream_t st) {
    typedef cw::Cfg<NS> C;
    // per device: a single process may drive several GPUs (lto_init_devices)
    static int n_sm_dev[64] = {0};
    static bool attr_dev[64] = {false};
    int dev = 0;
    { cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e; }
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (!attr_dev[dev]) {
        cudaError_t e = cudaDeviceGetAttribute(&n_sm_dev[dev], cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(cw::k_direct_cw<NS, ADAPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
        if (e != cudaSuccess) return e;
        attr_dev[dev] = true;
    }
    const int n_sm = n_sm_dev[dev];
    const long long n_tiles = (a.n_seg + 15) / 16;
    const long long n_pairs = (n_tiles + cw::NTILE - 1) / cw::NTILE;
    const int grid = (int)std::min<long long>(n_pairs, (long long)n_sm);
    cw::k_direct_cw<NS, ADAPT><<<grid, C::NTHREADS, C::SMEM, st>>>(a, n_tiles);
    return cudaGetLastError();
}

#ifdef LTO_K1_PROF
// counters of the last K1 / K2 launch (each warp overwrites its own): [block < 1024][warp < 16][K1P_N] (K1P_WORK, _BAR, _PACE, _STORE, _TOTAL, _STEPS)
extern "C" int lto_k1_prof_read(unsigned long long* out, int n_words) {
    const size_t n = std::min<size_t>((size_t)n_words, sizeof(cw::k1_prof) / sizeof(unsigned long long));
    return (int)cudaMemcpyFromSymbol(out, cw::k1_prof, n * sizeof(unsigned long long));
}
#endif

cudaError_t launch_direct_cw(const DirectArgs& a, int nstate, cudaStream_t st, int* n_launch) {
    *n_launch = 0;
    if (a.n_seg <= 0 || a.n_seg > (1ll << 34)) return cudaErrorNotSupported;
    if (a.cfg.mode != 0 && (a.cfg.err_norm != 0 || a.jac == nullptr)) return cudaErrorNotSupported;   // K2 covers the state-norm controller with Jacobian
    if (a.jac != nullptr && (reinterpret_cast<uintptr_t>(a.jac) & 15u) != 0) return cudaErrorNotSupported;   // bulk stores need 16-byte alignment
    cudaError_t e;
    if (a.jac == nullptr) {
        if (nstate == 7) e = launch_state<7>(a, st);
        else if (nstate == 6) e = launch_state<6>(a, st);
        else return cudaErrorNotSupported;
    } else if (a.cfg.mode != 0) {
        if (nstate == 7) e = launch_cw<7, true>(a, st);
        else if (nstate == 6) e = launch_cw<6, true>(a, st);
        else return cudaErrorNotSupported;
    } else if (nstate == 7) e = launch_cw<7, false>(a, st);
    else if (nstate == 6) e = launch_cw<6, false>(a, st);
    else return cudaErrorNotSupported;
    if (e == cudaSuccess) *n_launch = 1;
    return e;
}

}  // namespace lto
