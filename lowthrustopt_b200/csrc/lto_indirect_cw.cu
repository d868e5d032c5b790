// lto_indirect_cw.cu -- throughput kernel for the indirect method (K3), ndim = 12:
// defectCalc + jacobianCalc of multiShoot_CRTBP_indirect.jl:63-124 for a whole batch in one
// launch.  Each segment integrates [x | Phi] (12 + 144 components) with the adaptive
// order-8 pair and the OrdinaryDiffEq-style controller of lto_prop_generic.cuh
// (drive_rk8); Phi replaces ForwardDiff.jacobian(f, x0) (:121).
//
// Mapping (DESIGN.md section 5):
//   tile        = 32 segment SLOTS owned by one state warp (lane = slot); a CTA keeps
//                 NTILE = 2 tiles in flight.
//   state warp  = runs the nonlinear 12-dim system, the step-size controller and the
//                 per-slot work queue (a slot that finishes its segment pulls the next one
//                 from a global counter, so slots advance independently and no lane waits
//                 for the slowest segment of the batch).  Publishes, per attempted step,
//                 the 13 stage linearisations U, W, G (18 doubles per stage and slot) + h +
//                 control flags in shared memory.
//   column warp = 6 per CTA, shared by the tiles.  Warp w carries STM columns 2w (lanes
//                 0-15) and 2w+1 (lanes 16-31) of 16 slots at a time, so the two half-warps
//                 read the same stage record (a 128-bit load costs the minimum two
//                 shared-memory wavefronts); a tile is processed as two half-phases.
//                 A thread owns one whole column (12 components): every RK combination
//                 and the structured product A*phi stay in its ~240 registers, which is
//                 what limits the CTA to 8 warps (2 per SM sub-partition).
//   hand-off    = two mbarriers per tile (record full / columns done); the column warps
//                 alternate between the tiles, so one state warp's dependent chain is
//                 hidden behind the column work of the other tile.
// Step control uses the joint norm over x and Phi (LTO_NORM_STATE_SENS, the ForwardDiff
// semantics) or x alone: each column thread returns its partial sum of squared scaled
// errors and the state warp decides.  Between visits a column's candidate lives in a
// shared-memory stash and its current (last accepted) value in an L2-resident scratch, so an
// accepted step never waits on L2 and a rejected one costs one L2 read.
// The initial step is Hairer's estimate over the state components (the generic kernel
// and the CPU checker take it over x and Phi): the two paths may choose different step
// sequences and agree to the integration tolerance, not to rounding.
#include "lto_internal.h"
#include "lto_cw_common.cuh"
#include "lto_switch.h"
#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace lto {
namespace icw {

using namespace cwc;

constexpr int ND = 12;
constexpr int NTILE = 2;          // state warps = tiles in flight
constexpr int TS = 32;            // segment slots per tile
constexpr int HS = 16;            // slots per column half-phase
constexpr int NCW = 6;            // column warps
constexpr int NCT = 32 * NCW;     // column threads
constexpr int NC2 = 9;            // double2 per stage record: U[6] W[6] G[6]
constexpr int NW = NTILE + NCW;
constexpr int NTHREADS = 32 * NW;

enum { F_ACCEPT = 1, F_STORE = 2, F_RESET = 4, F_ACTIVE = 8 };   // F_STORE: the column threads store this slot's STM (only when the state warp could not, see STASH)

// ---- shared-memory plan ------------------------------------------------------
constexpr size_t REC_BYTES = (size_t)13 * NC2 * TS * sizeof(double2);      // stage records of one tile
constexpr size_t HDR_BYTES = (size_t)TS * (sizeof(double) + sizeof(int2)); // h, {flags, segment}
// Candidate stash, slot-major: the 12 columns of a slot are 1152 contiguous bytes in the output's own layout (column-major 12 x 12), so the
// state warp sends a finished segment's STM as ONE bulk store (full packets when `phi` is NVLink peer memory of the solver rank).  Slot stride
// 1168 B: 16-byte aligned for the bulk copy, and the 128-bit accesses of a quarter-warp (8 slots of one column) fall into 32 different banks.
constexpr int STASH_STRIDE = ND * ND + 2;
constexpr size_t CUR_BYTES = (size_t)TS * STASH_STRIDE * sizeof(double);
constexpr size_t ERR_BYTES = (size_t)ND * TS * sizeof(double);             // error partials per column and slot
constexpr size_t XN_BYTES = (size_t)2 * ND * TS * sizeof(double);          // the state x and its candidate (double buffer; keeps 24 registers free in the state warps)
constexpr int NXW = ND + 6;                                                // next-segment stash: x0, t0, tf, aL, 1/rho, aL/(4 rho), h0
constexpr size_t NXT_BYTES = (size_t)NXW * TS * sizeof(double);
constexpr size_t TILE_BYTES = REC_BYTES + HDR_BYTES + CUR_BYTES + ERR_BYTES + XN_BYTES + NXT_BYTES;
constexpr size_t BAR_BYTES = 128;                                          // 13 stage barriers, done, tile_done
constexpr size_t SMEM = NTILE * TILE_BYTES + NTILE * BAR_BYTES;
// Stage-level hand-off (columns start a tile while its state warp is still producing the later
// stages; one mbarrier per stage) was measured and is NOT faster: the 13 release-arrivals lengthen
// the state warp's chain and both warp kinds compete for the same issue slots.  Kept switchable.
constexpr bool STAGE_PIPE = false;
constexpr int START_STAGE = 4;
constexpr size_t SCRATCH_BYTES_PER_CTA = (size_t)NTILE * 2 * ND * NCT * sizeof(double);   // candidate columns (global)

struct TileSmem {
    double2* rec; double* hval; int2* hctl; double* cur; double* errp; double* xn; double* nx;
    unsigned bar_full, bar_done; volatile int* tile_done;
};

__device__ __forceinline__ TileSmem tile_smem(unsigned char* base, int t) {
    unsigned char* p = base + (size_t)t * TILE_BYTES;
    TileSmem s;
    s.rec = reinterpret_cast<double2*>(p); p += REC_BYTES;
    s.hval = reinterpret_cast<double*>(p); p += TS * sizeof(double);
    s.hctl = reinterpret_cast<int2*>(p); p += TS * sizeof(int2);
    s.cur = reinterpret_cast<double*>(p); p += CUR_BYTES;
    s.errp = reinterpret_cast<double*>(p); p += ERR_BYTES;
    s.xn = reinterpret_cast<double*>(p); p += XN_BYTES;
    s.nx = reinterpret_cast<double*>(p);
    unsigned char* b = base + (size_t)NTILE * TILE_BYTES + (size_t)t * BAR_BYTES;
    s.bar_full = smem_u32(b); s.bar_done = smem_u32(b + 13 * 8);         // bar_full + 8 j: stage j's record is published
    s.tile_done = reinterpret_cast<volatile int*>(b + 14 * 8);
    return s;
}

// ---------------------------------------------------------------------------
// Stage inputs of one 12-vector y = [r v lr lv] in Nystrom form for the (r, v) pair:
// only v', lr', lv' of every stage are kept (kv, kl, km); positions are rebuilt with
// G = B*B (lto_tableau.h).
// ---------------------------------------------------------------------------
struct KStore { double kv[13][3], kl[13][3], km[13][3]; };

template <int J, bool SPLIT = false>
__device__ __forceinline__ void stage_input(const KStore& K, const double (&y)[ND], double h, double h2,
                                            double (&R)[3], double (&V)[3], double (&L)[3], double (&M)[3]) {
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        if (J == 0) { R[q] = y[q]; V[q] = y[3 + q]; L[q] = y[6 + q]; M[q] = y[9 + q]; continue; }
        // SPLIT (state warps): two partial sums per combination (even / odd stage index) halve the dependent-FMA depth of the chain
        double av = 0.0, ar = 0.0, al = 0.0, am = 0.0, bv = 0.0, br = 0.0, bl = 0.0, bm = 0.0;
#pragma unroll
        for (int l = 0; l < J; ++l) {
            if (SPLIT && (l & 1)) {
                if (lto_tab::Bf(J, l) != 0.0) {
                    bv = fma(lto_tab::Bf(J, l), K.kv[l][q], bv);
                    bl = fma(lto_tab::Bf(J, l), K.kl[l][q], bl);
                    bm = fma(lto_tab::Bf(J, l), K.km[l][q], bm);
                }
                if (lto_tab::Gf(J, l) != 0.0) br = fma(lto_tab::Gf(J, l), K.kv[l][q], br);
            } else {
                if (lto_tab::Bf(J, l) != 0.0) {
                    av = fma(lto_tab::Bf(J, l), K.kv[l][q], av);
                    al = fma(lto_tab::Bf(J, l), K.kl[l][q], al);
                    am = fma(lto_tab::Bf(J, l), K.km[l][q], am);
                }
                if (lto_tab::Gf(J, l) != 0.0) ar = fma(lto_tab::Gf(J, l), K.kv[l][q], ar);
            }
        }
        if (SPLIT) { av += bv; ar += br; al += bl; am += bm; }
        V[q] = fma(h, av, y[3 + q]);
        R[q] = fma(h2, ar, fma(h * lto_tab::Cf(J), y[3 + q], y[q]));
        L[q] = fma(h, al, y[6 + q]);
        M[q] = fma(h, am, y[9 + q]);
    }
}


// State-only step control (LTO_NORM_STATE: K4, and K3 when the columns are not in the norm): the embedded estimate e = ga + gb is the
// sum of the differences ga ~ (k1 - k12) and gb ~ (k11 - k13), which can cancel; the controller then takes max(|e|, |ga|, |gb|)
// per component (lto_prop_generic.cuh drive_rk8 `robust`; DESIGN.md section 4).  A NaN estimate stays NaN.
__device__ __forceinline__ double rob_est(double e, double ga) {
    const double m = fmax(fabs(e), fmax(fabs(ga), fabs(e - ga)));
    return (e == e) ? m : e;
}

// 8th-order update (ode.jl:937) and, if ERR, the scaled squared error of the embedded
// estimate (ode.jl:940 with the controller's scaling atol + rtol*max(|y|, |ynew|)).
template <bool ERR, bool ROB = false>
__device__ __forceinline__ double step_finish(const KStore& K, const double (&y)[ND], double h, double h2, double atol, double rtol,
                                              double (&yn)[ND]) {
    double esum = 0.0;
    const double ce = h * lto_tab::ERRC, ce2 = h2 * lto_tab::ERRC;
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        double sv = 0.0, sr = 0.0, sl = 0.0, sm = 0.0;
#pragma unroll
        for (int l = 0; l < 13; ++l) {
            if (lto_tab::CHIf(l) != 0.0) {
                sv = fma(lto_tab::CHIf(l), K.kv[l][q], sv);
                sl = fma(lto_tab::CHIf(l), K.kl[l][q], sl);
                sm = fma(lto_tab::CHIf(l), K.km[l][q], sm);
            }
            if (lto_tab::CHIBf(l) != 0.0) sr = fma(lto_tab::CHIBf(l), K.kv[l][q], sr);
        }
        yn[q] = fma(h2, sr, fma(h, y[3 + q], y[q]));
        yn[3 + q] = fma(h, sv, y[3 + q]);
        yn[6 + q] = fma(h, sl, y[6 + q]);
        yn[9 + q] = fma(h, sm, y[9 + q]);
        if (ERR) {
            double e[4];
            e[0] = ce2 * (K.kv[0][q] - K.kv[11][q]);                                          // psi^T B = e_1 - e_12
            e[1] = ce * ((K.kv[0][q] + K.kv[10][q]) - (K.kv[11][q] + K.kv[12][q]));
            e[2] = ce * ((K.kl[0][q] + K.kl[10][q]) - (K.kl[11][q] + K.kl[12][q]));
            e[3] = ce * ((K.km[0][q] + K.km[10][q]) - (K.km[11][q] + K.km[12][q]));
            if (ROB) {
                double gr = 0.0;                                                              // (k1 - k12) of r' = v: -h B[11] . kv
#pragma unroll
                for (int l = 0; l < 11; ++l)
                    if (lto_tab::Bf(11, l) != 0.0) gr = fma(lto_tab::Bf(11, l), K.kv[l][q], gr);
                e[0] = rob_est(e[0], -ce2 * gr);
                e[1] = rob_est(e[1], ce * (K.kv[0][q] - K.kv[11][q]));
                e[2] = rob_est(e[2], ce * (K.kl[0][q] - K.kl[11][q]));
                e[3] = rob_est(e[3], ce * (K.km[0][q] - K.km[11][q]));
            }
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const double sc = fma(rtol, fmax(fabs(y[3 * b + q]), fabs(yn[3 * b + q])), atol);
                const double r = e[b] * fast_rcp(sc);
                esum = fma(r, r, esum);
            }
        }
    }
    return esum;
}

// ---------------------------------------------------------------------------
// Column thread: one attempted RK step of one STM column phi = [pr pv plr plv].
//   kv = U pr + C pv + G plv;  kl = -(W pr + U plv);  km = -plr - C^T plv   (lto_math.cuh sc_col)
// Stage 11 (index 10) enters only the error estimate: skipped when the columns are not
// part of the step-control norm.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void sym3_mul_nacc(const double M[6], const double v[3], double out[3]) {
    out[0] = fma(-M[0], v[0], fma(-M[3], v[1], fma(-M[4], v[2], out[0])));
    out[1] = fma(-M[3], v[0], fma(-M[1], v[1], fma(-M[5], v[2], out[1])));
    out[2] = fma(-M[4], v[0], fma(-M[5], v[1], fma(-M[2], v[2], out[2])));
}

template <int J>
__device__ __forceinline__ void col_stage(KStore& K, const double (&p)[ND], double h, double h2, double w2, const double2* __restrict__ rec,
                                          unsigned bar, unsigned par) {
    double R[3], V[3], L[3], M[3];
    stage_input<J>(K, p, h, h2, R, V, L, M);
    if (STAGE_PIPE && J > START_STAGE) mbar_wait(bar + 8 * J, par);   // the state warp may still be producing the later stages
    const double2* w = rec + J * NC2 * TS;
    double U[6], W[6], G[6];
    { const double2 a = w[0 * TS], b = w[1 * TS], c = w[2 * TS]; U[0] = a.x; U[1] = a.y; U[2] = b.x; U[3] = b.y; U[4] = c.x; U[5] = c.y; }
    { const double2 a = w[3 * TS], b = w[4 * TS], c = w[5 * TS]; W[0] = a.x; W[1] = a.y; W[2] = b.x; W[3] = b.y; W[4] = c.x; W[5] = c.y; }
    { const double2 a = w[6 * TS], b = w[7 * TS], c = w[8 * TS]; G[0] = a.x; G[1] = a.y; G[2] = b.x; G[3] = b.y; G[4] = c.x; G[5] = c.y; }
    double a[3] = {w2 * V[1], -w2 * V[0], 0.0};
    sym3_mul_acc(U, R, a);
    sym3_mul_acc(G, M, a);
    double b[3] = {0.0, 0.0, 0.0};
    sym3_mul_nacc(W, R, b);
    sym3_mul_nacc(U, M, b);
#pragma unroll
    for (int q = 0; q < 3; ++q) { K.kv[J][q] = a[q]; K.kl[J][q] = b[q]; }
    K.km[J][0] = fma(w2, M[1], -L[0]);
    K.km[J][1] = fma(-w2, M[0], -L[1]);
    K.km[J][2] = -L[2];
}

// The column warps run the same ~30 KB straight-line body; re-converging them a few times per
// attempt keeps their instruction-fetch windows together (one miss stream instead of six).
#ifndef LTO_ICW_NOLOCKSTEP
#define LTO_ICW_LOCKSTEP() asm volatile("bar.sync 1, %0;" ::"n"(NCT) : "memory")
#else
#define LTO_ICW_LOCKSTEP()
#endif

template <bool ERR>
__device__ __forceinline__ double col_attempt(const double (&p)[ND], double h, double w2, const double2* __restrict__ rec,
                                              unsigned bar, unsigned par, double atol, double rtol, double (&pn)[ND]) {
    const double h2 = h * h;
    KStore K;
    col_stage<0>(K, p, h, h2, w2, rec, bar, par);  col_stage<1>(K, p, h, h2, w2, rec, bar, par);  col_stage<2>(K, p, h, h2, w2, rec, bar, par);
    col_stage<3>(K, p, h, h2, w2, rec, bar, par);  col_stage<4>(K, p, h, h2, w2, rec, bar, par);  col_stage<5>(K, p, h, h2, w2, rec, bar, par);
    LTO_ICW_LOCKSTEP();
#ifdef LTO_ICW_FAKE   /* timing experiment only: half the stages (wrong results) */
#pragma unroll
    for (int j = 6; j < 13; ++j)
#pragma unroll
        for (int q = 0; q < 3; ++q) { K.kv[j][q] = K.kv[j - 6][q]; K.kl[j][q] = K.kl[j - 6][q]; K.km[j][q] = K.km[j - 6][q]; }
#else
    col_stage<6>(K, p, h, h2, w2, rec, bar, par);  col_stage<7>(K, p, h, h2, w2, rec, bar, par);  col_stage<8>(K, p, h, h2, w2, rec, bar, par);
    LTO_ICW_LOCKSTEP();
    col_stage<9>(K, p, h, h2, w2, rec, bar, par);
    if (ERR) col_stage<10>(K, p, h, h2, w2, rec, bar, par);
    LTO_ICW_LOCKSTEP();
    col_stage<11>(K, p, h, h2, w2, rec, bar, par); col_stage<12>(K, p, h, h2, w2, rec, bar, par);
#endif
    return step_finish<ERR>(K, p, h, h2, atol, rtol, pn);
}

template <bool JOINT>
__device__ __forceinline__ void column_warp(const IndirectArgs& a, int cw, int lane, unsigned char* smem) {
    const int col = 2 * cw + (lane >> 4);
    const int ct = cw * 32 + lane;
    const double w2 = 2.0 * a.c.omega;
    const double atol = a.cfg.atol, rtol = a.cfg.rtol;
    double* cand_base = a.scratch + (size_t)blockIdx.x * (SCRATCH_BYTES_PER_CTA / sizeof(double)) + ct;
    const bool wide = (reinterpret_cast<uintptr_t>(a.phi) & 31u) == 0;
    unsigned alive = (1u << NTILE) - 1u;
    unsigned visit = 0;
    long long c_wait = 0, c_work = 0, n_work = 0;
    const long long c_begin = clock64();
    while (alive) {
#pragma unroll 1
        for (int t = 0; t < NTILE; ++t) {
            if (!(alive & (1u << t))) continue;
            const TileSmem S = tile_smem(smem, t);
            const long long c0 = clock64();
            mbar_wait_parked(S.bar_full, visit & 1);                    // header + stage 0
            if (STAGE_PIPE && !*S.tile_done) mbar_wait(S.bar_full + 8 * START_STAGE, visit & 1);
            const long long c1 = clock64();
            c_wait += c1 - c0;
            const bool done = *S.tile_done != 0;
#pragma unroll 1
            for (int hf = 0; hf < 2; ++hf) {
                const int slot = hf * HS + (lane & (HS - 1));
                const int2 hc = S.hctl[slot];
                const double h = S.hval[slot];
                double2* sc = reinterpret_cast<double2*>(S.cur + (size_t)slot * STASH_STRIDE + col * ND);
                double* sn = cand_base + (size_t)(t * 2 + hf) * ND * NCT;
                // The CANDIDATE of the previous attempt lives in shared memory (sc), the CURRENT column (last accepted value) in
                // the L2-resident scratch (sn): an accepted step -- 99.7 % of them -- reads shared memory and refreshes the
                // scratch with fire-and-forget stores; only a rejected step pays an L2 read.
                double p[ND];
                if (hc.x & F_ACCEPT) {
#pragma unroll
                    for (int i = 0; i < ND; i += 2) {
                        const double2 v = sc[i >> 1];
                        p[i] = v.x; p[i + 1] = v.y; __stcg(sn + i * NCT, v.x); __stcg(sn + (i + 1) * NCT, v.y);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < ND; ++i) p[i] = __ldcg(sn + i * NCT);
                }
                if (hc.x & F_STORE) {                                  // column `col` of ForwardDiff.jacobian(f, x0) (:121)
                    // three 32-byte stores per column (96 contiguous bytes, 32-byte aligned): wide enough to travel as full
                    // packets when `phi` is NVLink peer memory of the solver rank
                    double* out = a.phi + (long long)hc.y * (ND * ND) + col * ND;
                    if (wide) {
#pragma unroll
                        for (int i = 0; i < ND; i += 4)
                            asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(out + i), "d"(p[i]), "d"(p[i + 1]), "d"(p[i + 2]), "d"(p[i + 3]) : "memory");
                    } else {
#pragma unroll
                        for (int i = 0; i < ND; ++i) out[i] = p[i];
                    }
                }
                if (hc.x & F_RESET) {
#pragma unroll
                    for (int i = 0; i < ND; ++i) { p[i] = (i == col) ? 1.0 : 0.0; __stcg(sn + i * NCT, p[i]); }
                }
                if (done) continue;
                double pn[ND];
                const double es = col_attempt<JOINT>(p, h, w2, S.rec + slot, S.bar_full, visit & 1, atol, rtol, pn);
#pragma unroll
                for (int i = 0; i < ND; i += 2) sc[i >> 1] = make_double2(pn[i], pn[i + 1]);
                if (JOINT) S.errp[col * TS + slot] = es;
            }
            if (done) alive &= ~(1u << t);
            else {
                fence_proxy_async();                                    // the stash may leave through the async proxy (state warp's bulk store)
                mbar_arrive(S.bar_done); c_work += clock64() - c1; n_work += 2;
            }
        }
        ++visit;
    }
    if (a.prof && lane == 0) {
        unsigned long long* o = a.prof + ((size_t)blockIdx.x * NW + NTILE + cw) * 4;
        o[0] = c_work; o[1] = c_wait; o[2] = n_work; o[3] = clock64() - c_begin;
    }
}

// ---------------------------------------------------------------------------
// State warp: right-hand side CRTBP_stateCostate_deriv! (src/CRTBP_stateCostate_deriv.jl:9-90)
// and its linearisation (lto_math.cuh sc_stage gives the reference formulation; this is the
// same arithmetic arranged for a short dependent chain: no divisions, no library calls
// except exp / pow).
// ---------------------------------------------------------------------------
struct LawConst { double aL, rho_inv, rho_inv_quarter_aL; };   // per slot: aL = thrustLimit*k/mass, 1/rho, aL/(4 rho)

template <bool LIN>
__device__ __forceinline__ void sc_eval(const double (&R)[3], const double (&V)[3], const double (&L)[3], const double (&M)[3],
                                        const SCConst& c, const LawConst& lw, double (&kv)[3], double (&kl)[3], double (&km)[3],
                                        double2* __restrict__ w, double* umag_out = nullptr) {
    const double w2 = 2.0 * c.omega;
    // ---- gravity (:69-70, :78-81) and its gradient
    const double dx1 = R[0] + c.mu, dx2 = dx1 - 1.0;
    const double yz = fma(R[1], R[1], R[2] * R[2]);
    const double i1 = fast_rsqrt(fma(dx1, dx1, yz)), i2 = fast_rsqrt(fma(dx2, dx2, yz));
    const double i1s = i1 * i1, i2s = i2 * i2;
    const double a31 = c.m1 * i1s * i1, a32 = c.mu * i2s * i2;
    const double a51 = 3.0 * a31 * i1s, a52 = 3.0 * a32 * i2s;
    const double gg = -(a31 + a32), s5 = a51 + a52;
    const double p1 = a51 * dx1, p2 = a52 * dx2, t = p1 + p2;
    double U[6];
    U[0] = fma(p1, dx1, fma(p2, dx2, 1.0 + gg));
    U[1] = fma(s5 * R[1], R[1], 1.0 + gg);
    U[2] = fma(s5 * R[2], R[2], gg);
    U[3] = t * R[1]; U[4] = t * R[2]; U[5] = s5 * R[1] * R[2];
    // ---- control law (:36-64): u_acc = -umag * lv/|lv| = -uon * lv
    const double n2 = fma(M[0], M[0], fma(M[1], M[1], M[2] * M[2]));
    const bool dead = !(n2 > 0.0);                                     // :59-64 NaN guard -> zero control
    const double in = dead ? 0.0 : fast_rsqrt(n2);
    const double n = n2 * in;
    double umag, dn = 0.0;
    if (c.p == 1.0) {                                                  // :41-43  0.5 (1 + tanh((n-1)/(2 rho))) aL
        const double y = fmin(fmax((n - 1.0) * lw.rho_inv, -700.0), 700.0);
        const double ey = exp(y);                                      // tanh(y/2) = 1 - 2/(e^y + 1)
        const double th = fma(-2.0, fast_rcp(ey + 1.0), 1.0);
        umag = fma(0.5 * lw.aL, th, 0.5 * lw.aL);
        dn = lw.rho_inv_quarter_aL * fma(-th, th, 1.0);
    } else if (c.p == 0.0) {                                           // :36-39
        umag = lw.aL;
    } else {                                                           // :45-50
        const double e = 1.0 / (c.p - 1.0);
        const double wv = (c.p == 2.0) ? 0.5 * n : pow(n / c.p, e);
        if (wv > lw.aL) umag = lw.aL;
        else { umag = wv; dn = dead ? 0.0 : e * wv * in; }
    }
    if (dead) { umag = 0.0; dn = 0.0; }
    if (!(n2 == n2)) umag = n2;                                        // a NaN costate stays NaN (reported through status[])
    if (umag_out) *umag_out = umag;
    const double uon = umag * in;
    // ---- derivatives (:78-88)
    kv[0] = fma(-uon, M[0], fma(-a31, dx1, fma(-a32, dx2, fma(w2, V[1], R[0]))));
    kv[1] = fma(-uon, M[1], fma(gg, R[1], fma(-w2, V[0], R[1])));
    kv[2] = fma(-uon, M[2], gg * R[2]);
    kl[0] = -fma(U[0], M[0], fma(U[3], M[1], U[4] * M[2]));
    kl[1] = -fma(U[3], M[0], fma(U[1], M[1], U[5] * M[2]));
    kl[2] = -fma(U[4], M[0], fma(U[5], M[1], U[2] * M[2]));
    km[0] = fma(w2, M[1], -L[0]);
    km[1] = fma(-w2, M[0], -L[1]);
    km[2] = -L[2];
    if (LIN) {
        // G = -uon I + (uon - dn) lh lh^T,  lh = lv/|lv|
        const double cd = uon - dn;
        const double l0 = M[0] * in, l1 = M[1] * in, l2 = M[2] * in;
        const double c0 = cd * l0, c1 = cd * l1;
        // W = d(U lv)/dr = sum_b [ h_b d_b d_b^T + a5_b (d_b lv^T + lv d_b^T) ] + (e1 + e2) I,  d_b = (dx_b, y, z)
        const double ylz = fma(R[1], M[1], R[2] * M[2]);
        const double e1 = a51 * fma(dx1, M[0], ylz), e2 = a52 * fma(dx2, M[0], ylz);
        const double h1 = -5.0 * e1 * i1s, h2 = -5.0 * e2 * i2s;
        const double ee = e1 + e2, hs = h1 + h2;
        const double hx = fma(h1, dx1, h2 * dx2);
        const double sM0 = s5 * M[0];
        w[0 * TS] = make_double2(U[0], U[1]);
        w[1 * TS] = make_double2(U[2], U[3]);
        w[2 * TS] = make_double2(U[4], U[5]);
        w[3 * TS] = make_double2(fma(h1 * dx1, dx1, fma(h2 * dx2, dx2, fma(2.0 * t, M[0], ee))),        // W_xx
                                 fma(hs * R[1], R[1], fma(2.0 * s5 * R[1], M[1], ee)));                 // W_yy
        w[4 * TS] = make_double2(fma(hs * R[2], R[2], fma(2.0 * s5 * R[2], M[2], ee)),                  // W_zz
                                 fma(hx, R[1], fma(t, M[1], sM0 * R[1])));                              // W_xy
        w[5 * TS] = make_double2(fma(hx, R[2], fma(t, M[2], sM0 * R[2])),                               // W_xz
                                 fma(hs * R[1], R[2], s5 * fma(R[1], M[2], M[1] * R[2])));              // W_yz
        w[6 * TS] = make_double2(fma(c0, l0, -uon), fma(c1, l1, -uon));
        w[7 * TS] = make_double2(fma(cd * l2, l2, -uon), c0 * l1);
        w[8 * TS] = make_double2(c0 * l2, c1 * l2);
    }
}

// One out-of-line copy of the right-hand side serves all 13 stages: the state warp's code
// must stay small, or its instruction stream evicts the column warps' loop body from the
// instruction cache (ncu: stall_no_inst was the top stall of BOTH warp kinds).
struct Out9 { double v[9]; };
// Arguments and results travel in registers (the device ABI returns this struct in registers): no local-memory round trip
// on the state warp's dependent chain.
__device__ __noinline__ Out9 sc_eval_call(double r0, double r1, double r2, double v0, double v1, double v2, double l0, double l1, double l2,
                                          double m0, double m1, double m2, double mu, double mu1, double omega, double pexp, double aL,
                                          double rho_inv, double rq, double2* w) {
    const double R[3] = {r0, r1, r2}, V[3] = {v0, v1, v2}, L[3] = {l0, l1, l2}, M[3] = {m0, m1, m2};
    SCConst c; c.mu = mu; c.m1 = mu1; c.omega = omega; c.p = pexp;
    LawConst lw; lw.aL = aL; lw.rho_inv = rho_inv; lw.rho_inv_quarter_aL = rq;
    double kv[3], kl[3], km[3];
    sc_eval<true>(R, V, L, M, c, lw, kv, kl, km, w);
    Out9 o;
#pragma unroll
    for (int q = 0; q < 3; ++q) { o.v[q] = kv[q]; o.v[3 + q] = kl[q]; o.v[6 + q] = km[q]; }
    return o;
}

template <int J>
__device__ __forceinline__ void state_stage(KStore& K, const double (&x)[ND], double h, double h2, const SCConst& c, const LawConst& lw,
                                            double2* __restrict__ rec, unsigned bar) {
    double R[3], V[3], L[3], M[3];
    stage_input<J>(K, x, h, h2, R, V, L, M);
    const Out9 o = sc_eval_call(R[0], R[1], R[2], V[0], V[1], V[2], L[0], L[1], L[2], M[0], M[1], M[2], c.mu, c.m1, c.omega, c.p, lw.aL, lw.rho_inv,
                                lw.rho_inv_quarter_aL, rec + J * NC2 * TS);
    if (STAGE_PIPE && J > 0) mbar_arrive(bar + 8 * J);     // stage J's record is published (stage 0 goes out with the header)
#pragma unroll
    for (int q = 0; q < 3; ++q) { K.kv[J][q] = o.v[q]; K.kl[J][q] = o.v[3 + q]; K.km[J][q] = o.v[6 + q]; }
}

// state warps keep x in shared memory (stride TS between components): loaded per stage, live only through the combination
template <int J>
__device__ __forceinline__ void state_stage_s(KStore& K, const double* __restrict__ xs, double h, double h2, const SCConst& c, const LawConst& lw,
                                              double2* __restrict__ rec, unsigned bar) {
    double x[ND];
#pragma unroll
    for (int i = 0; i < ND; ++i) x[i] = xs[i * TS];
    state_stage<J>(K, x, h, h2, c, lw, rec, bar);
}

__device__ __forceinline__ double rms12(const double (&e)[ND], const double (&y)[ND], double atol, double rtol) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < ND; ++i) { const double q = e[i] * fast_rcp(fma(rtol, fabs(y[i]), atol)); s = fma(q, q, s); }
    return sqrt(s * (1.0 / (double)ND));
}

__device__ __noinline__ Out9 sc_eval_state_call(double r0, double r1, double r2, double v0, double v1, double v2, double l0, double l1, double l2,
                                                double m0, double m1, double m2, double mu, double mu1, double omega, double pexp, double aL,
                                                double rho_inv, double rq);

// Off the critical path: while the column warps work on the attempt just published, every slot that has no successor yet claims
// its NEXT segment from the work queue, loads it, and runs the Hairer-Norsett-Wanner initial-step estimate over the state
// components (drive_rk8 in lto_prop_generic.cuh) -- queue atomic, scattered loads and two extra right-hand sides (~4-5 k cycles,
// needed on nearly every visit because some slot of the 32 is always about to finish) used to sit in front of the next attempt.
// The result waits in the tile's shared-memory stash until the slot's current segment finishes.  A slot claims just in time
// (`soon`: it is idle, or the attempt just published reaches t1), so no segment is hoarded while other slots run dry.
__device__ __forceinline__ void prepare_next(const IndirectArgs& a, const TileSmem& S, int slot, long long& nseg, bool& exhausted, bool soon) {
    const unsigned fullmask = 0xffffffffu;
    const bool want = soon && !exhausted && nseg < 0;
    if (!__any_sync(fullmask, want)) return;
    const double atol = a.cfg.atol, rtol = a.cfg.rtol;
    double x[ND];
    double t0 = 0.0, tf = 0.0, aL = 0.0, rho_inv = 1.0, rq = 0.0;
    bool got = false;
    if (want) {
        const long long idx = (long long)atomicAdd(a.counter, 1ull);
        if (idx < a.n_seg) {
            got = true; nseg = idx;
            const long long ia = lto_node_a(idx, a.npt), it = lto_traj_of(idx, a.npt);
#pragma unroll
            for (int i = 0; i < ND; ++i) x[i] = a.x0[ia * ND + i];
            t0 = a.t0[ia]; tf = a.t1[ia];
            if (!(t0 < tf)) tf = t0;                                      // empty span: one zero-length step, Phi = I
            const double tl = a.thrustLimit_arr ? a.thrustLimit_arr[it] : a.c.thrustLimit;
            const double rho = a.rho_arr ? a.rho_arr[it] : a.c.rho;
            aL = tl * a.c.kthr / a.c.mass;                                // :33
            rho_inv = 1.0 / rho;
            rq = aL / (4.0 * rho);
        } else {
            exhausted = true;
        }
    }
    if (!got) {
#pragma unroll
        for (int i = 0; i < ND; ++i) x[i] = 0.0;
    }
    const double span = tf - t0;
    const Out9 o0 = sc_eval_state_call(x[0], x[1], x[2], x[3], x[4], x[5], x[6], x[7], x[8], x[9], x[10], x[11], a.c.mu, a.c.m1, a.c.omega, a.c.p, aL,
                                       rho_inv, rq);
    double f0[ND], y1[ND];
#pragma unroll
    for (int q = 0; q < 3; ++q) { f0[q] = x[3 + q]; f0[3 + q] = o0.v[q]; f0[6 + q] = o0.v[3 + q]; f0[9 + q] = o0.v[6 + q]; }
    const double d0 = rms12(x, x, atol, rtol), d1 = rms12(f0, x, atol, rtol);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * (d0 / d1);
    h0 = fmin(h0, span);
#pragma unroll
    for (int i = 0; i < ND; ++i) y1[i] = fma(h0, f0[i], x[i]);
    const Out9 o1 = sc_eval_state_call(y1[0], y1[1], y1[2], y1[3], y1[4], y1[5], y1[6], y1[7], y1[8], y1[9], y1[10], y1[11], a.c.mu, a.c.m1, a.c.omega, a.c.p,
                                       aL, rho_inv, rq);
#pragma unroll
    for (int q = 0; q < 3; ++q) { const double v1 = y1[3 + q]; y1[q] = v1 - f0[q]; y1[3 + q] = o1.v[q] - f0[3 + q]; y1[6 + q] = o1.v[3 + q] - f0[6 + q]; y1[9 + q] = o1.v[6 + q] - f0[9 + q]; }
    const double d2 = rms12(y1, x, atol, rtol) / h0;
    const double dm = fmax(d1, d2);
    const double h1 = (dm <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : inv_eighth_root(dm / 0.01);
    if (got) {
        double* nx = S.nx + slot;
#pragma unroll
        for (int i = 0; i < ND; ++i) nx[i * TS] = x[i];
        nx[(ND + 0) * TS] = t0; nx[(ND + 1) * TS] = tf; nx[(ND + 2) * TS] = aL; nx[(ND + 3) * TS] = rho_inv; nx[(ND + 4) * TS] = rq;
        nx[(ND + 5) * TS] = fmin(fmin(100.0 * h0, h1), span);
    }
}

template <bool JOINT>
__device__ __forceinline__ void state_warp(const IndirectArgs& a, int t, int lane, unsigned char* smem) {
    const TileSmem S = tile_smem(smem, t);
    const int slot = lane;
    const unsigned fullmask = 0xffffffffu;
    const double atol = a.cfg.atol, rtol = a.cfg.rtol;
    const double inv_ne = JOINT ? 1.0 / (double)(ND * (ND + 1)) : 1.0 / (double)ND;
    const bool bulk = (reinterpret_cast<uintptr_t>(a.phi) & 15u) == 0;
    int xi = 0;                                                           // which half of the double buffer holds x
    double* const xbuf = S.xn + slot;
#pragma unroll
    for (int i = 0; i < ND; ++i) { xbuf[i * TS] = 0.0; xbuf[(ND + i) * TS] = 0.0; }
    double tcur = 0.0, tf = 0.0, h = 0.0, span = 1.0, esum = 0.0;
    LawConst lw; lw.aL = 0.0; lw.rho_inv = 1.0; lw.rho_inv_quarter_aL = 0.0;
    long long seg = -1, ia = 0;
    int na = 0, nt = 0, status = 0;
    bool active = false, lastrej = false, last = false, have = false, exhausted = false;
    long long nseg = -1;                                                  // successor segment claimed and staged by prepare_next()
    unsigned visit = 0;
    double2* rec = S.rec + slot;
    long long c_wait = 0, c_work = 0, c_pre = 0;
    const long long c_begin = clock64();
    prepare_next(a, S, slot, nseg, exhausted, true);
    while (true) {
        int flags = 0, store_seg = 0;
        bool finished = false;
        const long long c0 = clock64();
        long long c1 = c0;
        if (have) {
            mbar_wait_parked(S.bar_done, (visit - 1) & 1);
            c1 = clock64();
            c_wait += c1 - c0;
            if (active) {
                double s2 = esum;
                if (JOINT) {
#pragma unroll
                    for (int c = 0; c < ND; ++c) s2 += S.errp[c * TS + slot];
                }
                const double u = s2 * inv_ne;                           // eest^2: eest <= 1 <=> u <= 1, eest^(-1/8) = u^(-1/16)
                if (!(u == u)) { status = LTO_ST_NAN; finished = true; }
                else {
                    double q = (u == 0.0) ? 5.0 : ((u < 1e300) ? 0.9 * inv_sixteenth_root(u) : 0.2);
                    q = fmin(5.0, fmax(0.2, q));
                    if (u <= 1.0) {
                        ++na; flags |= F_ACCEPT;
                        xi ^= 1;                                          // the candidate becomes x
                        if (last) { tcur = tf; finished = true; }
                        else { tcur += h; if (lastrej) q = fmin(q, 1.0); lastrej = false; }
                    } else {
                        lastrej = true; q = fmin(q, 1.0);
                    }
                    h *= q;
                }
            }
        }
        if (active && !finished) {                                       // drive_rk8's loop-top checks
            if (h < span * 1e-12) { status = LTO_ST_HMIN; finished = true; }
            else if (nt >= a.cfg.max_attempts) { status = LTO_ST_MAXSTEPS; finished = true; }
        }
        if (active && finished) {
            // ---- defect = x(t1) - XC_all[:, i+1] (multiShoot_CRTBP_indirect.jl:82)
            bool nan = false;
            const double* xs = xbuf + xi * ND * TS;
#pragma unroll
            for (int i = 0; i < ND; ++i) {
                const double xv = xs[i * TS];
                nan |= !(xv == xv);
                a.defect[seg * ND + i] = a.x_target ? xv - a.x_target[ia * ND + i] : xv;
            }
            if (nan && status == 0) status = LTO_ST_NAN;
            if (a.status) a.status[seg] = status;
            if (a.nsteps_out) { a.nsteps_out[2 * seg] = na; a.nsteps_out[2 * seg + 1] = nt; }
            // column j of ForwardDiff.jacobian(f, x0) (:121) is the slot's stash row j: after an accepted last step the stash IS the STM
            if (bulk && (flags & F_ACCEPT)) bulk_store(a.phi + seg * (long long)(ND * ND), smem_u32(S.cur + (size_t)slot * STASH_STRIDE), ND * ND * sizeof(double));
            else flags |= F_STORE;                                      // ended in error (the last accepted columns are in the L2 scratch), or unaligned `phi`
            store_seg = (int)seg;
            active = false;
        }
        auto take_successor = [&]() {                                    // the successor prepared by prepare_next()
            if (!active && nseg >= 0) {
                seg = nseg; nseg = -1; ia = lto_node_a(seg, a.npt);
                const double* nx = S.nx + slot;
#pragma unroll
                for (int i = 0; i < ND; ++i) xbuf[(xi * ND + i) * TS] = nx[i * TS];
                tcur = nx[(ND + 0) * TS]; tf = nx[(ND + 1) * TS];
                span = tf - tcur;
                lw.aL = nx[(ND + 2) * TS]; lw.rho_inv = nx[(ND + 3) * TS]; lw.rho_inv_quarter_aL = nx[(ND + 4) * TS];
                h = nx[(ND + 5) * TS];
                na = 0; nt = 0; status = 0; lastrej = false;
                active = true; flags |= F_RESET;
            }
        };
        take_successor();
        if (!__any_sync(fullmask, active)) {                             // nobody has work (only after segments ended in error): claim on demand
            prepare_next(a, S, slot, nseg, exhausted, true);
            take_successor();
        }
        if (!__any_sync(fullmask, active)) {
            S.hval[slot] = 0.0; S.hctl[slot] = make_int2(flags, store_seg);
            if (lane == 0) *S.tile_done = 1;
            mbar_arrive(S.bar_full);
            bulk_store_wait_all();                                       // the last bulk stores must have completed before the CTA retires
            break;
        }
        // ---- one attempted step (13 stages); a fresh slot first picks its initial step
        const long long c2 = clock64();
        c_pre += c2 - c1;
        KStore K;
        const double* xs = xbuf + xi * ND * TS;
        state_stage_s<0>(K, xs, 0.0, 0.0, a.c, lw, rec, S.bar_full);
        last = false;
        if (tcur + h >= tf) { h = tf - tcur; last = true; }
        if (active) ++nt;
        S.hval[slot] = h; S.hctl[slot] = make_int2(flags | (active ? F_ACTIVE : 0), store_seg);
        if (STAGE_PIPE) mbar_arrive(S.bar_full);                         // header + stage 0
        const double h2 = h * h;
        state_stage_s<1>(K, xs, h, h2, a.c, lw, rec, S.bar_full);  state_stage_s<2>(K, xs, h, h2, a.c, lw, rec, S.bar_full);  state_stage_s<3>(K, xs, h, h2, a.c, lw, rec, S.bar_full);
        state_stage_s<4>(K, xs, h, h2, a.c, lw, rec, S.bar_full);  state_stage_s<5>(K, xs, h, h2, a.c, lw, rec, S.bar_full);  state_stage_s<6>(K, xs, h, h2, a.c, lw, rec, S.bar_full);
        state_stage_s<7>(K, xs, h, h2, a.c, lw, rec, S.bar_full);  state_stage_s<8>(K, xs, h, h2, a.c, lw, rec, S.bar_full);  state_stage_s<9>(K, xs, h, h2, a.c, lw, rec, S.bar_full);
        state_stage_s<10>(K, xs, h, h2, a.c, lw, rec, S.bar_full); state_stage_s<11>(K, xs, h, h2, a.c, lw, rec, S.bar_full); state_stage_s<12>(K, xs, h, h2, a.c, lw, rec, S.bar_full);
        {
            double x[ND], xn[ND];
#pragma unroll
            for (int i = 0; i < ND; ++i) x[i] = xs[i * TS];
            esum = step_finish<true, !JOINT>(K, x, h, h2, atol, rtol, xn);
            double* xc = xbuf + (xi ^ 1) * ND * TS;
#pragma unroll
            for (int i = 0; i < ND; ++i) xc[i * TS] = xn[i];
        }
        bulk_store_wait_read();                                          // the column warps overwrite the stash in this visit
        if (!STAGE_PIPE) mbar_arrive(S.bar_full);                        // the whole attempt's record
        c_work += clock64() - c2;
        have = true; ++visit;
        prepare_next(a, S, slot, nseg, exhausted, last || !active);      // while the column warps work on this attempt
    }
    if (a.prof && lane == 0) {
        unsigned long long* o = a.prof + ((size_t)blockIdx.x * NW + t) * 4;
        o[0] = c_work; o[1] = c_wait; o[2] = visit; o[3] = clock64() - c_begin;
        a.prof[(size_t)gridDim.x * NW * 4 + (size_t)blockIdx.x * NTILE + t] = c_pre;
    }
}

template <bool JOINT>
__global__ void __launch_bounds__(NTHREADS, 1) k_indirect_cw(IndirectArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < NTILE) {
        const TileSmem S = tile_smem(smem_raw, threadIdx.x);
        for (int j = 0; j < 13; ++j) mbar_init(S.bar_full + 8 * j, 32);
        mbar_init(S.bar_done, NCT);
        *S.tile_done = 0;
    }
    __syncthreads();
    // warps 3 and 7 (both on SM sub-partition 3) are the state warps; the other three sub-partitions
    // each host two column warps that run the same instruction stream side by side
    if ((warp & 3) == 3) state_warp<JOINT>(a, warp >> 2, lane, smem_raw);
    else column_warp<JOINT>(a, warp - (warp >> 2), lane, smem_raw);
}

// ---------------------------------------------------------------------------
// K4 (indirect): defect-only -- defectCalc of multiShoot_CRTBP_indirect.jl:63-90 as the SOC step (:197), the
// 20-point line search (:232-241) and the per-iteration check (:328) call it.  One lane per segment slot, the
// same RK step, controller and work queue as the state warps above, with nothing published: every warp of the
// CTA is a "state warp".  Step control over the state alone (a plain `solve`, no dual numbers).
// ---------------------------------------------------------------------------
#ifndef LTO_K4I_INLINE
#define LTO_K4I_INLINE 0
#endif
__device__ __noinline__ Out9 sc_eval_state_call(double r0, double r1, double r2, double v0, double v1, double v2, double l0, double l1, double l2,
                                                double m0, double m1, double m2, double mu, double mu1, double omega, double pexp, double aL,
                                                double rho_inv, double rq) {
    const double R[3] = {r0, r1, r2}, V[3] = {v0, v1, v2}, L[3] = {l0, l1, l2}, M[3] = {m0, m1, m2};
    SCConst c; c.mu = mu; c.m1 = mu1; c.omega = omega; c.p = pexp;
    LawConst lw; lw.aL = aL; lw.rho_inv = rho_inv; lw.rho_inv_quarter_aL = rq;
    double kv[3], kl[3], km[3];
    sc_eval<false>(R, V, L, M, c, lw, kv, kl, km, nullptr);
    Out9 o;
#pragma unroll
    for (int q = 0; q < 3; ++q) { o.v[q] = kv[q]; o.v[3 + q] = kl[q]; o.v[6 + q] = km[q]; }
    return o;
}

template <int J>
__device__ __forceinline__ void state_only_stage(KStore& K, const double (&x)[ND], double h, double h2, const SCConst& c, const LawConst& lw) {
    double R[3], V[3], L[3], M[3];
    stage_input<J>(K, x, h, h2, R, V, L, M);
#if LTO_K4I_INLINE
    double kv[3], kl[3], km[3];
    sc_eval<false>(R, V, L, M, c, lw, kv, kl, km, nullptr);
#pragma unroll
    for (int q = 0; q < 3; ++q) { K.kv[J][q] = kv[q]; K.kl[J][q] = kl[q]; K.km[J][q] = km[q]; }
#else
    const Out9 o = sc_eval_state_call(R[0], R[1], R[2], V[0], V[1], V[2], L[0], L[1], L[2], M[0], M[1], M[2], c.mu, c.m1, c.omega, c.p, lw.aL,
                                      lw.rho_inv, lw.rho_inv_quarter_aL);
#pragma unroll
    for (int q = 0; q < 3; ++q) { K.kv[J][q] = o.v[q]; K.kl[J][q] = o.v[3 + q]; K.km[J][q] = o.v[6 + q]; }
#endif
}

// The cost pass's stage: sc_eval_state_call's derivatives plus the stage's thrust-acceleration magnitude |a_u| = umag of the control
// law (CRTBP_stateCostate_deriv.jl:36-53: zero when |lv| = 0, the clamped branch for p > 1) in v[9].
struct Out10 { double v[10]; };
__device__ __noinline__ Out10 sc_eval_quad_call(double r0, double r1, double r2, double v0, double v1, double v2, double l0, double l1, double l2,
                                                double m0, double m1, double m2, double mu, double mu1, double omega, double pexp, double aL,
                                                double rho_inv, double rq) {
    const double R[3] = {r0, r1, r2}, V[3] = {v0, v1, v2}, L[3] = {l0, l1, l2}, M[3] = {m0, m1, m2};
    SCConst c; c.mu = mu; c.m1 = mu1; c.omega = omega; c.p = pexp;
    LawConst lw; lw.aL = aL; lw.rho_inv = rho_inv; lw.rho_inv_quarter_aL = rq;
    double kv[3], kl[3], km[3];
    Out10 o;
    sc_eval<false>(R, V, L, M, c, lw, kv, kl, km, nullptr, &o.v[9]);
#pragma unroll
    for (int q = 0; q < 3; ++q) { o.v[q] = kv[q]; o.v[3 + q] = kl[q]; o.v[6 + q] = km[q]; }
    return o;
}

// Stage J of K4.  QUAD: also s_dv += b_J umag_J and s_e += b_J umag_J^2 with the weights b of the 8th-order update (step_finish), so
// that h s_dv and h s_e are the update's quadratures of |a_u| and |a_u|^2 over the step.
template <int J, bool QUAD>
__device__ __forceinline__ void k4_stage(KStore& K, const double (&x)[ND], double h, double h2, const SCConst& c, const LawConst& lw,
                                         double& s_dv, double& s_e) {
    if (!QUAD) { state_only_stage<J>(K, x, h, h2, c, lw); return; }
    double R[3], V[3], L[3], M[3];
    stage_input<J>(K, x, h, h2, R, V, L, M);
    const Out10 o = sc_eval_quad_call(R[0], R[1], R[2], V[0], V[1], V[2], L[0], L[1], L[2], M[0], M[1], M[2], c.mu, c.m1, c.omega, c.p, lw.aL,
                                      lw.rho_inv, lw.rho_inv_quarter_aL);
#pragma unroll
    for (int q = 0; q < 3; ++q) { K.kv[J][q] = o.v[q]; K.kl[J][q] = o.v[3 + q]; K.km[J][q] = o.v[6 + q]; }
    if (J == 0) { s_dv = 0.0; s_e = 0.0; }
    if (lto_tab::CHIf(J) != 0.0) {
        const double u = o.v[9];
        s_dv = fma(lto_tab::CHIf(J), u, s_dv);
        s_e = fma(lto_tab::CHIf(J), u * u, s_e);
    }
}

// The switch pass's scan of one accepted step [t, t + h] from x (start) to xn (end), out of line so that K4's main loop does not grow:
// writes the step's switches after the segment's `count` (at most `cap` per segment) and returns the new count (lto_switch.h).
__device__ __noinline__ int sw_step_call(double r0, double r1, double r2, double lr0, double lr1, double lr2, double lv0, double lv1, double lv2,
                                         double s0, double s1, double s2, double sr0, double sr1, double sr2, double sv0, double sv1, double sv2,
                                         double mu, double mu1, double omega, double t, double h, int count, int cap, double* t_out,
                                         int32_t* dir_out) {
    SwEnd e0, e1;
    sw_end(r0, r1, r2, lr0, lr1, lr2, lv0, lv1, lv2, mu, mu1, omega, e0);
    sw_end(s0, s1, s2, sr0, sr1, sr2, sv0, sv1, sv2, mu, mu1, omega, e1);
    return sw_scan(e0, e1, t, h, count, cap, t_out, dir_out);
}

constexpr int K4I_THREADS = 128;

// QUAD = false: the defect-only kernel k_indirect_state.  QUAD = true (k_indirect_state_cost): the same steps (the quadratures are not in
// the error norm, so the step sequence and every state are bitwise those of QUAD = false) and, per segment, a.quad[2 seg] =
// int |a_u| dt and a.quad[2 seg + 1] = int |a_u|^2 dt, accumulated over the accepted steps only (NaN for a segment whose status is not
// LTO_ST_OK: it never reached t1).  SW (k_indirect_state_switch): the same steps again (the scan is not in the error norm either) and,
// per segment, the switches of |lv| - 1 located on every accepted step (sw_step_call) in a.sw_t / a.sw_dir (at most a.max_switch),
// their count in a.sw_count (0 for a segment whose status is not LTO_ST_OK) and the sides of |lv| - 1 at the segment's start and
// propagated end in a.sw_side.  `a` is taken by value: so
// k_indirect_state compiles to the same SASS as when this body was its own (through a reference, the register allocation changed).
template <bool QUAD, bool SW>
__device__ __forceinline__ void k4_body(IndirectArgs a) {
    const unsigned fullmask = 0xffffffffu;
    double atol = a.cfg.atol, rtol = a.cfg.rtol;                          // per slot: state_tol_scale(p, rho) of the slot's segment
    double x[ND], xn[ND];
#pragma unroll
    for (int i = 0; i < ND; ++i) { x[i] = 0.0; xn[i] = 0.0; }
    double tcur = 0.0, tf = 0.0, h = 0.0, span = 1.0, esum = 0.0;
    LawConst lw; lw.aL = 0.0; lw.rho_inv = 1.0; lw.rho_inv_quarter_aL = 0.0;
    long long seg = -1, ia = 0;
    int na = 0, nt = 0, status = 0;
    bool active = false, lastrej = false, last = false, have = false, exhausted = false;
    double q_dv = 0.0, q_e = 0.0, s_dv = 0.0, s_e = 0.0;                  // QUAD: the segment's quadratures and the attempted step's sums
    int n_sw = 0;                                                         // SW: the segment's switches so far
    while (true) {
        bool finished = false;
        if (have && active) {
            const double eest = sqrt(esum * (1.0 / (double)ND));
            if (!(eest == eest)) { status = LTO_ST_NAN; finished = true; }
            else {
                double q = (eest == 0.0) ? 5.0 : 0.9 * inv_eighth_root(eest);
                q = fmin(5.0, fmax(0.2, q));
                if (eest <= 1.0) {
                    ++na;
                    if (SW)
                        n_sw = sw_step_call(x[0], x[1], x[2], x[6], x[7], x[8], x[9], x[10], x[11], xn[0], xn[1], xn[2], xn[6], xn[7], xn[8],
                                            xn[9], xn[10], xn[11], a.c.mu, a.c.m1, a.c.omega, tcur, h, n_sw, a.max_switch,
                                            a.sw_t + seg * a.max_switch, a.sw_dir + seg * a.max_switch);
#pragma unroll
                    for (int i = 0; i < ND; ++i) x[i] = xn[i];
                    if (QUAD) { q_dv = fma(h, s_dv, q_dv); q_e = fma(h, s_e, q_e); }
                    if (last) { tcur = tf; finished = true; }
                    else { tcur += h; if (lastrej) q = fmin(q, 1.0); lastrej = false; }
                } else {
                    lastrej = true; q = fmin(q, 1.0);
                }
                h *= q;
            }
        }
        if (active && !finished) {
            if (h < span * 1e-12) { status = LTO_ST_HMIN; finished = true; }
            else if (nt >= a.cfg.max_attempts) { status = LTO_ST_MAXSTEPS; finished = true; }
        }
        if (active && finished) {
            bool nan = false;
#pragma unroll
            for (int i = 0; i < ND; ++i) nan |= !(x[i] == x[i]);
            if (nan && status == 0) status = LTO_ST_NAN;
#pragma unroll
            for (int i = 0; i < ND; ++i) a.defect[seg * ND + i] = a.x_target ? x[i] - a.x_target[ia * ND + i] : x[i];   // :82
            if (a.status) a.status[seg] = status;
            if (a.nsteps_out) { a.nsteps_out[2 * seg] = na; a.nsteps_out[2 * seg + 1] = nt; }
            if (QUAD) {                                                   // a segment that did not reach t1 has no cost: NaN
                const double nanv = __longlong_as_double(0x7ff8000000000000ll);
                a.quad[2 * seg] = status ? nanv : q_dv; a.quad[2 * seg + 1] = status ? nanv : q_e;
            }
            if (SW) {                                                     // a segment that did not reach t1 has no switches
                a.sw_count[seg] = status ? 0 : n_sw;
                a.sw_side[seg] = sw_side(a.x0[ia * ND + 9], a.x0[ia * ND + 10], a.x0[ia * ND + 11]) | (sw_side(x[9], x[10], x[11]) << 1);
            }
            active = false;
        }
        bool fresh = false;
        if (!active && !exhausted) {
            const long long idx = (long long)atomicAdd(a.counter, 1ull);
            if (idx < a.n_seg) {
                seg = idx; ia = lto_node_a(seg, a.npt);
                const long long it = lto_traj_of(seg, a.npt);
#pragma unroll
                for (int i = 0; i < ND; ++i) x[i] = a.x0[ia * ND + i];
                tcur = a.t0[ia]; tf = a.t1[ia];
                if (!(tcur < tf)) tf = tcur;
                span = tf - tcur;
                const double tl = a.thrustLimit_arr ? a.thrustLimit_arr[it] : a.c.thrustLimit;
                const double rho = a.rho_arr ? a.rho_arr[it] : a.c.rho;
                lw.aL = tl * a.c.kthr / a.c.mass;                         // CRTBP_stateCostate_deriv.jl:33
                lw.rho_inv = 1.0 / rho;
                lw.rho_inv_quarter_aL = lw.aL / (4.0 * rho);
                { const double ts = state_tol_scale(a.c.p, rho); atol = a.cfg.atol * ts; rtol = a.cfg.rtol * ts; }
                na = 0; nt = 0; status = 0; lastrej = false;
                if (QUAD) { q_dv = 0.0; q_e = 0.0; }
                if (SW) n_sw = 0;
                active = true; fresh = true;
            } else {
                exhausted = true;
            }
        }
        if (!__any_sync(fullmask, active)) break;
        KStore K;
        k4_stage<0, QUAD>(K, x, 0.0, 0.0, a.c, lw, s_dv, s_e);
        if (__any_sync(fullmask, fresh)) {
            // Hairer-Norsett-Wanner initial step (drive_rk8 in lto_prop_generic.cuh)
            double f0[ND], y1[ND];
#pragma unroll
            for (int q = 0; q < 3; ++q) { f0[q] = x[3 + q]; f0[3 + q] = K.kv[0][q]; f0[6 + q] = K.kl[0][q]; f0[9 + q] = K.km[0][q]; }
            const double d0 = rms12(x, x, atol, rtol), d1 = rms12(f0, x, atol, rtol);
            double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * (d0 / d1);
            h0 = fmin(h0, span);
#pragma unroll
            for (int i = 0; i < ND; ++i) y1[i] = fma(h0, f0[i], x[i]);
            {
                const double R1[3] = {y1[0], y1[1], y1[2]}, V1[3] = {y1[3], y1[4], y1[5]}, L1[3] = {y1[6], y1[7], y1[8]}, M1[3] = {y1[9], y1[10], y1[11]};
                double kv1[3], kl1[3], km1[3];
                sc_eval<false>(R1, V1, L1, M1, a.c, lw, kv1, kl1, km1, nullptr);
#pragma unroll
                for (int q = 0; q < 3; ++q) { y1[q] = V1[q] - f0[q]; y1[3 + q] = kv1[q] - f0[3 + q]; y1[6 + q] = kl1[q] - f0[6 + q]; y1[9 + q] = km1[q] - f0[9 + q]; }
            }
            const double d2 = rms12(y1, x, atol, rtol) / h0;
            const double dm = fmax(d1, d2);
            const double h1 = (dm <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : inv_eighth_root(dm / 0.01);
            if (fresh) h = fmin(fmin(100.0 * h0, h1), span);
        }
        last = false;
        if (tcur + h >= tf) { h = tf - tcur; last = true; }
        if (active) ++nt;
        const double h2 = h * h;
        k4_stage<1, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);  k4_stage<2, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);  k4_stage<3, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);
        k4_stage<4, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);  k4_stage<5, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);  k4_stage<6, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);
        k4_stage<7, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);  k4_stage<8, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);  k4_stage<9, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);
        k4_stage<10, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e); k4_stage<11, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e); k4_stage<12, QUAD>(K, x, h, h2, a.c, lw, s_dv, s_e);
        esum = step_finish<true, true>(K, x, h, h2, atol, rtol, xn);
        have = true;
    }
}

__global__ void __launch_bounds__(K4I_THREADS, 2) k_indirect_state(IndirectArgs a) { k4_body<false, false>(a); }
__global__ void __launch_bounds__(K4I_THREADS, 2) k_indirect_state_cost(IndirectArgs a) { k4_body<true, false>(a); }
__global__ void __launch_bounds__(K4I_THREADS, 2) k_indirect_state_switch(IndirectArgs a) { k4_body<false, true>(a); }

}  // namespace icw

size_t indirect_cwv2_scratch_bytes(int n_sm) {
    return (size_t)n_sm * icw::SCRATCH_BYTES_PER_CTA;
}

template <bool JOINT>
static cudaError_t launch_icw(const IndirectArgs& a, cudaStream_t st) {
    // per device: a single process may drive several GPUs (lto_init_devices)
    static int n_sm_dev[64] = {0};
    static bool attr_dev[64] = {false};
    int dev = 0;
    { cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e; }
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (!attr_dev[dev]) {
        cudaError_t e = cudaDeviceGetAttribute(&n_sm_dev[dev], cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(icw::k_indirect_cw<JOINT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)icw::SMEM);
        if (e != cudaSuccess) return e;
        attr_dev[dev] = true;
    }
    const int n_sm = n_sm_dev[dev];
    cudaError_t e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    const long long per_cta = (long long)icw::NTILE * icw::TS;
    const int grid = (int)std::min<long long>((a.n_seg + per_cta - 1) / per_cta, (long long)n_sm);
    icw::k_indirect_cw<JOINT><<<grid, icw::NTHREADS, icw::SMEM, st>>>(a);
    return cudaGetLastError();
}

static cudaError_t launch_k4i(const IndirectArgs& a, cudaStream_t st) {
    int dev = 0, n_sm = 0;
    cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned long long), st); if (e != cudaSuccess) return e;
    const long long blocks = (a.n_seg + icw::K4I_THREADS - 1) / icw::K4I_THREADS;
    const int grid = (int)std::min<long long>(blocks, (long long)n_sm * 2);
    icw::k_indirect_state<<<grid, icw::K4I_THREADS, 0, st>>>(a);
    return cudaGetLastError();
}

namespace icw {
// Per trajectory, its segments' quadratures summed in segment order (no atomics: the sum does not depend on the batch around it).
__global__ void k_cost_sum(const double* __restrict__ quad, const int32_t* __restrict__ seg_status, long long n_traj, int seg_per_traj,
                           double dv_scale, double e_scale, double* __restrict__ dv, double* __restrict__ energy, int32_t* __restrict__ status) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_traj) return;
    double sd = 0.0, se = 0.0;
    int w = 0;
    for (int i = 0; i < seg_per_traj; ++i) {
        const long long s = j * seg_per_traj + i;
        sd += quad[2 * s]; se += quad[2 * s + 1];
        w = max(w, (int)seg_status[s]);
    }
    dv[j] = sd * dv_scale; energy[j] = se * e_scale;
    if (status) status[j] = w;
}
}  // namespace icw

cudaError_t launch_indirect_cost(const IndirectArgs& a, long long n_traj, double dv_scale, double e_scale, double* dv, double* energy,
                                 int32_t* status_traj, cudaStream_t st, int* n_launch) {
    *n_launch = 0;
    if (a.phi != nullptr || a.counter == nullptr || a.quad == nullptr || a.status == nullptr || a.cfg.controller != 0 || a.npt < 2 ||
        a.n_seg <= 0 || a.n_seg > 0x7fffffffll || a.n_seg != n_traj * (a.npt - 1))
        return cudaErrorNotSupported;
    int dev = 0, n_sm = 0;
    cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned long long), st); if (e != cudaSuccess) return e;
    const long long blocks = (a.n_seg + icw::K4I_THREADS - 1) / icw::K4I_THREADS;
    const int grid = (int)std::min<long long>(blocks, (long long)n_sm * 2);
    icw::k_indirect_state_cost<<<grid, icw::K4I_THREADS, 0, st>>>(a);
    e = cudaGetLastError(); if (e != cudaSuccess) return e;
    *n_launch = 1;
    icw::k_cost_sum<<<(unsigned)((n_traj + 127) / 128), 128, 0, st>>>(a.quad, a.status, n_traj, a.npt - 1, dv_scale, e_scale, dv, energy,
                                                                      status_traj);
    e = cudaGetLastError(); if (e != cudaSuccess) return e;
    *n_launch = 2;
    return cudaSuccess;
}

namespace icw {
// Per trajectory, its segments' switches in time order with the node rule between them: where the side of |lv| - 1 at segment i's
// propagated end and at node i + 1 (segment i + 1's start) differ, one switch at t_{i+1} in the direction of node i + 1's side.  The
// first `cap` switches are written (NaN / 0 in the unused slots), n_switch is the true total (-1 where the worst segment status is not
// LTO_ST_OK).  No atomics: a row's result does not depend on the batch around it.
__global__ void k_switch_gather(const int32_t* __restrict__ seg_status, const int32_t* __restrict__ sw_count, const int32_t* __restrict__ sw_side,
                                const double* __restrict__ sw_t, const int32_t* __restrict__ sw_dir, const double* __restrict__ t_node,
                                long long n_traj, int npt, int cap, double* __restrict__ t_switch, int32_t* __restrict__ direction,
                                int32_t* __restrict__ n_switch, int32_t* __restrict__ on_start, int32_t* __restrict__ status) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_traj) return;
    const int ns = npt - 1;
    const long long s0 = j * ns;
    int w = 0;
    for (int i = 0; i < ns; ++i) w = max(w, (int)seg_status[s0 + i]);
    double* to = t_switch + j * cap;
    int32_t* dout = direction + j * cap;
    int n = 0;
    if (w == 0) {
        int end_prev = 0;
        for (int i = 0; i < ns; ++i) {
            const long long s = s0 + i;
            const int sd = sw_side[s];
            if (i > 0 && (sd & 1) != end_prev) {                          // the node rule at t_i
                if (n < cap) { to[n] = t_node[j * npt + i]; dout[n] = (sd & 1) ? 1 : -1; }
                ++n;
            }
            const int c = sw_count[s];
            for (int k = 0; k < c && k < cap && n + k < cap; ++k) { to[n + k] = sw_t[s * cap + k]; dout[n + k] = sw_dir[s * cap + k]; }
            n += c;
            end_prev = sd >> 1;
        }
    }
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    for (int k = w == 0 ? min(n, cap) : 0; k < cap; ++k) { to[k] = nanv; dout[k] = 0; }
    n_switch[j] = w ? -1 : n;
    on_start[j] = sw_side[s0] & 1;
    if (status) status[j] = w;
}
}  // namespace icw

cudaError_t launch_indirect_switch(const IndirectArgs& a, long long n_traj, const double* t_node, double* t_switch, int32_t* direction,
                                   int32_t* n_switch, int32_t* on_start, int32_t* status_traj, cudaStream_t st, int* n_launch) {
    *n_launch = 0;
    if (a.phi != nullptr || a.counter == nullptr || a.status == nullptr || a.sw_t == nullptr || a.sw_dir == nullptr || a.sw_count == nullptr ||
        a.sw_side == nullptr || a.max_switch < 1 || a.cfg.controller != 0 || a.npt < 2 || a.n_seg <= 0 || a.n_seg > 0x7fffffffll ||
        a.n_seg != n_traj * (a.npt - 1))
        return cudaErrorNotSupported;
    int dev = 0, n_sm = 0;
    cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned long long), st); if (e != cudaSuccess) return e;
    const long long blocks = (a.n_seg + icw::K4I_THREADS - 1) / icw::K4I_THREADS;
    const int grid = (int)std::min<long long>(blocks, (long long)n_sm * 2);
    icw::k_indirect_state_switch<<<grid, icw::K4I_THREADS, 0, st>>>(a);
    e = cudaGetLastError(); if (e != cudaSuccess) return e;
    *n_launch = 1;
    icw::k_switch_gather<<<(unsigned)((n_traj + 127) / 128), 128, 0, st>>>(a.status, a.sw_count, a.sw_side, a.sw_t, a.sw_dir, t_node, n_traj,
                                                                           a.npt, a.max_switch, t_switch, direction, n_switch, on_start,
                                                                           status_traj);
    e = cudaGetLastError(); if (e != cudaSuccess) return e;
    *n_launch = 2;
    return cudaSuccess;
}

cudaError_t launch_indirect_cw(const IndirectArgs& a, int ndim, cudaStream_t st, int* n_launch) {
    *n_launch = 0;
    if (ndim == 12 && a.phi == nullptr && a.counter != nullptr && a.cfg.controller == 0 && a.n_seg > 0 && a.n_seg <= 0x7fffffffll) {
        cudaError_t e = launch_k4i(a, st);
        if (e == cudaSuccess) *n_launch = 1;
        return e;
    }
    if (ndim != 12 || a.phi == nullptr || a.counter == nullptr || a.scratch == nullptr || a.cfg.controller != 0 || a.n_seg <= 0 ||
        a.n_seg > 0x7fffffffll)
        return cudaErrorNotSupported;
    const cudaError_t e = (a.cfg.err_norm != 0) ? launch_icw<true>(a, st) : launch_icw<false>(a, st);
    if (e == cudaSuccess) *n_launch = 1;
    return e;
}

}  // namespace lto
