// lto_direct_qp.cu -- the linear subproblem of the DIRECT solver on the device, batched over trajectories
// (SURVEY section 8(f) row 4): optimizeTraj of src/multiShoot_CRTBP_direct.jl:248-403 in the setting the demo runs
// (flagEnd = false, allowImpulsive = false): every bound of the JuMP model collapses to an equality (tf_jump, p1_jump, p2_jump,
// dV_jump pinned, :288-302), so the problem Ipopt is handed is the equality-constrained convex QP
//
//     min  sum_i w_i |u_i + du_i|^2                                   (quadCost :367-368, w from the node spacing :323-325)
//     s.t. defect + Jac_full [dX; du] = 0                              (:337, the linearised dynamics)
//          dX_1[1:6] = b0,  dX_N[1:6] = bf  (+ dX_1[7] = mass - X_all[7,1] when nstate = 7)   (:270, :374-375)
//
// whose KKT conditions are ONE symmetric indefinite linear system.  Ordering the unknowns node by node
//     [nu_0 | dX_1 du_1 lambda_1 | dX_2 du_2 lambda_2 | ... | dX_N du_N | nu_f]
// makes it banded with half-bandwidth 2 nstate + 2 (14 / 16): 456 / 516 unknowns for the demo's 30 nodes.  The matrix is
// never assembled: a row's entries are generated from the Jacobian blocks of lto_direct_defect_jac[_traj] at the moment the
// row enters the elimination window.
//
// Solver: Gaussian elimination with partial pivoting inside the band (LAPACK dgbsv's algorithm), ONE WARP PER TRAJECTORY.
// The active window -- rows j..j+bw, columns j..j+2bw (the upper band doubles through row interchanges) -- lives in shared
// memory as a 32 x 64 circular buffer; lanes are the window's columns (2 bw <= 32), the multipliers are applied to the
// right-hand side on the fly, finished pivot rows go to an HBM workspace for the back substitution.
#include "lto_internal.h"
#include "lto_cw_common.cuh"
#include <algorithm>

namespace lto {
namespace dqp {

constexpr int WR = 32, WC = 64;               // window rows / columns (circular)
constexpr int UROW = 34;                      // stored pivot row: pivot, 32 upper entries, rhs
constexpr int WARPS = 4;
constexpr int SM_PER_WARP = WR * WC + WR + WC;   // window, rhs, solution window (doubles)

enum { K_NU0 = 0, K_X = 1, K_U = 2, K_L = 3, K_NUF = 4 };
struct Idx { int kind, node, comp; };

template <int NS>
struct Geo {
    static constexpr int B = 2 * NS + 3;               // unknowns per interior node: dX, du, lambda
    static constexpr int M0 = 6 + (NS == 7 ? 1 : 0);   // initial-state constraints (:270, :374)
    static constexpr int BW = 2 * NS + 2;              // half-bandwidth
    static_assert(2 * BW <= 32, "one lane per window column");
    __host__ __device__ static int total(int N) { return M0 + (N - 1) * B + NS + 3 + 6; }
    __device__ static Idx decode(int R, int N) {
        Idx d;
        if (R < M0) { d.kind = K_NU0; d.node = 0; d.comp = R; return d; }
        R -= M0;
        d.node = R / B;
        const int off = R - d.node * B;
        if (off < NS) { d.kind = K_X; d.comp = off; }
        else if (off < NS + 3) { d.kind = K_U; d.comp = off - NS; }
        else { d.kind = (d.node == N - 1) ? K_NUF : K_L; d.comp = off - NS - 3; }
        return d;
    }
};

struct QpArgs {
    const double *jac, *defect, *X_all, *u_all, *t, *b0, *bf;
    double *work, *x_update, *u_update;
    int32_t* status;
    long long n_traj;
    int n_nodes;
};

__device__ __forceinline__ double node_weight(const double* __restrict__ t, int i, int N) {
    // dt_temp of :323-325: half the spacing on either side of the node
    double w = 0.0;
    if (i < N - 1) w += 0.5 * (t[i + 1] - t[i]);
    if (i > 0) w += 0.5 * (t[i] - t[i - 1]);
    else if (N == 1) w = 0.0;
    return w;
}

// K[a][b] of the KKT matrix (symmetric); jac: per segment NS x 2(NS+3) column-major blocks [X_i, X_{i+1}, u_i, u_{i+1}] (:125)
template <int NS>
__device__ __forceinline__ double kkt_entry(int a, int b, int N, const double* __restrict__ jac, const double* __restrict__ t) {
    typedef Geo<NS> G;
    if (a < 0 || b < 0 || a >= G::total(N) || b >= G::total(N)) return 0.0;
    Idx p = G::decode(a, N), q = G::decode(b, N);
    if (q.kind == K_L || q.kind == K_NU0 || q.kind == K_NUF) { const Idx s = p; p = q; q = s; }   // p: multiplier (if any), q: variable
    if (p.kind == K_L) {
        int col = -1;
        if (q.kind == K_X) { if (q.node == p.node) col = q.comp; else if (q.node == p.node + 1) col = NS + q.comp; }
        else if (q.kind == K_U) { if (q.node == p.node) col = 2 * NS + q.comp; else if (q.node == p.node + 1) col = 2 * NS + 3 + q.comp; }
        if (col < 0) return 0.0;
        return -jac[((long long)p.node * (2 * (NS + 3)) + col) * NS + p.comp];                  // A_dyn = -Jac_full (:337)
    }
    if (p.kind == K_NU0) return (q.kind == K_X && q.node == 0 && q.comp == p.comp) ? 1.0 : 0.0;
    if (p.kind == K_NUF) return (q.kind == K_X && q.node == N - 1 && q.comp == p.comp) ? 1.0 : 0.0;
    if (p.kind == K_U && q.kind == K_U && p.node == q.node && p.comp == q.comp) return 2.0 * node_weight(t, p.node, N);   // Hessian of quadCost
    return 0.0;
}

template <int NS>
__device__ __forceinline__ double kkt_rhs(int a, int N, const QpArgs& A, long long traj) {
    typedef Geo<NS> G;
    const Idx p = G::decode(a, N);
    if (p.kind == K_NU0) return A.b0[traj * G::M0 + p.comp];
    if (p.kind == K_NUF) return A.bf[traj * 6 + p.comp];
    if (p.kind == K_L) return A.defect[(traj * (N - 1) + p.node) * NS + p.comp];                // A_dyn z = defect (:337)
    if (p.kind == K_U) return -2.0 * node_weight(A.t + traj * N, p.node, N) * A.u_all[(traj * N + p.node) * 3 + p.comp];   // -gradient of quadCost
    return 0.0;
}

// Outputs of the dual instantiation (nstate 6): the multipliers of the defect rows and the node costates they map to.
struct DualArgs {
    const int32_t* seg_status;                // K1's status per segment, n_traj x (n_nodes-1)
    double *mult, *XC, *du_max;               // 6 x (n_nodes-1), 12 x n_nodes, 1 per trajectory
    double kappa;                             // default_mass / kthr: u in N = kappa x the nondimensional acceleration
};

// K7's body.  DUAL = false: the primal step (x_update, u_update) of lto_direct_qp.  DUAL = true (NS = 6): the back substitution keeps
// the K_L unknowns -- the multipliers lambda_i of segment i's defect -- instead, and an epilogue maps them to node costates.
template <int NS, bool DUAL>
__device__ __forceinline__ void qp_body(QpArgs A, DualArgs D) {
    typedef Geo<NS> G;
    constexpr int BW = G::BW;
    extern __shared__ __align__(16) double smem_d[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // wid < WARPS, so | is +.  Written as | because that is what the compiler made of + when this was the kernel's own body (it knew
    // the launch bound there): k_direct_qp<NS> keeps the instructions it had.
    const long long traj = ((long long)blockIdx.x * WARPS) | wid;
    if (traj >= A.n_traj) return;
    const int N = A.n_nodes, TOT = G::total(N);
    double* W = smem_d + (size_t)wid * SM_PER_WARP;          // W[(row & 31) * 64 + (col & 63)]
    double* rw = W + WR * WC;                                // right-hand side of the window rows
    double* xs = rw + WR;                                    // solution window (back substitution)
    const double* jac = A.jac + traj * (long long)(N - 1) * NS * 2 * (NS + 3);
    const double* tt = A.t + traj * N;
    double* U = A.work + traj * (long long)TOT * UROW;
    const unsigned full = 0xffffffffu;

    auto load_row = [&](int R) {
        if (R >= TOT) return;
        double* row = W + (R & (WR - 1)) * WC;
        // the row's life spans columns R-BW .. R+2BW (fill-in included): clear them, then generate the band entries
        for (int k = lane; k <= 3 * BW; k += 32) row[(R - BW + k) & (WC - 1)] = 0.0;
        __syncwarp();
        for (int k = lane; k <= 2 * BW; k += 32) {
            const int C = R - BW + k;
            if (C >= 0 && C < TOT) row[C & (WC - 1)] = kkt_entry<NS>(R, C, N, jac, tt);
        }
        if (lane == 0) rw[R & (WR - 1)] = kkt_rhs<NS>(R, N, A, traj);
    };

    for (int R = 0; R <= BW; ++R) load_row(R);
    __syncwarp();
    bool singular = false;
    // ---------------- elimination with partial pivoting inside the band
#pragma unroll 1
    for (int j = 0; j < TOT; ++j) {
        // pivot search over rows j .. j+BW of column j
        double v = 0.0;
        if (lane <= BW && j + lane < TOT) v = fabs(W[((j + lane) & (WR - 1)) * WC + (j & (WC - 1))]);
        int pi = lane;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(full, v, o);
            const int oi = __shfl_xor_sync(full, pi, o);
            if (ov > v || (ov == v && oi < pi)) { v = ov; pi = oi; }
        }
        const int p = j + pi;
        if (!(v > 0.0)) singular = true;
        double* rj = W + (j & (WR - 1)) * WC;
        if (p != j) {                                        // row interchange over the window's columns j .. j+2BW
            double* rp = W + (p & (WR - 1)) * WC;
            for (int k = lane; k <= 2 * BW; k += 32) {
                const int c = (j + k) & (WC - 1);
                const double a = rj[c]; rj[c] = rp[c]; rp[c] = a;
            }
            if (lane == 0) { const double a = rw[j & (WR - 1)]; rw[j & (WR - 1)] = rw[p & (WR - 1)]; rw[p & (WR - 1)] = a; }
        }
        __syncwarp();
        const double piv = rj[j & (WC - 1)];
        const double prow = rj[(j + 1 + lane) & (WC - 1)];  // columns j+1 .. j+32 (beyond j+2BW: zeros / cleared slots)
        const double prhs = rw[j & (WR - 1)];
        // the finished pivot row, for the back substitution
        U[(long long)j * UROW + 1 + lane] = (lane < 2 * BW && j + 1 + lane < TOT) ? prow : 0.0;
        if (lane == 0) { U[(long long)j * UROW] = piv; U[(long long)j * UROW + 33] = prhs; }
        const double ip = 1.0 / piv;
#pragma unroll 1
        for (int r = 1; r <= BW; ++r) {
            if (j + r >= TOT) break;
            double* rr = W + ((j + r) & (WR - 1)) * WC;
            const double f = rr[j & (WC - 1)] * ip;
            if (f != 0.0) {
                if (lane < 2 * BW) rr[(j + 1 + lane) & (WC - 1)] = fma(-f, prow, rr[(j + 1 + lane) & (WC - 1)]);
                if (lane == 0) rw[(j + r) & (WR - 1)] = fma(-f, prhs, rw[(j + r) & (WR - 1)]);
            }
        }
        __syncwarp();
        load_row(j + BW + 1);                                // the next row enters the window
        __syncwarp();
    }
    __threadfence_block();
    // ---------------- back substitution
    for (int k = lane; k < WC; k += 32) xs[k] = 0.0;
    __syncwarp();
    double un = U[(long long)(TOT - 1) * UROW + 1 + lane], pn = U[(long long)(TOT - 1) * UROW], rn = U[(long long)(TOT - 1) * UROW + 33];
    bool bad = singular;
    double du = 0.0;                                         // DUAL: max |du| (N)
#pragma unroll 1
    for (int j = TOT - 1; j >= 0; --j) {
        const double u = un, piv = pn, rhs = rn;
        if (j > 0) { un = U[(long long)(j - 1) * UROW + 1 + lane]; pn = U[(long long)(j - 1) * UROW]; rn = U[(long long)(j - 1) * UROW + 33]; }
        double s = (j + 1 + lane < TOT) ? u * xs[(j + 1 + lane) & (WC - 1)] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(full, s, o);
        const double x = (rhs - s) / piv;
        bad |= !(fabs(x) <= 1.79e308);
        __syncwarp();
        if (lane == 0) {
            xs[j & (WC - 1)] = x;
            const Idx d = G::decode(j, N);
            if (!DUAL) {
                if (d.kind == K_X) A.x_update[(traj * N + d.node) * NS + d.comp] = x;          // X_jump (:391)
                else if (d.kind == K_U) A.u_update[(traj * N + d.node) * 3 + d.comp] = x;      // u_jump (:392)
            } else {
                if (d.kind == K_L) D.mult[(traj * (N - 1) + d.node) * NS + d.comp] = x;
                else if (d.kind == K_U) { const double a = fabs(x); if (!(a <= du)) du = a; }   // NaN sticks
            }
        }
        __syncwarp();
    }
    if (!DUAL) {
        if (A.status && lane == 0) A.status[traj] = bad ? LTO_ST_NAN : 0;
        return;
    }
    // ---------------- dual epilogue: status, then the costates of every node from the multipliers lane 0 stored
    int worst = bad ? LTO_ST_NAN : LTO_OK;
    for (int k = lane; k < N - 1; k += 32) worst = max(worst, (int)D.seg_status[traj * (N - 1) + k]);
    worst = __reduce_max_sync(full, worst);
    if (lane == 0) { A.status[traj] = worst; D.du_max[traj] = du; }
    __threadfence_block();
    __syncwarp();
    const double* lam = D.mult + traj * (long long)(N - 1) * NS;
    for (int k = lane; k < N * NS; k += 32) {
        const int i = k / NS, c = k - i * NS;
        // p_i = Jx(i, i)^T lambda_i (forward leg); the last node: p = -Jx(N-2, N-1)^T lambda_{N-2} (backward leg)
        const int seg = i < N - 1 ? i : N - 2, col = i < N - 1 ? c : NS + c;
        const double* Jc = jac + ((long long)seg * (2 * (NS + 3)) + col) * NS;
        const double* l = lam + (long long)seg * NS;
        double p = 0.0;
#pragma unroll
        for (int r = 0; r < NS; ++r) p = fma(Jc[r], l[r], p);
        if (i == N - 1) p = -p;
        double* xc = D.XC + (traj * N + i) * 12;
        xc[c] = A.X_all[(traj * N + i) * NS + c];
        xc[NS + c] = worst == LTO_OK ? -p / (D.kappa * D.kappa) : nan("");              // [lr; lv] = -p / kappa^2
    }
}

template <int NS>
__global__ void __launch_bounds__(32 * WARPS) k_direct_qp(QpArgs A) {
    qp_body<NS, false>(A, DualArgs());
}

__global__ void __launch_bounds__(32 * WARPS) k_direct_qp_dual(QpArgs A, DualArgs D) {
    qp_body<6, true>(A, D);
}

}  // namespace dqp

size_t direct_qp_workspace_bytes(long long n_traj, int n_nodes, int nstate) {
    const int tot = nstate == 7 ? dqp::Geo<7>::total(n_nodes) : dqp::Geo<6>::total(n_nodes);
    return (size_t)n_traj * (size_t)tot * dqp::UROW * sizeof(double);
}

cudaError_t launch_direct_qp(const double* jac, const double* defect, const double* X_all, const double* u_all, const double* t,
                             const double* b0, const double* bf, double* work, double* x_update, double* u_update, int32_t* status,
                             long long n_traj, int n_nodes, int nstate, cudaStream_t st) {
    if (n_traj <= 0 || n_nodes < 2 || (nstate != 6 && nstate != 7)) return cudaErrorInvalidValue;
    dqp::QpArgs A;
    A.jac = jac; A.defect = defect; A.X_all = X_all; A.u_all = u_all; A.t = t; A.b0 = b0; A.bf = bf;
    A.work = work; A.x_update = x_update; A.u_update = u_update; A.status = status; A.n_traj = n_traj; A.n_nodes = n_nodes;
    const long long blocks = (n_traj + dqp::WARPS - 1) / dqp::WARPS;
    if (blocks > 0x7fffffffll) return cudaErrorInvalidValue;
    const size_t smem = (size_t)dqp::WARPS * dqp::SM_PER_WARP * sizeof(double);
    cudaError_t e;
    if (nstate == 6) {
        e = cudaFuncSetAttribute(dqp::k_direct_qp<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); if (e != cudaSuccess) return e;
        dqp::k_direct_qp<6><<<(int)blocks, 32 * dqp::WARPS, smem, st>>>(A);
    } else {
        e = cudaFuncSetAttribute(dqp::k_direct_qp<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); if (e != cudaSuccess) return e;
        dqp::k_direct_qp<7><<<(int)blocks, 32 * dqp::WARPS, smem, st>>>(A);
    }
    return cudaGetLastError();
}

cudaError_t launch_direct_qp_dual(const double* jac, const double* defect, const double* X_all, const double* u_all, const double* t,
                                  const double* b0, const double* bf, const int32_t* seg_status, double kappa, double* work, double* mult,
                                  double* XC, double* du_max, int32_t* status, long long n_traj, int n_nodes, cudaStream_t st) {
    if (n_traj <= 0 || n_nodes < 2) return cudaErrorInvalidValue;
    dqp::QpArgs A;
    A.jac = jac; A.defect = defect; A.X_all = X_all; A.u_all = u_all; A.t = t; A.b0 = b0; A.bf = bf;
    A.work = work; A.x_update = nullptr; A.u_update = nullptr; A.status = status; A.n_traj = n_traj; A.n_nodes = n_nodes;
    dqp::DualArgs D;
    D.seg_status = seg_status; D.mult = mult; D.XC = XC; D.du_max = du_max; D.kappa = kappa;
    const long long blocks = (n_traj + dqp::WARPS - 1) / dqp::WARPS;
    if (blocks > 0x7fffffffll) return cudaErrorInvalidValue;
    const size_t smem = (size_t)dqp::WARPS * dqp::SM_PER_WARP * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(dqp::k_direct_qp_dual, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dqp::k_direct_qp_dual<<<(int)blocks, 32 * dqp::WARPS, smem, st>>>(A, D);
    return cudaGetLastError();
}

}  // namespace lto
