// lto_solve.cu -- C ABI of the device-side Newton update and of the batched indirect solver
// (SURVEY section 8(f) rows 1-2; include/lto_b200.h).
//
//   lto_indirect_newton[_dev]   optimizeTraj_OLS's  xc_update = -sparse(Jac_full) \ defect_vec
//                               (src/multiShoot_CRTBP_indirect.jl:149-183) for n_traj trajectories, straight from the
//                               Phi_i blocks and defects the propagation kernels leave in HBM (lto_newton.cu)
//   lto_indirect_solve_batch    the whole iteration loop of multiShoot_CRTBP_indirect (:254-345) for n_traj independent
//                               trajectories at once, every array resident on the device: STM pass, Newton update, second
//                               order correction (:187-214), 20-point line search (:221-246), end-state pins (:324-325),
//                               defect check (:328-336).  Per iteration the host reads back ONE integer (how many
//                               trajectories are still iterating).
//   The *_nd forms take the system dimension (12: the reference's system; 14: with mass, see lto_b200.h); the others are ndim = 12.
//   lto_indirect_reduce_fuel_batch   reduceFuel_indirect's rho continuation (HelperFunctions.jl:105-193) for n_traj ladders: the
//                               same iteration engine, with the ladder state machine (lto_ladder.h) run on the device when a call ends.
// Built on the public device-pointer entry points (lto_indirect_dev, lto_sumsq_dev) and a few row-wise helper kernels.
#include "lto_internal.h"
#include "lto_handle.h"
#include "lto_ladder.h"
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

namespace lto {
size_t indirect_newton_workspace_bytes(long long n_traj, int n_nodes, int ndim);
cudaError_t launch_indirect_newton(const double* phi, const double* defect, double* work, double* update, int32_t* status,
                                   long long n_traj, int n_nodes, int ndim, bool adjoints_only, cudaStream_t st);
cudaError_t launch_indirect_newton_resolve(const double* defect, double* work, double* update, int32_t* status, long long n_traj, int n_nodes,
                                           int ndim, bool adjoints_only, cudaStream_t st);

size_t direct_qp_workspace_bytes(long long n_traj, int n_nodes, int nstate);
cudaError_t launch_direct_qp(const double* jac, const double* defect, const double* X_all, const double* u_all, const double* t,
                             const double* b0, const double* bf, double* work, double* x_update, double* u_update, int32_t* status,
                             long long n_traj, int n_nodes, int nstate, cudaStream_t st);

namespace slv {

constexpr int NA = 20;      // line-search points: alpha_all = LinRange(0.1, 1, 20)  (multiShoot_CRTBP_indirect.jl:227)

// out[r] = max_i |v[r*len + i]|  (NaN propagates: norm(defect[:], Inf) of :332 is NaN when any entry is)
__global__ void __launch_bounds__(256) k_rowmaxabs(const double* __restrict__ v, long long n_rows, long long len, double* __restrict__ out) {
    const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n_rows) return;
    const double* p = v + row * len;
    double m = 0.0; bool bad = false;
    for (long long i = lane; i < len; i += 32) { const double x = fabs(p[i]); bad |= !(x == x); m = fmax(m, x); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) out[row] = bad ? nan("") : m;
}

// out[a][j][e] = x[j][e] + scale[a*n_rows + j] * u[j][e]   (a = blockIdx.y; in-place on x or u allowed when gridDim.y == 1)
__global__ void __launch_bounds__(256) k_axpy_rows(const double* x, const double* u, const double* __restrict__ scale, double* out,
                                                   long long n_rows, long long len) {
    const long long total = n_rows * len;
    const long long a = blockIdx.y;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long j = i / len;
        const double s = scale[a * n_rows + j];
        out[a * total + i] = (s == 0.0) ? x[i] : fma(s, u[i], x[i]);   // a masked row is copied exactly (its update may hold NaN)
    }
}

// second-order-correction mask (:190): active && norm(xc_update, Inf) < 1e-1
__global__ void k_soc_mask(const double* __restrict__ umax, const int* __restrict__ active, double* __restrict__ mask, long long n) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) mask[j] = (active[j] && umax[j] < 1e-1) ? 1.0 : 0.0;
}

// line search (:243-245): alpha = alpha_all[er .== minimum(er)][1] of row j, whose trials are ers[a*n + j]
__device__ __forceinline__ double best_alpha(const double* __restrict__ ers, const double* __restrict__ alpha_all, long long n, long long j,
                                             int n_alpha) {
    // minimum() propagates NaN in Julia, and then no entry compares equal: the reference would throw.  Here a NaN merit
    // value never wins; if all are NaN the full step is taken and the NaN surfaces in the defect check.
    double best = INFINITY; int ib = -1;
    for (int a = 0; a < n_alpha; ++a) { const double e = ers[(long long)a * n + j]; if (e < best) { best = e; ib = a; } }
    return ib >= 0 ? alpha_all[ib] : 1.0;
}
// scale = alpha for iterating trajectories, 0 otherwise
__global__ void k_pick_alpha(const double* __restrict__ ers, const double* __restrict__ alpha_all, const int* __restrict__ active,
                             double* __restrict__ alpha, double* __restrict__ scale, long long n, int use_ls, int n_alpha = NA) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double al = use_ls ? best_alpha(ers, alpha_all, n, j, n_alpha) : 1.0;
    alpha[j] = al;
    scale[j] = active[j] ? al : 0.0;
}
// the same for the nsel work-set rows idx[k] of a gathered line search (ers[a*nsel + k])
__global__ void k_pick_alpha_sel(const double* __restrict__ ers, const double* __restrict__ alpha_all, const int* __restrict__ idx,
                                 double* __restrict__ scale, long long nsel) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nsel) scale[idx[k]] = best_alpha(ers, alpha_all, nsel, k, NA);
}

// Rows of the work set a gathered pass takes: those at their nominal pass (wit < 0), or those due a line search (wit >= 3, :300).
__global__ void k_select(const int* __restrict__ wit, int* __restrict__ sel, long long n, int line_search) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) sel[j] = line_search ? (wit[j] >= 3) : (wit[j] < 0);
}
// idx[k] = the k-th selected row (pos: exclusive prefix sum of sel)
__global__ void k_index_of(const int* __restrict__ sel, const int* __restrict__ pos, int* __restrict__ idx, long long n) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && sel[j]) idx[pos[j]] = (int)j;
}
// dst[a][k][e] = src[idx[k]][e] for a < reps
__global__ void __launch_bounds__(256) k_gather_rows(const double* __restrict__ src, const int* __restrict__ idx, double* __restrict__ dst,
                                                     long long nsel, long long len, int reps) {
    const long long total = nsel * len;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total * reps; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i % total, k = r / len;
        dst[i] = src[(long long)idx[k] * len + (r - k * len)];
    }
}
// dst[idx[k]][e] = src[k][e]
__global__ void __launch_bounds__(256) k_scatter_rows(const double* __restrict__ src, const int* __restrict__ idx, double* __restrict__ dst,
                                                      long long nsel, long long len) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nsel * len; i += (long long)gridDim.x * blockDim.x) {
        const long long k = i / len;
        dst[(long long)idx[k] * len + (i - k * len)] = src[i];
    }
}
// line-search trials of the selected rows: out[a][k][e] = x[idx[k]][e] + alpha_all[a] * u[idx[k]][e]  (k_axpy_rows's arithmetic)
__global__ void __launch_bounds__(256) k_ls_trials(const double* __restrict__ x, const double* __restrict__ u, const int* __restrict__ idx,
                                                   const double* __restrict__ alpha_all, double* __restrict__ out, long long nsel, long long len) {
    const long long total = nsel * len;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total * NA; i += (long long)gridDim.x * blockDim.x) {
        const long long a = i / total, r = i - a * total, k = r / len;
        const long long s = (long long)idx[k] * len + (r - k * len);
        out[i] = fma(alpha_all[a], u[s], x[s]);
    }
}

// End of a solver call's step for the rows of the indirect engine's work set, each with its own iteration counter wit[j]
// (-1: the call has just started and waits for its nominal pass).  phase 0: after the nominal pass (:274) of the rows with
// wit < 0 (the others only count); phase 1: after a Newton iteration of every row.  Same rules as k_iter_end:
// er = norm(defect[:], Inf); abort above 1e3 (:333-336); maxIter (:282-286); loop condition er > 1e-10; NaN -> flag 2.
// count[0]: rows still iterating; count[1]: of these, the ones whose next iteration runs the line search (iterCount > 3).
__global__ void k_call_end(const double* __restrict__ er, int* __restrict__ active, const int* __restrict__ orig, int* __restrict__ wit,
                           int* __restrict__ iters, int* __restrict__ flag, double* __restrict__ er_full, unsigned long long* __restrict__ count,
                           long long n, int phase, int max_iter) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int c = wit[j];
    bool go = true;
    if (phase == 1 || c < 0) {
        c = phase == 0 ? 0 : c + 1;
        wit[j] = c;
        const int o = orig[j];
        const double e = er[j];
        er_full[o] = e;
        if (c > 0) iters[o] = c;
        go = e > 1e-10;                                   // NaN -> false: the reference's while-condition ends the loop as well
        if (!(e == e)) flag[o] = 2;
        if (go && !(e <= 1e3)) { go = false; flag[o] = 1; }
        if (go && c >= max_iter) { go = false; flag[o] = 1; }
        active[j] = go ? 1 : 0;
    }
    if (go) { atomicAdd(&count[0], 1ull); if (c >= 3) atomicAdd(&count[1], 1ull); }
}

// The continuation ladder's hook (lto_ladder.h), one warp per work-set row whose solver call just ended (active[j] == 0).  The
// call's status is that of lto_indirect_solve_batch (k_call_end's flag, 2 when a node is non-finite, as k_retire_rows reports it).
// A ladder that goes on accepts XC_new as its start or resets the row to the accepted start (acc), sets the call's rho and
// re-enters the work set at its nominal pass (count[0], count[2]); a ladder that ends writes its row to the caller-ordered outputs.
__global__ void __launch_bounds__(256) k_ladder_hook(double* __restrict__ XC, const double* __restrict__ Def, double* __restrict__ RH,
                                                     int* __restrict__ active, const int* __restrict__ orig, int* __restrict__ wit,
                                                     int* __restrict__ iters, int* __restrict__ flag, LadderState* __restrict__ ladder,
                                                     const double* __restrict__ draws, double* __restrict__ acc, double* __restrict__ XCout,
                                                     double* __restrict__ DefOut, int* __restrict__ status, int* __restrict__ calls,
                                                     int* __restrict__ newton_iters, double* __restrict__ rho_last, unsigned long long* __restrict__ count, long long n,
                                                     long long LX, long long LD) {
    const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (j >= n || active[j]) return;
    const long long o = orig[j];
    double* x = XC + j * LX;
    bool bad = false;
    for (long long i = lane; i < LX; i += 32) bad |= !(fabs(x[i]) <= 1.7976931348623157e308);
    bad = __any_sync(0xffffffffu, bad);
    int go = 0, take = 0;
    if (lane == 0) {
        const int st = bad ? 2 : flag[o];
        newton_iters[o] += iters[o];
        LadderState s = ladder[o];
        int fin = 0;
        go = ladder_step(&s, st, draws + o * LADDER_DRAWS, &take, &fin);
        ladder[o] = s;
        if (go) {
            RH[j] = s.rho; wit[j] = -1; active[j] = 1; flag[o] = 0; iters[o] = 0; calls[o] += 1;
            atomicAdd(&count[0], 1ull); atomicAdd(&count[2], 1ull);
        } else {
            status[o] = fin; rho_last[o] = s.rho;
        }
    }
    go = __shfl_sync(0xffffffffu, go, 0);
    take = __shfl_sync(0xffffffffu, take, 0);
    double* a = acc + o * LX;
    if (go) {
        if (take) { for (long long i = lane; i < LX; i += 32) a[i] = x[i]; }
        else      { for (long long i = lane; i < LX; i += 32) x[i] = a[i]; }
    } else {
        for (long long i = lane; i < LX; i += 32) XCout[o * LX + i] = x[i];
        for (long long i = lane; i < LD; i += 32) DefOut[o * LD + i] = Def[j * LD + i];
    }
}

// RH: rho_current on entry, the rho of the first call on return
__global__ void k_ladder_init(double* __restrict__ RH, const double* __restrict__ rho_target, LadderState* __restrict__ ladder,
                              int* __restrict__ calls, int* __restrict__ newton_iters, long long n) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    LadderState s;
    RH[j] = ladder_init(&s, RH[j], rho_target[j]);
    ladder[j] = s; calls[j] = 1; newton_iters[j] = 0;
}

// tile the per-trajectory parameter arrays for the NA trial copies
__global__ void k_tile(const double* __restrict__ src, double* __restrict__ dst, long long n, int reps) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n * reps) dst[i] = src[i % n];
}

// end of an iteration (:328-341): er = norm(defect[:], Inf); iterCount += 1; abort above 1e3; loop condition er > 1e-10.
// Rows are the WORK SET (trajectories still iterating); orig[row] is the trajectory's index in the caller's arrays.
//   flag: 0 converged / still iterating, 1 gave up (maxIter or abort), 2 the defects went NaN (the reference's evident intent at
//   :339-341; its own test looks at XC_all[1,1] only, a pinned entry that can never be NaN -- a latent bug that is NOT mirrored:
//   a NaN trajectory must not come back as "converged", the continuation driver would walk on from it)
__global__ void k_iter_end(const double* __restrict__ er, int* __restrict__ active, const int* __restrict__ orig, int* __restrict__ iters,
                           int* __restrict__ flag, double* __restrict__ er_full, unsigned long long* __restrict__ n_active, long long n, int it,
                           int max_iter, double tol = 1e-10, double abort_above = 1e3, int force_first = 0) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int o = orig[j];
    const double e = er[j];
    er_full[o] = e;
    if (it > 0) iters[o] = it;
    bool go = e > tol || (force_first && it == 0);        // NaN -> false: the reference's while-condition ends the loop as well
    if (!(e == e)) flag[o] = 2;
    if (go && !(e <= abort_above) && !(force_first && it == 0)) { go = false; flag[o] = 1; }   // "Not likely to converge. Aborting." (:333-336)
    if (go && it >= max_iter) { go = false; flag[o] = 1; }   // "Reached max iteration count" (:282-286)
    active[j] = go ? 1 : 0;
    if (go) atomicAdd(n_active, 1ull);
}

// exclusive prefix sum of the active flags (one block; the work set is at most a few 10^5 rows)
__global__ void __launch_bounds__(1024) k_scan_active(const int* __restrict__ active, int* __restrict__ pos, long long n) {
    __shared__ int part[1024];
    const long long per = (n + 1023) / 1024, lo = threadIdx.x * per, hi = lo + per < n ? lo + per : n;
    int c = 0;
    for (long long i = lo; i < hi; ++i) c += active[i] ? 1 : 0;
    part[threadIdx.x] = c;
    __syncthreads();
    if (threadIdx.x == 0) { int acc = 0; for (int i = 0; i < 1024; ++i) { const int v = part[i]; part[i] = acc; acc += v; } }
    __syncthreads();
    int run = part[threadIdx.x];
    for (long long i = lo; i < hi; ++i) { pos[i] = run; run += active[i] ? 1 : 0; }
}

// rows that stopped iterating leave the work set: their rows go to the caller-ordered result arrays
// (flag != NULL: a retired row with a non-finite entry is reported as status_flag 2 -- the "over the whole trajectory" form of :339-341)
__global__ void __launch_bounds__(256) k_retire_rows(const double* __restrict__ src, double* __restrict__ dst_full, const int* __restrict__ orig,
                                                     const int* __restrict__ active, long long n_rows, long long len, int* __restrict__ flag = nullptr) {
    const long long total = n_rows * len;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long j = i / len;
        if (!active[j]) {
            const double v = src[i];
            dst_full[(long long)orig[j] * len + (i - j * len)] = v;
            if (flag && !(fabs(v) <= 1.7976931348623157e308)) flag[orig[j]] = 2;
        }
    }
}
// the rows still iterating move to the front (into `dst`, same order)
template <class V>
__global__ void __launch_bounds__(256) k_compact_rows(const V* __restrict__ src, V* __restrict__ dst, const int* __restrict__ pos,
                                                      const int* __restrict__ active, long long n_rows, long long len) {
    const long long total = n_rows * len;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long j = i / len;
        if (active[j]) dst[(long long)pos[j] * len + (i - j * len)] = src[i];
    }
}
// line-search scale table scale[a*n + j] = alpha_a, and initial bookkeeping
__global__ void k_fill_ls(const double* __restrict__ alpha_all, double* __restrict__ table, long long n, int n_alpha = NA) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n * n_alpha) table[i] = alpha_all[i / n];
}
// right-hand sides of the direct solver's end constraints (multiShoot_CRTBP_direct.jl:374-375, :270; dV = 0):
//   b0 = state_0 - X_all[1:6, 1] (, mass - X_all[7, 1]),  bf = state_f - X_all[1:6, end]
__global__ void k_direct_ends(const double* __restrict__ X, const double* __restrict__ s0, const double* __restrict__ sf, const int* __restrict__ orig,
                              double mass, double* __restrict__ b0, double* __restrict__ bf, long long n, int N, int ns) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int m0 = 6 + (ns == 7 ? 1 : 0);
    const long long o = orig[j];
    for (int k = 0; k < 6; ++k) {
        b0[j * m0 + k] = s0[o * 6 + k] - X[(j * N) * ns + k];
        bf[j * 6 + k] = sf[o * 6 + k] - X[(j * N + N - 1) * ns + k];
    }
    if (ns == 7) b0[j * m0 + 6] = mass - X[(j * N) * ns + 6];
}
__global__ void k_set_int(int* __restrict__ v, int value, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = value;
}
__global__ void k_iota(int* __restrict__ orig, int* __restrict__ active, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { orig[i] = (int)i; active[i] = 1; }
}

static inline unsigned nblk(long long n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace slv
}  // namespace lto

using namespace lto;

// ---- the iteration engine of the batched indirect solver (multiShoot_CRTBP_indirect :254-345, p as given) ----
// The work set holds the trajectories whose solver call is running, compacted to the front after every step; every row has
// its own iteration counter wit[j] (-1: the call has just started and waits for its nominal pass).  When a row's call ends,
// `hook` decides what becomes of it: lto_indirect_solve_batch_nd retires it into the caller-ordered outputs; the continuation
// ladder either retires it or starts its next call in place (it then re-enters at its nominal pass, in the same step).
// Per step the host reads back one set of counts.
struct EngineArrays {
    double *XC, *Def, *RH, *XCout, *DefOut, *ErOut;
    int *active, *orig, *wit, *iters, *flag;
    unsigned long long* count;         // [0] rows iterating, [1] of them due a line search, [2] rows the hook restarted
};

template <class Setup, class Hook>
static int indirect_engine(lto_handle* h, const lto_indirect_params* p, int ND, long long T, int N, int max_iter, int flag_adjointsOnly,
                           const double* XC_all, const double* t_TU, const double* thrustLimit_traj, const double* rho_traj,
                           size_t extra_bytes, EngineArrays* w, Setup&& setup, Hook&& hook) {
    const int NA = slv::NA;
    const long long ns = T * (N - 1), nn = T * N;
    const long long LX = (long long)N * ND, LD = (long long)(N - 1) * ND;      // row lengths: states / defects of one trajectory
    cudaStream_t st = h->s_compute;
    // ---- device arrays.  "work" arrays hold the trajectories still iterating (compacted to the front after every step);
    // "out" arrays are in the caller's order and receive a trajectory's rows when it stops.
    const size_t bXC = al(nn * ND * 8), bT = al(nn * 8), bPar = al(T * 8), bDef = al(ns * ND * 8), bPhi = al(ns * ND * ND * 8);
    const size_t bTrX = al((size_t)NA * nn * ND * 8), bTrD = al((size_t)NA * ns * ND * 8), bTrT = al((size_t)NA * nn * 8), bTrP = al((size_t)NA * T * 8);
    const size_t bVec = al((size_t)NA * T * 8), bInt = al(T * 4);
    size_t need = bXC * 4 + bT + bPar * 2 + bDef * 3 + bPhi + bTrX + bTrD + bTrT + bTrP * 2 + bVec * 8 + bInt * 9 + al(NA * 8) + 256 + al(extra_bytes);
    int rc = ensure(h, &h->d_slv, &h->d_slv_cap, need); if (rc) return rc;
    char* q = (char*)h->d_slv;
    auto take = [&](size_t b) { char* r = q; q += b; return r; };
    double* dXC = (double*)take(bXC); double* dXS = (double*)take(bXC); double* dUp = (double*)take(bXC); double* dUp2 = dXS;   // the SOC state buffer is free again when the SOC update is computed
    double* dXCout = (double*)take(bXC);
    double* dT = (double*)take(bT);
    double* dTL = thrustLimit_traj ? (double*)take(bPar) : nullptr; double* dRH = rho_traj ? (double*)take(bPar) : nullptr;
    double* dDef = (double*)take(bDef); double* dDs = (double*)take(bDef); double* dDefOut = (double*)take(bDef); double* dPhi = (double*)take(bPhi);
    double* dTrX = (double*)take(bTrX); double* dTrD = (double*)take(bTrD); double* dTrT = (double*)take(bTrT);
    double* dTrTL = thrustLimit_traj ? (double*)take(bTrP) : nullptr; double* dTrRH = rho_traj ? (double*)take(bTrP) : nullptr;
    double* dEr = (double*)take(bVec); double* dUmax = (double*)take(bVec); double* dMask = (double*)take(bVec);
    double* dErs = (double*)take(bVec); double* dAlpha = (double*)take(bVec); double* dScale = (double*)take(bVec);
    double* dLsTable = (double*)take(bVec); double* dErOut = (double*)take(bVec);
    int* dActive = (int*)take(bInt); int* dIters = (int*)take(bInt); int* dFlag = (int*)take(bInt);
    int* dOrig = (int*)take(bInt); int* dOrig2 = (int*)take(bInt); int* dPos = (int*)take(bInt);
    int* dWit = (int*)take(bInt); int* dSel = (int*)take(bInt); int* dIdx = (int*)take(bInt);
    double* dAlphaAll = (double*)take(al(NA * 8));
    unsigned long long* dCount = (unsigned long long*)take(256);
    char* dExtra = take(al(extra_bytes));
    *w = EngineArrays{dXC, dDef, dRH, dXCout, dDefOut, dErOut, dActive, dOrig, dWit, dIters, dFlag, dCount};
    // ---- inputs
    CK(h, cudaMemcpyAsync(dXC, XC_all, nn * ND * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dT, t_TU, nn * 8, cudaMemcpyHostToDevice, st));
    if (dTL) CK(h, cudaMemcpyAsync(dTL, thrustLimit_traj, T * 8, cudaMemcpyHostToDevice, st));
    if (dRH) CK(h, cudaMemcpyAsync(dRH, rho_traj, T * 8, cudaMemcpyHostToDevice, st));
    double alpha_all[slv::NA];
    for (int a = 0; a < NA; ++a) alpha_all[a] = 0.1 + (double)a * ((1.0 - 0.1) / (double)(NA - 1));      // LinRange(0.1, 1, 20)
    alpha_all[NA - 1] = 1.0;
    CK(h, cudaMemcpyAsync(dAlphaAll, alpha_all, NA * 8, cudaMemcpyHostToDevice, st));
    rc = setup(dExtra); if (rc) return rc;
    CK(h, cudaStreamSynchronize(st));                                     // alpha_all is a stack array
    CK(h, cudaMemsetAsync(dIters, 0, T * 4, st));
    CK(h, cudaMemsetAsync(dFlag, 0, T * 4, st));
    slv::k_iota<<<slv::nblk(T, 256), 256, 0, st>>>(dOrig, dActive, T);
    slv::k_set_int<<<slv::nblk(T, 256), 256, 0, st>>>(dWit, -1, T);                           // every call starts at its nominal pass
    h->launches += 2;
    CK(h, cudaEventRecord(h->ev_t0, st));

    long long nc = T;                                                     // size of the work set
    auto defect_pass = [&](const double* X, const double* T_, const double* tl, const double* rh, long long ntr, double* D) -> int {
        return lto_indirect_dev(h, p, ntr * (N - 1), N, ND, X, T_, nullptr, nullptr, tl, rh, D, nullptr, nullptr, nullptr);
    };
    auto rowmax = [&](const double* v, long long rows, long long len, double* out) {
        slv::k_rowmaxabs<<<slv::nblk(rows * 32, 256), 256, 0, st>>>(v, rows, len, out); h->launches += 1;
    };
    auto axpy = [&](const double* x, const double* u, const double* scale, double* out, long long rows, long long len, int reps) {
        dim3 g(std::min<unsigned>(slv::nblk(rows * len, 256), 148u * 16u), (unsigned)reps);
        slv::k_axpy_rows<<<g, 256, 0, st>>>(x, u, scale, out, rows, len); h->launches += 1;
    };
    auto grid_for = [&](long long n) { return std::min<unsigned>(slv::nblk(n, 256), 148u * 16u); };
    // idx[0..nsel) = the work-set rows at their nominal pass (line_search = 0) or due a line search (1)
    auto select = [&](int line_search) {
        slv::k_select<<<slv::nblk(nc, 256), 256, 0, st>>>(dWit, dSel, nc, line_search);
        slv::k_scan_active<<<1, 1024, 0, st>>>(dSel, dPos, nc);
        slv::k_index_of<<<slv::nblk(nc, 256), 256, 0, st>>>(dSel, dPos, dIdx, nc);
        h->launches += 3;
    };
    auto gather = [&](const double* src, double* dst, long long nsel, long long len, int reps) {
        slv::k_gather_rows<<<grid_for(nsel * len * reps), 256, 0, st>>>(src, dIdx, dst, nsel, len, reps); h->launches += 1;
    };
    auto scatter = [&](const double* src, double* dst, long long nsel, long long len) {
        slv::k_scatter_rows<<<grid_for(nsel * len), 256, 0, st>>>(src, dIdx, dst, nsel, len); h->launches += 1;
    };
    // end of a step: bookkeeping, the hook on the rows whose call ended, compaction of the rest.  Reads back the counts.
    unsigned long long cnt[3] = {0, 0, 0};
    auto step_end = [&](int phase) -> int {
        CK(h, cudaMemsetAsync(dCount, 0, 3 * 8, st));
        slv::k_call_end<<<slv::nblk(nc, 256), 256, 0, st>>>(dEr, dActive, dOrig, dWit, dIters, dFlag, dErOut, dCount, nc, phase, max_iter);
        h->launches += 1;
        int rc2 = hook(nc); if (rc2) return rc2;
        CK(h, cudaMemcpyAsync(cnt, dCount, 3 * 8, cudaMemcpyDeviceToHost, st));
        CK(h, cudaStreamSynchronize(st));
        const long long na = (long long)cnt[0];
        if (na > 0 && na < nc) {
            slv::k_scan_active<<<1, 1024, 0, st>>>(dActive, dPos, nc);
            // XC, defects (through free buffers), times, parameters, original indices, iteration counters
            slv::k_compact_rows<double><<<grid_for(nc * LX), 256, 0, st>>>(dXC, dXS, dPos, dActive, nc, LX);
            CK(h, cudaMemcpyAsync(dXC, dXS, (size_t)na * LX * 8, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<double><<<grid_for(nc * LD), 256, 0, st>>>(dDef, dDs, dPos, dActive, nc, LD);
            CK(h, cudaMemcpyAsync(dDef, dDs, (size_t)na * LD * 8, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<double><<<grid_for(nc * N), 256, 0, st>>>(dT, dUp, dPos, dActive, nc, N);
            CK(h, cudaMemcpyAsync(dT, dUp, (size_t)na * N * 8, cudaMemcpyDeviceToDevice, st));
            if (dTL) { slv::k_compact_rows<double><<<grid_for(nc), 256, 0, st>>>(dTL, dUmax, dPos, dActive, nc, 1); CK(h, cudaMemcpyAsync(dTL, dUmax, (size_t)na * 8, cudaMemcpyDeviceToDevice, st)); }
            if (dRH) { slv::k_compact_rows<double><<<grid_for(nc), 256, 0, st>>>(dRH, dUmax, dPos, dActive, nc, 1); CK(h, cudaMemcpyAsync(dRH, dUmax, (size_t)na * 8, cudaMemcpyDeviceToDevice, st)); }
            slv::k_compact_rows<int><<<grid_for(nc), 256, 0, st>>>(dOrig, dOrig2, dPos, dActive, nc, 1);
            CK(h, cudaMemcpyAsync(dOrig, dOrig2, (size_t)na * 4, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<int><<<grid_for(nc), 256, 0, st>>>(dWit, dOrig2, dPos, dActive, nc, 1);
            CK(h, cudaMemcpyAsync(dWit, dOrig2, (size_t)na * 4, cudaMemcpyDeviceToDevice, st));
            slv::k_set_int<<<slv::nblk(na, 256), 256, 0, st>>>(dActive, 1, na);      // the compacted work set: all iterating
            h->launches += 7 + (dTL ? 1 : 0) + (dRH ? 1 : 0);
        }
        nc = na;
        return 0;
    };

    long long n_fresh = nc;                                               // rows at the nominal pass of a new call
    for (;;) {
        // ---- nominal runs (:274) of the calls that start; a call that converges there ends after 0 iterations
        while (n_fresh > 0) {
            if (n_fresh == nc) {
                rc = defect_pass(dXC, dT, dTL, dRH, nc, dDef); if (rc) return rc;
                rowmax(dDef, nc, LD, dEr);
            } else {
                select(0);
                gather(dXC, dTrX, n_fresh, LX, 1); gather(dT, dTrT, n_fresh, N, 1);
                if (dTL) gather(dTL, dTrTL, n_fresh, 1, 1);
                if (dRH) gather(dRH, dTrRH, n_fresh, 1, 1);
                rc = defect_pass(dTrX, dTrT, dTrTL, dTrRH, n_fresh, dTrD); if (rc) return rc;
                rowmax(dTrD, n_fresh, LD, dErs);
                scatter(dTrD, dDef, n_fresh, LD); scatter(dErs, dEr, n_fresh, 1);
            }
            rc = step_end(0); if (rc) return rc;
            n_fresh = (long long)cnt[2];
        }
        if (nc == 0) break;
        const long long n_ls = (long long)cnt[1];
        // ---- one Newton iteration of every row of the work set
        // jacobianCalc (:290): one launch, Phi_i of every segment of every trajectory still iterating (and the defects, unchanged)
        rc = lto_indirect_dev(h, p, nc * (N - 1), N, ND, dXC, dT, nullptr, nullptr, dTL, dRH, dDef, nullptr, nullptr, dPhi); if (rc) return rc;
        // optimizeTraj_OLS (:149-183)
        rc = lto_indirect_newton_nd_dev(h, ND, nc, N, flag_adjointsOnly, dPhi, dDef, dUp, nullptr); if (rc) return rc;
        // second-order correction (:187-214), only where norm(xc_update, Inf) < 1e-1
        rowmax(dUp, nc, LX, dUmax);
        slv::k_soc_mask<<<slv::nblk(nc, 256), 256, 0, st>>>(dUmax, dActive, dMask, nc); h->launches += 1;
        axpy(dXC, dUp, dMask, dXS, nc, LX, 1);                                                 // XC_all_soc (:194)
        rc = defect_pass(dXS, dT, dTL, dRH, nc, dDs); if (rc) return rc;                       // :197
        rc = lto_indirect_newton_resolve_nd_dev(h, ND, nc, N, flag_adjointsOnly, dDs, dUp2, nullptr); if (rc) return rc;   // :207 (same Jacobian: stored reflections replayed)
        axpy(dUp, dUp2, dMask, dUp, nc, LX, 1);                                                // xc_update += xc_update_soc (:213)
        // line search (:298-302) for the rows whose iterCount > 3: all 20 x n trial trajectories in one launch
        if (n_ls == nc) {
            slv::k_fill_ls<<<slv::nblk(nc * NA, 256), 256, 0, st>>>(dAlphaAll, dLsTable, nc);
            slv::k_tile<<<slv::nblk((long long)NA * nc * N, 256), 256, 0, st>>>(dT, dTrT, nc * N, NA);
            if (dTL) slv::k_tile<<<slv::nblk((long long)NA * nc, 256), 256, 0, st>>>(dTL, dTrTL, nc, NA);
            if (dRH) slv::k_tile<<<slv::nblk((long long)NA * nc, 256), 256, 0, st>>>(dRH, dTrRH, nc, NA);
            h->launches += 2 + (dTL ? 1 : 0) + (dRH ? 1 : 0);
            axpy(dXC, dUp, dLsTable, dTrX, nc, LX, NA);                                        // XC_all + xc_update*alpha (:235)
        } else if (n_ls > 0) {                                                                 // only the rows due one, gathered
            select(1);
            slv::k_ls_trials<<<grid_for((long long)NA * n_ls * LX), 256, 0, st>>>(dXC, dUp, dIdx, dAlphaAll, dTrX, n_ls, LX); h->launches += 1;
            gather(dT, dTrT, n_ls, N, NA);
            if (dTL) gather(dTL, dTrTL, n_ls, 1, NA);
            if (dRH) gather(dRH, dTrRH, n_ls, 1, NA);
        }
        if (n_ls > 0) {
            rc = defect_pass(dTrX, dTrT, dTrTL, dTrRH, (long long)NA * n_ls, dTrD); if (rc) return rc;   // :238
            rc = lto_sumsq_dev(h, dTrD, (long long)NA * n_ls, LD, dErs); if (rc) return rc;    // er[ind] = sum(defect[:].^2) (:241)
        }
        slv::k_pick_alpha<<<slv::nblk(nc, 256), 256, 0, st>>>(dErs, dAlphaAll, dActive, dAlpha, dScale, nc, n_ls == nc); h->launches += 1;
        if (n_ls > 0 && n_ls < nc) { slv::k_pick_alpha_sel<<<slv::nblk(n_ls, 256), 256, 0, st>>>(dErs, dAlphaAll, dIdx, dScale, n_ls); h->launches += 1; }
        axpy(dXC, dUp, dScale, dXC, nc, LX, 1);                                                // XC_all = XC_all + xc_update*alpha (:304)
        // the end states cannot have moved (:324-325): their update entries are exact zeros (lto_newton.cu; 14-dim: the 7-element pins)
        rc = defect_pass(dXC, dT, dTL, dRH, nc, dDef); if (rc) return rc;                      // :328
        rowmax(dDef, nc, LD, dEr);                                                             // :332
        rc = step_end(1); if (rc) return rc;
        n_fresh = (long long)cnt[2];
    }
    CK(h, cudaEventRecord(h->ev_t1, st));
    return 0;
}

extern "C" {

static inline bool valid_ndim(int ndim) { return ndim == 12 || ndim == 14; }

int lto_indirect_newton_nd_dev(lto_handle* h, int ndim, int64_t n_traj, int n_nodes, int flag_adjointsOnly, const double* phi,
                               const double* defect, double* xc_update, int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) return fail(h, LTO_ERR_ARG, "device-pointer entry points need a single-device handle (lto_init)");
    if (!valid_ndim(ndim)) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (n_traj == 0) return LTO_SUCCESS;
    if (!phi || !defect || !xc_update) return fail(h, LTO_ERR_ARG, "null array argument");
    if (((uintptr_t)phi & 15u) != 0) return fail(h, LTO_ERR_ARG, "phi must be 16-byte aligned");
    CK(h, cudaSetDevice(h->device));
    h->nwt_traj = 0;
    int rc = ensure(h, &h->d_nwt, &h->d_nwt_cap, indirect_newton_workspace_bytes(n_traj, n_nodes, ndim)); if (rc) return rc;
    cudaError_t e = launch_indirect_newton(phi, defect, (double*)h->d_nwt, xc_update, status, n_traj, n_nodes, ndim, flag_adjointsOnly != 0,
                                           h->s_compute);
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "newton kernel launch: %s", cudaGetErrorString(e));
    h->launches += 1;
    h->nwt_traj = n_traj; h->nwt_nodes = n_nodes; h->nwt_adj = flag_adjointsOnly != 0; h->nwt_ndim = ndim;
    return LTO_SUCCESS;
}

int lto_indirect_newton_dev(lto_handle* h, int64_t n_traj, int n_nodes, int flag_adjointsOnly, const double* phi,
                            const double* defect, double* xc_update, int32_t* status) {
    return lto_indirect_newton_nd_dev(h, 12, n_traj, n_nodes, flag_adjointsOnly, phi, defect, xc_update, status);
}

int lto_indirect_newton_resolve_nd_dev(lto_handle* h, int ndim, int64_t n_traj, int n_nodes, int flag_adjointsOnly, const double* defect,
                                       double* xc_update, int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) return fail(h, LTO_ERR_ARG, "device-pointer entry points need a single-device handle (lto_init)");
    if (!valid_ndim(ndim)) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
    if (n_traj == 0) return LTO_SUCCESS;
    if (!defect || !xc_update) return fail(h, LTO_ERR_ARG, "null array argument");
    if (h->nwt_traj != n_traj || h->nwt_nodes != n_nodes || h->nwt_adj != (flag_adjointsOnly != 0) || h->nwt_ndim != ndim || !h->d_nwt)
        return fail(h, LTO_ERR_ARG, "lto_indirect_newton_resolve_dev: no factorisation of this shape, dimension and mode is held "
                                    "(call lto_indirect_newton_dev first)");
    if (((uintptr_t)defect & 15u) != 0) return fail(h, LTO_ERR_ARG, "defect must be 16-byte aligned");
    CK(h, cudaSetDevice(h->device));
    cudaError_t e = launch_indirect_newton_resolve(defect, (double*)h->d_nwt, xc_update, status, n_traj, n_nodes, ndim, flag_adjointsOnly != 0,
                                                   h->s_compute);
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "newton resolve kernel launch: %s", cudaGetErrorString(e));
    h->launches += 1;
    return LTO_SUCCESS;
}

int lto_indirect_newton_resolve_dev(lto_handle* h, int64_t n_traj, int n_nodes, int flag_adjointsOnly, const double* defect,
                                    double* xc_update, int32_t* status) {
    return lto_indirect_newton_resolve_nd_dev(h, 12, n_traj, n_nodes, flag_adjointsOnly, defect, xc_update, status);
}

int lto_indirect_newton_nd(lto_handle* h, int ndim, int64_t n_traj, int n_nodes, int flag_adjointsOnly, const double* phi,
                           const double* defect, double* xc_update, int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (!valid_ndim(ndim)) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (n_traj == 0) return LTO_SUCCESS;
    if (!phi || !defect || !xc_update) return fail(h, LTO_ERR_ARG, "null array argument");
    const long long ND = ndim;
    if (h->n_child > 0) {
        const long long N = n_nodes;
        return split_trajectories(h, n_traj, [&](lto_handle* c, long long u0, long long nu) {
            return lto_indirect_newton_nd(c, ndim, nu, n_nodes, flag_adjointsOnly, phi + u0 * (N - 1) * ND * ND, defect + u0 * (N - 1) * ND,
                                          xc_update + u0 * N * ND, status ? status + u0 : nullptr);
        });
    }
    CK(h, cudaSetDevice(h->device));
    const long long ns = n_traj * (long long)(n_nodes - 1), nn = n_traj * (long long)n_nodes;
    const size_t bP = al(ns * ND * ND * 8), bD = al(ns * ND * 8), bU = al(nn * ND * 8), bS = al(n_traj * 4);
    int rc = ensure(h, &h->d_out, &h->d_out_cap, bP + bD + bU + bS); if (rc) return rc;
    char* q = (char*)h->d_out;
    double* dP = (double*)q; q += bP; double* dD = (double*)q; q += bD; double* dU = (double*)q; q += bU; int32_t* dS = (int32_t*)q;
    CK(h, cudaMemcpyAsync(dP, phi, ns * ND * ND * 8, cudaMemcpyHostToDevice, h->s_compute));
    CK(h, cudaMemcpyAsync(dD, defect, ns * ND * 8, cudaMemcpyHostToDevice, h->s_compute));
    CK(h, cudaEventRecord(h->ev_t0, h->s_compute));
    rc = lto_indirect_newton_nd_dev(h, ndim, n_traj, n_nodes, flag_adjointsOnly, dP, dD, dU, dS); if (rc) return rc;
    CK(h, cudaEventRecord(h->ev_t1, h->s_compute));
    CK(h, cudaMemcpyAsync(xc_update, dU, nn * ND * 8, cudaMemcpyDeviceToHost, h->s_compute));
    if (status) CK(h, cudaMemcpyAsync(status, dS, n_traj * 4, cudaMemcpyDeviceToHost, h->s_compute));
    CK(h, cudaStreamSynchronize(h->s_compute));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

int lto_indirect_newton(lto_handle* h, int64_t n_traj, int n_nodes, int flag_adjointsOnly, const double* phi,
                        const double* defect, double* xc_update, int32_t* status) {
    return lto_indirect_newton_nd(h, 12, n_traj, n_nodes, flag_adjointsOnly, phi, defect, xc_update, status);
}

// ---- direct method: the QP of optimizeTraj (multiShoot_CRTBP_direct.jl:248-403, flagEnd = false, allowImpulsive = false) ----
int lto_direct_qp_dev(lto_handle* h, int64_t n_traj, int n_nodes, int nstate, const double* jac, const double* defect,
                      const double* u_all, const double* t_TU, const double* b0, const double* bf, double* x_update, double* u_update,
                      int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) return fail(h, LTO_ERR_ARG, "device-pointer entry points need a single-device handle (lto_init)");
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (nstate != 6 && nstate != 7) return fail(h, LTO_ERR_ARG, "nstate must be 6 or 7 (got %d)", nstate);
    if (n_traj == 0) return LTO_SUCCESS;
    if (!jac || !defect || !u_all || !t_TU || !b0 || !bf || !x_update || !u_update) return fail(h, LTO_ERR_ARG, "null array argument");
    CK(h, cudaSetDevice(h->device));
    h->nwt_traj = 0;                                                      // the workspace is shared with the indirect Newton update
    int rc = ensure(h, &h->d_nwt, &h->d_nwt_cap, direct_qp_workspace_bytes(n_traj, n_nodes, nstate)); if (rc) return rc;
    cudaError_t e = launch_direct_qp(jac, defect, nullptr, u_all, t_TU, b0, bf, (double*)h->d_nwt, x_update, u_update, status, n_traj, n_nodes,
                                     nstate, h->s_compute);
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "direct QP kernel launch: %s", cudaGetErrorString(e));
    h->launches += 1;
    return LTO_SUCCESS;
}

int lto_direct_qp(lto_handle* h, int64_t n_traj, int n_nodes, int nstate, const double* jac, const double* defect, const double* u_all,
                  const double* t_TU, const double* b0, const double* bf, double* x_update, double* u_update, int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (nstate != 6 && nstate != 7) return fail(h, LTO_ERR_ARG, "nstate must be 6 or 7 (got %d)", nstate);
    if (n_traj == 0) return LTO_SUCCESS;
    if (!jac || !defect || !u_all || !t_TU || !b0 || !bf || !x_update || !u_update) return fail(h, LTO_ERR_ARG, "null array argument");
    const long long N = n_nodes, NS = nstate, NV = 2 * (NS + 3), M0 = 6 + (nstate == 7 ? 1 : 0);
    if (h->n_child > 0) {
        return split_trajectories(h, n_traj, [&](lto_handle* c, long long u0, long long nu) {
            return lto_direct_qp(c, nu, n_nodes, nstate, jac + u0 * (N - 1) * NS * NV, defect + u0 * (N - 1) * NS, u_all + u0 * N * 3, t_TU + u0 * N,
                                 b0 + u0 * M0, bf + u0 * 6, x_update + u0 * N * NS, u_update + u0 * N * 3, status ? status + u0 : nullptr);
        });
    }
    CK(h, cudaSetDevice(h->device));
    const long long T = n_traj, ns = T * (N - 1), nn = T * N;
    const size_t bJ = al(ns * NS * NV * 8), bD = al(ns * NS * 8), bU = al(nn * 3 * 8), bT = al(nn * 8), bB0 = al(T * M0 * 8), bBf = al(T * 6 * 8),
                 bXo = al(nn * NS * 8), bS = al(T * 4);
    int rc = ensure(h, &h->d_out, &h->d_out_cap, bJ + bD + bU * 2 + bT + bB0 + bBf + bXo + bS); if (rc) return rc;
    char* q = (char*)h->d_out;
    auto take = [&](size_t b) { char* r = q; q += b; return r; };
    double* dJ = (double*)take(bJ); double* dD = (double*)take(bD); double* dU = (double*)take(bU); double* dT = (double*)take(bT);
    double* dB0 = (double*)take(bB0); double* dBf = (double*)take(bBf); double* dXo = (double*)take(bXo); double* dUo = (double*)take(bU);
    int32_t* dS = (int32_t*)take(bS);
    cudaStream_t st = h->s_compute;
    CK(h, cudaMemcpyAsync(dJ, jac, ns * NS * NV * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dD, defect, ns * NS * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dU, u_all, nn * 3 * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dT, t_TU, nn * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dB0, b0, T * M0 * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dBf, bf, T * 6 * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaEventRecord(h->ev_t0, st));
    rc = lto_direct_qp_dev(h, n_traj, n_nodes, nstate, dJ, dD, dU, dT, dB0, dBf, dXo, dUo, dS); if (rc) return rc;
    CK(h, cudaEventRecord(h->ev_t1, st));
    CK(h, cudaMemcpyAsync(x_update, dXo, nn * NS * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(u_update, dUo, nn * 3 * 8, cudaMemcpyDeviceToHost, st));
    if (status) CK(h, cudaMemcpyAsync(status, dS, T * 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

// multiShoot_CRTBP_direct's SQP loop (:465-594) resident on the device, for n_traj independent trajectories in the demo's setting
// (flagEnd = false, allowImpulsive = false, dV1 = dV2 = 0: tau1, tau2, tf stay fixed, so state_0 / state_f are constants of the call).
int lto_direct_solve_batch(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nstate, int nsteps, int max_iter,
                           double* X_all, double* u_all, const double* t_TU, const double* state_0, const double* state_f, double mass,
                           double* defect, int32_t* iters, double* er_out) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (nstate != 6 && nstate != 7) return fail(h, LTO_ERR_ARG, "nstate must be 6 or 7 (got %d)", nstate);
    if (max_iter < 0) return fail(h, LTO_ERR_ARG, "negative max_iter");
    if (p->mode != LTO_FIXED) return fail(h, LTO_ERR_ARG, "lto_direct_solve_batch runs the reference's fixed-grid ode7_8 path (LTO_FIXED)");
    if (n_traj == 0) return LTO_SUCCESS;
    if (!X_all || !u_all || !t_TU || !state_0 || !state_f) return fail(h, LTO_ERR_ARG, "null array argument");
    const long long N = n_nodes, NS = nstate, NV = 2 * (NS + 3), M0 = 6 + (nstate == 7 ? 1 : 0);
    if (h->n_child > 0) {
        return split_trajectories(h, n_traj, [&](lto_handle* c, long long u0, long long nu) {
            return lto_direct_solve_batch(c, p, nu, n_nodes, nstate, nsteps, max_iter, X_all + u0 * N * NS, u_all + u0 * N * 3, t_TU + u0 * N,
                                          state_0 + u0 * 6, state_f + u0 * 6, mass, defect ? defect + u0 * (N - 1) * NS : nullptr,
                                          iters ? iters + u0 : nullptr, er_out ? er_out + u0 : nullptr);
        });
    }
    if (n_traj > 0x7fffffffll) return fail(h, LTO_ERR_ARG, "too many trajectories");
    CK(h, cudaSetDevice(h->device));
    const int NA = 10;                                                    // alpha_all = LinRange(0.1, 1, 10)  (:411)
    const long long T = n_traj, ns = T * (N - 1), nn = T * N;
    const long long LX = N * NS, LU = N * 3, LD = (N - 1) * NS;
    cudaStream_t st = h->s_compute;
    const size_t bX = al(nn * NS * 8), bU = al(nn * 3 * 8), bT = al(nn * 8), bD = al(ns * NS * 8), bJ = al(ns * NS * NV * 8), bE = al(T * 6 * 8),
                 bB0 = al(T * M0 * 8), bVec = al((size_t)NA * T * 8), bInt = al(T * 4), bErr = al((size_t)NA * ns * 8);
    size_t need = bX * 3 + bU * 3 + bT + bD * 3 + bJ + bE * 2 + bB0 + bE + (size_t)NA * (bX + bU + bT + bD) + bVec * 6 + bInt * 6 + bErr + al(NA * 8) + 256;
    int rc = ensure(h, &h->d_slv, &h->d_slv_cap, need); if (rc) return rc;
    char* q = (char*)h->d_slv;
    auto take = [&](size_t b) { char* r = q; q += b; return r; };
    double* dX = (double*)take(bX); double* dXu = (double*)take(bX); double* dXout = (double*)take(bX);
    double* dU = (double*)take(bU); double* dUu = (double*)take(bU); double* dUout = (double*)take(bU);
    double* dT = (double*)take(bT);
    double* dDef = (double*)take(bD); double* dDtmp = (double*)take(bD); double* dDefOut = (double*)take(bD);
    double* dJ = (double*)take(bJ);
    double* dS0 = (double*)take(bE); double* dSf = (double*)take(bE); double* dB0 = (double*)take(bB0); double* dBf = (double*)take(bE);
    double* dTrX = (double*)take((size_t)NA * bX); double* dTrU = (double*)take((size_t)NA * bU); double* dTrT = (double*)take((size_t)NA * bT);
    double* dTrD = (double*)take((size_t)NA * bD);
    double* dEr = (double*)take(bVec); double* dErs = (double*)take(bVec); double* dAlpha = (double*)take(bVec); double* dScale = (double*)take(bVec);
    double* dLsTable = (double*)take(bVec); double* dErOut = (double*)take(bVec);
    int* dActive = (int*)take(bInt); int* dIters = (int*)take(bInt); int* dFlag = (int*)take(bInt);
    int* dOrig = (int*)take(bInt); int* dOrig2 = (int*)take(bInt); int* dPos = (int*)take(bInt);
    double* dErrs = (double*)take(bErr);
    double* dAlphaAll = (double*)take(al(NA * 8));
    unsigned long long* dCount = (unsigned long long*)take(256);
    CK(h, cudaMemcpyAsync(dX, X_all, nn * NS * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dU, u_all, nn * 3 * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dT, t_TU, nn * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dS0, state_0, T * 6 * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaMemcpyAsync(dSf, state_f, T * 6 * 8, cudaMemcpyHostToDevice, st));
    double alpha_all[10];
    for (int a = 0; a < NA; ++a) alpha_all[a] = 0.1 + (double)a * ((1.0 - 0.1) / (double)(NA - 1));
    alpha_all[NA - 1] = 1.0;
    CK(h, cudaMemcpyAsync(dAlphaAll, alpha_all, NA * 8, cudaMemcpyHostToDevice, st));
    CK(h, cudaStreamSynchronize(st));
    CK(h, cudaMemsetAsync(dIters, 0, T * 4, st));
    CK(h, cudaMemsetAsync(dFlag, 0, T * 4, st));
    slv::k_iota<<<slv::nblk(T, 256), 256, 0, st>>>(dOrig, dActive, T);
    h->launches += 1;
    CK(h, cudaEventRecord(h->ev_t0, st));
    long long nc = T;
    auto grid_for = [&](long long n) { return std::min<unsigned>(slv::nblk(n, 256), 148u * 16u); };
    auto defect_pass = [&](const double* X, const double* U, const double* T_, long long ntr, double* D, double* J) -> int {
        return lto_direct_dev(h, p, ntr * (N - 1), n_nodes, nstate, nsteps, X, nullptr, U, nullptr, T_, nullptr, D, dErrs, nullptr, J);
    };
    auto rowmax = [&](const double* v, long long rows, long long len, double* out) {
        slv::k_rowmaxabs<<<slv::nblk(rows * 32, 256), 256, 0, st>>>(v, rows, len, out); h->launches += 1;
    };
    auto axpy = [&](const double* x, const double* u, const double* scale, double* out, long long rows, long long len, int reps) {
        dim3 g(std::min<unsigned>(slv::nblk(rows * len, 256), 148u * 16u), (unsigned)reps);
        slv::k_axpy_rows<<<g, 256, 0, st>>>(x, u, scale, out, rows, len); h->launches += 1;
    };
    auto iter_end = [&](int it, long long* n_next) -> int {
        CK(h, cudaMemsetAsync(dCount, 0, 8, st));
        // `er = 1.0` before the loop (:490): every trajectory does one iteration whatever its first defect; no abort rule in the direct solver
        slv::k_iter_end<<<slv::nblk(nc, 256), 256, 0, st>>>(dEr, dActive, dOrig, dIters, dFlag, dErOut, dCount, nc, it, max_iter, 1e-6, INFINITY, 1);
        slv::k_retire_rows<<<grid_for(nc * LX), 256, 0, st>>>(dX, dXout, dOrig, dActive, nc, LX);
        slv::k_retire_rows<<<grid_for(nc * LU), 256, 0, st>>>(dU, dUout, dOrig, dActive, nc, LU);
        slv::k_retire_rows<<<grid_for(nc * LD), 256, 0, st>>>(dDef, dDefOut, dOrig, dActive, nc, LD);
        h->launches += 4;
        unsigned long long na = 0;
        CK(h, cudaMemcpyAsync(&na, dCount, 8, cudaMemcpyDeviceToHost, st));
        CK(h, cudaStreamSynchronize(st));
        if (na > 0 && (long long)na < nc) {
            slv::k_scan_active<<<1, 1024, 0, st>>>(dActive, dPos, nc);
            slv::k_compact_rows<double><<<grid_for(nc * LX), 256, 0, st>>>(dX, dXu, dPos, dActive, nc, LX);
            CK(h, cudaMemcpyAsync(dX, dXu, (size_t)na * LX * 8, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<double><<<grid_for(nc * LU), 256, 0, st>>>(dU, dUu, dPos, dActive, nc, LU);
            CK(h, cudaMemcpyAsync(dU, dUu, (size_t)na * LU * 8, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<double><<<grid_for(nc * LD), 256, 0, st>>>(dDef, dDtmp, dPos, dActive, nc, LD);
            CK(h, cudaMemcpyAsync(dDef, dDtmp, (size_t)na * LD * 8, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<double><<<grid_for(nc * N), 256, 0, st>>>(dT, dTrT, dPos, dActive, nc, N);
            CK(h, cudaMemcpyAsync(dT, dTrT, (size_t)na * N * 8, cudaMemcpyDeviceToDevice, st));
            slv::k_compact_rows<int><<<grid_for(nc), 256, 0, st>>>(dOrig, dOrig2, dPos, dActive, nc, 1);
            CK(h, cudaMemcpyAsync(dOrig, dOrig2, (size_t)na * 4, cudaMemcpyDeviceToDevice, st));
            slv::k_set_int<<<slv::nblk((long long)na, 256), 256, 0, st>>>(dActive, 1, (long long)na);
            h->launches += 7;
        }
        *n_next = (long long)na;
        return 0;
    };

    // ---- first nominal run (:486); er starts at 1.0 (:490)
    rc = defect_pass(dX, dU, dT, nc, dDef, nullptr); if (rc) return rc;
    rowmax(dDef, nc, LD, dEr);
    long long n_next = 0;
    rc = iter_end(0, &n_next); if (rc) return rc;
    int it = 0;
    while (n_next > 0 && it < max_iter) {
        nc = n_next;
        ++it;
        rc = defect_pass(dX, dU, dT, nc, dDef, dJ); if (rc) return rc;                          // jacobianCalc (:500): all blocks in one launch
        slv::k_direct_ends<<<slv::nblk(nc, 256), 256, 0, st>>>(dX, dS0, dSf, dOrig, mass, dB0, dBf, nc, n_nodes, nstate); h->launches += 1;
        rc = lto_direct_qp_dev(h, nc, n_nodes, nstate, dJ, dDef, dU, dT, dB0, dBf, dXu, dUu, nullptr); if (rc) return rc;   // optimizeTraj (:248-403)
        const int use_ls = it > 10;                                                               // :559-561
        if (use_ls) {
            slv::k_fill_ls<<<slv::nblk(nc * NA, 256), 256, 0, st>>>(dAlphaAll, dLsTable, nc, NA);
            slv::k_tile<<<slv::nblk((long long)NA * nc * N, 256), 256, 0, st>>>(dT, dTrT, nc * N, NA);
            h->launches += 2;
            axpy(dX, dXu, dLsTable, dTrX, nc, LX, NA);                                            // X_all + x_update*alpha (:418)
            axpy(dU, dUu, dLsTable, dTrU, nc, LU, NA);                                            // u_all + u_update*alpha (:419)
            rc = defect_pass(dTrX, dTrU, dTrT, (long long)NA * nc, dTrD, nullptr); if (rc) return rc;   // :422, all 10 x n trial trajectories in one launch
            rc = lto_sumsq_dev(h, dTrD, (long long)NA * nc, LD, dErs); if (rc) return rc;         // er[ind] = sum(defect[:].^2) (:424)
        }
        slv::k_pick_alpha<<<slv::nblk(nc, 256), 256, 0, st>>>(dErs, dAlphaAll, dActive, dAlpha, dScale, nc, use_ls, NA); h->launches += 1;
        axpy(dX, dXu, dScale, dX, nc, LX, 1);                                                     // :563
        axpy(dU, dUu, dScale, dU, nc, LU, 1);                                                     // :564
        rc = defect_pass(dX, dU, dT, nc, dDef, nullptr); if (rc) return rc;                       // :585
        rowmax(dDef, nc, LD, dEr);                                                                // :588
        rc = iter_end(it, &n_next); if (rc) return rc;
    }
    CK(h, cudaEventRecord(h->ev_t1, st));
    CK(h, cudaMemcpyAsync(X_all, dXout, nn * NS * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(u_all, dUout, nn * 3 * 8, cudaMemcpyDeviceToHost, st));
    if (defect) CK(h, cudaMemcpyAsync(defect, dDefOut, ns * NS * 8, cudaMemcpyDeviceToHost, st));
    if (iters) CK(h, cudaMemcpyAsync(iters, dIters, T * 4, cudaMemcpyDeviceToHost, st));
    if (er_out) CK(h, cudaMemcpyAsync(er_out, dErOut, T * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

int lto_indirect_solve_batch_nd(lto_handle* h, const lto_indirect_params* p, int ndim, int64_t n_traj, int n_nodes, int max_iter,
                                int flag_adjointsOnly, double* XC_all, const double* t_TU, const double* thrustLimit_traj,
                                const double* rho_traj, double* defect, int32_t* status_flag, int32_t* iters, double* er_out) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (!valid_ndim(ndim)) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (max_iter < 0) return fail(h, LTO_ERR_ARG, "negative max_iter");
    if (n_traj == 0) return LTO_SUCCESS;
    if (!XC_all || !t_TU) return fail(h, LTO_ERR_ARG, "null array argument");
    if (h->n_child > 0) {                                                 // independent solver instances: no communication between the devices
        const long long N = n_nodes;
        return split_trajectories(h, n_traj, [&](lto_handle* c, long long u0, long long nu) {
            return lto_indirect_solve_batch_nd(c, p, ndim, nu, n_nodes, max_iter, flag_adjointsOnly, XC_all + u0 * N * ndim, t_TU + u0 * N,
                                               thrustLimit_traj ? thrustLimit_traj + u0 : nullptr, rho_traj ? rho_traj + u0 : nullptr,
                                               defect ? defect + u0 * (N - 1) * ndim : nullptr, status_flag ? status_flag + u0 : nullptr,
                                               iters ? iters + u0 : nullptr, er_out ? er_out + u0 : nullptr);
        });
    }
    CK(h, cudaSetDevice(h->device));
    const long long T = n_traj, N = n_nodes, ns = T * (N - 1), nn = T * N;
    if (T > 0x7fffffffll) return fail(h, LTO_ERR_ARG, "too many trajectories");
    const long long LX = N * ndim, LD = (N - 1) * ndim;
    cudaStream_t st = h->s_compute;
    EngineArrays w{};
    // the hook retires every row whose call ended (every row starts together: one call per trajectory)
    int rc = indirect_engine(h, p, ndim, T, n_nodes, max_iter, flag_adjointsOnly, XC_all, t_TU, thrustLimit_traj, rho_traj, 0, &w,
                             [](char*) { return 0; },
                             [&](long long nc) -> int {
                                 slv::k_retire_rows<<<std::min<unsigned>(slv::nblk(nc * LX, 256), 148u * 16u), 256, 0, st>>>(w.XC, w.XCout, w.orig, w.active, nc, LX, w.flag);
                                 slv::k_retire_rows<<<std::min<unsigned>(slv::nblk(nc * LD, 256), 148u * 16u), 256, 0, st>>>(w.Def, w.DefOut, w.orig, w.active, nc, LD);
                                 h->launches += 2;
                                 return 0;
                             });
    if (rc) return rc;
    // ---- outputs (every trajectory has been retired into the caller-ordered arrays by now)
    CK(h, cudaMemcpyAsync(XC_all, w.XCout, nn * ndim * 8, cudaMemcpyDeviceToHost, st));
    if (defect) CK(h, cudaMemcpyAsync(defect, w.DefOut, ns * ndim * 8, cudaMemcpyDeviceToHost, st));
    if (iters) CK(h, cudaMemcpyAsync(iters, w.iters, T * 4, cudaMemcpyDeviceToHost, st));
    if (er_out) CK(h, cudaMemcpyAsync(er_out, w.ErOut, T * 8, cudaMemcpyDeviceToHost, st));
    std::vector<int32_t> flag((size_t)T);
    CK(h, cudaMemcpyAsync(flag.data(), w.flag, T * 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    if (status_flag) {
        for (long long j = 0; j < T; ++j) status_flag[j] = flag[(size_t)j];                    // (non-finite nodes were flagged when the row was retired)
    }
    return LTO_SUCCESS;
}

// reduceFuel_indirect (HelperFunctions.jl:105-193) for n_traj independent ladders (lto_ladder.h), every solver call on the device:
// maxIter = max_iter, p = 1, flag_adjointsOnly = false.  A ladder's next call enters the work set as soon as its last one ends.
int lto_indirect_reduce_fuel_batch(lto_handle* h, const lto_indirect_params* p, int ndim, int64_t n_traj, int n_nodes, int max_iter,
                                   double* XC_all, const double* t_TU, const double* thrustLimit_traj, const double* rho_current,
                                   const double* rho_target, const double* backoff_uniform, double* defect, int32_t* status,
                                   int32_t* calls, int32_t* newton_iters, double* rho_last) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (p->p != 1.0) return fail(h, LTO_ERR_ARG, "the rho continuation needs p = 1 (got p = %g)", p->p);
    if (!valid_ndim(ndim)) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    if (max_iter < 0) return fail(h, LTO_ERR_ARG, "negative max_iter");
    if (n_traj == 0) return LTO_SUCCESS;
    if (!XC_all || !t_TU || !rho_current || !rho_target || !backoff_uniform || !defect || !status) return fail(h, LTO_ERR_ARG, "null array argument");
    if (h->n_child > 0) {
        const long long N = n_nodes;
        return split_trajectories(h, n_traj, [&](lto_handle* c, long long u0, long long nu) {
            return lto_indirect_reduce_fuel_batch(c, p, ndim, nu, n_nodes, max_iter, XC_all + u0 * N * ndim, t_TU + u0 * N,
                                                  thrustLimit_traj ? thrustLimit_traj + u0 : nullptr, rho_current + u0, rho_target + u0,
                                                  backoff_uniform + u0 * LADDER_DRAWS, defect + u0 * (N - 1) * ndim, status + u0,
                                                  calls ? calls + u0 : nullptr, newton_iters ? newton_iters + u0 : nullptr,
                                                  rho_last ? rho_last + u0 : nullptr);
        });
    }
    CK(h, cudaSetDevice(h->device));
    const long long T = n_traj, N = n_nodes, ns = T * (N - 1), nn = T * N;
    if (T > 0x7fffffffll) return fail(h, LTO_ERR_ARG, "too many trajectories");
    const long long LX = N * ndim, LD = (N - 1) * ndim;
    cudaStream_t st = h->s_compute;
    // caller-ordered ladder arrays after the engine's: accepted starts, ladder states, draws, rho targets, the outputs
    const size_t bAcc = al(nn * ndim * 8), bLad = al(T * sizeof(LadderState)), bDraw = al(T * LADDER_DRAWS * 8), bVec = al(T * 8), bInt = al(T * 4);
    double* dAcc = nullptr; LadderState* dLad = nullptr; double* dDraw = nullptr; double* dTgt = nullptr; double* dRhoLast = nullptr;
    int* dStatus = nullptr; int* dCalls = nullptr; int* dNit = nullptr;
    EngineArrays w{};
    int rc = indirect_engine(h, p, ndim, T, n_nodes, max_iter, 0, XC_all, t_TU, thrustLimit_traj, rho_current,
                             bAcc + bLad + bDraw + bVec * 2 + bInt * 3, &w,
                             [&](char* q) -> int {
                                 dAcc = (double*)q; q += bAcc; dLad = (LadderState*)q; q += bLad; dDraw = (double*)q; q += bDraw;
                                 dTgt = (double*)q; q += bVec; dRhoLast = (double*)q; q += bVec;
                                 dStatus = (int*)q; q += bInt; dCalls = (int*)q; q += bInt; dNit = (int*)q;
                                 CK(h, cudaMemcpyAsync(dAcc, w.XC, nn * ndim * 8, cudaMemcpyDeviceToDevice, st));      // the first start
                                 CK(h, cudaMemcpyAsync(dDraw, backoff_uniform, T * LADDER_DRAWS * 8, cudaMemcpyHostToDevice, st));
                                 CK(h, cudaMemcpyAsync(dTgt, rho_target, T * 8, cudaMemcpyHostToDevice, st));
                                 slv::k_ladder_init<<<slv::nblk(T, 256), 256, 0, st>>>(w.RH, dTgt, dLad, dCalls, dNit, T);
                                 h->launches += 1;
                                 return 0;
                             },
                             [&](long long nc) -> int {
                                 slv::k_ladder_hook<<<slv::nblk(nc * 32, 256), 256, 0, st>>>(w.XC, w.Def, w.RH, w.active, w.orig, w.wit, w.iters, w.flag,
                                                                                        dLad, dDraw, dAcc, w.XCout, w.DefOut, dStatus, dCalls, dNit,
                                                                                        dRhoLast, w.count, nc, LX, LD);
                                 h->launches += 1;
                                 return 0;
                             });
    if (rc) return rc;
    CK(h, cudaMemcpyAsync(XC_all, w.XCout, nn * ndim * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(defect, w.DefOut, ns * ndim * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(status, dStatus, T * 4, cudaMemcpyDeviceToHost, st));
    if (calls) CK(h, cudaMemcpyAsync(calls, dCalls, T * 4, cudaMemcpyDeviceToHost, st));
    if (newton_iters) CK(h, cudaMemcpyAsync(newton_iters, dNit, T * 4, cudaMemcpyDeviceToHost, st));
    if (rho_last) CK(h, cudaMemcpyAsync(rho_last, dRhoLast, T * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

int lto_indirect_solve_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, int max_iter,
                             int flag_adjointsOnly, double* XC_all, const double* t_TU, const double* thrustLimit_traj,
                             const double* rho_traj, double* defect, int32_t* status_flag, int32_t* iters, double* er_out) {
    return lto_indirect_solve_batch_nd(h, p, 12, n_traj, n_nodes, max_iter, flag_adjointsOnly, XC_all, t_TU, thrustLimit_traj, rho_traj,
                                       defect, status_flag, iters, er_out);
}

}  // extern "C"
