// lto_newton.cu -- the Newton update of the indirect solver on the device, batched over trajectories
// (SURVEY section 8(f) row 1): optimizeTraj_OLS of src/multiShoot_CRTBP_indirect.jl:149-218, i.e.
//
//     xc_update = -sparse(Jac_full) \ defect_vec                                   (:181-182)
//
// where Jac_full is the block-bidiagonal band [Phi_i | -I] of jacobianCalc (:114-138) with the columns of
// the first node's and the last node's states emptied (:141-142) and, with flag_adjointsOnly, the state
// columns of nodes 1..N-1 removed (:169-178).  The reference hands that matrix to SuiteSparseQR; the
// structurally empty columns get a zero update.  Here the same least-squares problem is solved by a
// Householder QR that walks the band node by node (the classical sequential orthogonal factorisation of an
// almost-block-diagonal boundary-value system), so nothing but Phi_i, defect_i and the update ever exists
// -- no Jac_full, no 255 MB device-to-host copy per iteration, no serial sparse QR per trajectory.
//
// Two systems (ND = dimension, NP = ND / 2 = pinned components per end node = rows carried between nodes):
//   12-dim [r v | lr lv]      the reference's system; pins: r, v of the first and of the last node.
//   14-dim [r v m | lr lv lm] the system with mass (solvers._end_pins(7)); pins: r, v, m of the first node (0..6),
//                             r, v and lm of the last node (0..5, 13) -- the final mass is solved for.
//
//   full mode (NU = ND unknowns per node).  The pinned end states are kept as unknowns and pinned by the
//     NP equations [I 0] delta_1 = 0 / (pin rows) delta_N = 0: the system is square and non-singular, so this
//     is the same solution (the pinned entries are returned as exact zeros).  Node i's panel is
//         rows 0..NP-1    carry   [ C_i    0   | c_i ]     (i = 1: [I 0 | 0])
//         rows NP..NR-1   defects [ Phi_i  -I  | -d_i ]    (i = N: pin rows, zero rows)
//     ND reflections annihilate the delta_i columns: rows 0..ND-1 = [R_i S_i | s_i] are stored, rows ND..NR-1
//     involve delta_{i+1} only and become the next carry.  (12-dim: NR = 18, 25 columns; 14-dim: NR = 21, 29 columns.)
//   adjoints-only mode (NU = NP).  Over-determined; after the NU reflections on delta_i the ND remaining rows are
//     compressed onto the NU columns of delta_{i+1} by NU more reflections, rows NU..2NU-1 are carried, rows
//     2NU..NR-1 are pure residual and dropped.  The unknowns are the costates of nodes 0..N-2 and the unpinned
//     components of the last node: its costates at 12 dims, m, lr, lv (columns 6..12) at 14 dims.
//   back substitution  R_i delta_i = s_i - S_i delta_{i+1},  i = N..1.
//
// Mapping: ONE WARP PER TRAJECTORY.  Forward sweep: lane = panel column (2 NU + 1 of them, at most 29), the column's NR
// rows live in registers with compile-time indices; the Householder vector of the pivot lane is handed to the
// other lanes through a per-warp shared-memory buffer (one __syncwarp per reflection).  The stored factor
// rows go to a workspace in HBM (coalesced: lanes = consecutive columns of one row).  Back substitution:
// lane = row.  The sweep is a dependent chain (latency bound, ~2-3 k cycles per node); throughput comes
// from the 1,024 trajectories of a continuation batch running side by side (7 warps per SM).
#include "lto_internal.h"
#include "lto_cw_common.cuh"
#include <algorithm>

namespace lto {
namespace nwt {

constexpr int WARPS = 4;          // trajectories per CTA

// Geometry of the update with NU unknowns per node: NU = 12 / 6 is the 12-dim system (full / adjoints-only),
// NU = 14 / 7 the 14-dim one.  Stored rows stay 16-byte aligned for the double2 loads.
template <int NU>
struct Geo {
    static constexpr int ND = (NU == 12 || NU == 6) ? 12 : 14;   // system dimension (the reference's solver: 12, :258, :324-325)
    static constexpr int NP = ND / 2;                            // pins per end node = carried rows: 6 / 7
    static constexpr int NR = NP + ND;                           // panel rows: 18 / 21
    static constexpr int WROW = 2 * ND + 2;                      // doubles per stored factor row (2 ND + 1 used): 26 / 30
    static constexpr int VROW = (NR + 2) & ~1;                   // doubles per stored reflection: v[0..NR-1] (zero above the pivot), gamma, pad: 20 / 22
    static constexpr int VBUF = VROW;                            // doubles per Householder hand-off buffer (NR + gamma)
    static constexpr int NREF = ND;                              // reflections per node (full: ND sweeps; adjoints-only: NP sweeps + NP compressions)
    static constexpr int C0 = ND - NU;                           // first kept column of nodes 0..N-2 (0, or NP = the costates)
    static constexpr int C0L = (NU == ND) ? 0 : 6;               // of the last node (adjoints-only: everything after r, v that is not pinned)
    static_assert(NU == ND || NU == NP, "NU is ND (full) or ND / 2 (adjoints-only)");
    static_assert(2 * NU + 1 <= 32 && NR + 1 <= 32, "one warp holds the panel");
};

__host__ __device__ constexpr size_t wbytes_per_node(int nd) { return (size_t)nd * (2 * nd + 2) * sizeof(double); }
__host__ __device__ constexpr size_t vbytes_per_node(int nd) { return (size_t)nd * ((nd / 2 + nd + 2) & ~1) * sizeof(double); }
static_assert(wbytes_per_node(12) == 12 * Geo<12>::WROW * sizeof(double) && vbytes_per_node(12) == Geo<12>::NREF * Geo<12>::VROW * sizeof(double), "");
static_assert(wbytes_per_node(14) == 14 * Geo<14>::WROW * sizeof(double) && vbytes_per_node(14) == Geo<14>::NREF * Geo<14>::VROW * sizeof(double), "");

template <int NU>
__device__ __forceinline__ void load_rows(double (&nx)[Geo<NU>::ND], int lane, bool have, bool next_is_last, const double* __restrict__ phi_seg,
                                          const double* __restrict__ d_seg) {
    // rows NP..NR-1 of the next panel: [Phi_i(:, kept of node i) | -I(:, kept of node i+1) | -d_i]
    using G = Geo<NU>;
    constexpr int ND = G::ND, C0 = G::C0;
#pragma unroll
    for (int r = 0; r < ND; ++r) nx[r] = 0.0;
    if (!have) return;
    if (lane < NU) {
        const double2* p = reinterpret_cast<const double2*>(phi_seg + (C0 + lane) * ND);     // column-major block: 96 / 112 contiguous bytes
#pragma unroll
        for (int r = 0; r < ND; r += 2) { const double2 v = __ldg(p + r / 2); nx[r] = v.x; nx[r + 1] = v.y; }
    } else if (lane < 2 * NU) {
        const int c = (next_is_last ? G::C0L : C0) + lane - NU;
#pragma unroll
        for (int r = 0; r < ND; ++r) nx[r] = (r == c) ? -1.0 : 0.0;
    } else if (lane == 2 * NU) {
#pragma unroll
        for (int r = 0; r < ND; ++r) nx[r] = -__ldg(d_seg + r);
    }
}

// One Householder reflection: pivot column = lane PL, pivot row PR; rows PR..NR-1; applied to lanes > PL.
// The pivot lane only publishes its raw column x; every lane forms x.a_c and |x|^2 itself, and alpha, v_k, gamma are computed
// redundantly by all lanes, so nothing waits on a single lane's sqrt / reciprocal or on a shuffle:
//     v = x - alpha e_k,   H y = y + v (v.y) / (alpha v_k),   v.y = x.y - alpha y_k,   alpha v_k = -|x| (|x_k| + |x|)
template <int NU, int PL, int PR>
__device__ __forceinline__ void reflect(double (&a)[Geo<NU>::NR], int lane, double* __restrict__ vb, double* __restrict__ vstore) {
    constexpr int NR = Geo<NU>::NR, VBUF = Geo<NU>::VBUF, VROW = Geo<NU>::VROW;
    double2* v2 = reinterpret_cast<double2*>(vb + ((PL & 1) ? VBUF : 0));   // double buffer: one __syncwarp per reflection
    double* v1 = reinterpret_cast<double*>(v2);
    if (lane == PL) {
#pragma unroll
        for (int i = 0; i < NR / 2; ++i) v2[i] = make_double2(a[2 * i], a[2 * i + 1]);   // the whole column: 9 / 10 x 16 bytes (+ 8)
        if (NR & 1) v1[NR - 1] = a[NR - 1];
    }
    __syncwarp();
    double x[NR];
#pragma unroll
    for (int i = 0; i < NR / 2; ++i) { const double2 t = v2[i]; x[2 * i] = t.x; x[2 * i + 1] = t.y; }
    if (NR & 1) x[NR - 1] = v1[NR - 1];
    // |x|^2 and x.a_c as independent short chains; no lane waits for another lane's result
    double d[4] = {0.0, 0.0, 0.0, 0.0}, g[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int r = PR; r < NR; ++r) {
        d[(r - PR) & 3] = fma(x[r], a[r], d[(r - PR) & 3]);
        g[(r - PR) & 3] = fma(x[r], x[r], g[(r - PR) & 3]);
    }
    const double dot = (d[0] + d[1]) + (d[2] + d[3]);
    const double sigma = (g[0] + g[1]) + (g[2] + g[3]);
    double alpha = 0.0, vk = 0.0, gamma = 0.0;
    if (sigma > 0.0) {
        const double inv = cwc::fast_rsqrt(sigma), nrm = sigma * inv;
        alpha = (x[PR] >= 0.0) ? -nrm : nrm;
        vk = x[PR] - alpha;
        gamma = -inv * cwc::fast_rcp(fabs(x[PR]) + nrm);
    } else if (!(sigma == 0.0)) {
        alpha = sigma; gamma = sigma;                            // NaN: propagate (reported through status[])
    }
    if (vstore && lane <= NR) {                                  // keep the reflection for lto_indirect_newton_resolve (index = PR):
        // v = x below the pivot row, v_k at it, zeros above it, then gamma: NR + 1 lanes store contiguous doubles
        double mine = (lane < NR) ? v1[lane] : gamma;
        mine = (lane < PR) ? 0.0 : ((lane == PR) ? vk : mine);
        vstore[PR * VROW + lane] = mine;
    }
    if (lane >= PL) {
        // the pivot lane runs the same update (x.x = sigma gives t = -1: its sub-diagonal becomes rounding-level, never read again)
        const double t = fma(-alpha, a[PR], dot) * gamma;
        a[PR] = (lane == PL) ? alpha : fma(vk, t, a[PR]);
#pragma unroll
        for (int r = PR + 1; r < NR; ++r) a[r] = fma(x[r], t, a[r]);
    }
}

// the NU reflections on the columns of delta_i
template <int NU, int K>
__device__ __forceinline__ void sweep(double (&a)[Geo<NU>::NR], int lane, double* vb, double* vs) {
    if constexpr (K < NU) {
        reflect<NU, K, K>(a, lane, vb, vs);
        sweep<NU, K + 1>(a, lane, vb, vs);
    }
}
// compression of rows NU..NR-1 onto the next node's NP columns (adjoints-only mode)
template <int NU, int K>
__device__ __forceinline__ void compress(double (&a)[Geo<NU>::NR], int lane, double* vb, double* vs) {
    if constexpr (K < Geo<NU>::NP) {
        reflect<NU, NU + K, NU + K>(a, lane, vb, vs);
        compress<NU, K + 1>(a, lane, vb, vs);
    }
}

// Back substitution R_i delta_i = s_i - S_i delta_{i+1}, i = N..1: lane = row of the stored factor.
template <int NU>
__device__ __forceinline__ void back_substitute(const double* __restrict__ W_t, double* __restrict__ update, int32_t* __restrict__ status,
                                                long long traj, int N, int lane) {
    using G = Geo<NU>;
    constexpr int ND = G::ND, WROW = G::WROW;
    const unsigned full = 0xffffffffu;
    double dn[NU];                      // delta_{i+1}, replicated in every lane
#pragma unroll
    for (int c = 0; c < NU; ++c) dn[c] = 0.0;
    bool bad = false;
    const int rl = (lane < NU) ? lane : 0;
    double2 rowv[WROW / 2], nxt[WROW / 2];
    {
        const double2* p = reinterpret_cast<const double2*>(W_t + ((long long)(N - 1) * ND + rl) * WROW);
#pragma unroll
        for (int q = 0; q < WROW / 2; ++q) nxt[q] = p[q];
    }
#pragma unroll 1
    for (int i = N - 1; i >= 0; --i) {
#pragma unroll
        for (int q = 0; q < WROW / 2; ++q) rowv[q] = nxt[q];
        if (i > 0) {
            const double2* p = reinterpret_cast<const double2*>(W_t + ((long long)(i - 1) * ND + rl) * WROW);
#pragma unroll
            for (int q = 0; q < WROW / 2; ++q) nxt[q] = p[q];
        }
        double row[WROW];
#pragma unroll
        for (int q = 0; q < WROW / 2; ++q) { row[2 * q] = rowv[q].x; row[2 * q + 1] = rowv[q].y; }
        double y = row[2 * NU];
#pragma unroll
        for (int j = 0; j < NU; ++j) y = fma(-row[NU + j], dn[j], y);
        double diag = 1.0;
#pragma unroll
        for (int c = 0; c < NU; ++c) diag = (lane == c) ? row[c] : diag;
        const double invd = cwc::fast_rcp(diag);
        double mine = 0.0;
#pragma unroll
        for (int c = NU - 1; c >= 0; --c) {
            const double xc = __shfl_sync(full, y * invd, c);
            dn[c] = xc;
            mine = (lane == c) ? xc : mine;
            if (lane < c) y = fma(-row[c], xc, y);
        }
        if (NU == ND && (i == 0 || i == N - 1)) {                 // pinned end states: structurally empty columns (:141-142)
#pragma unroll
            for (int c = 0; c < 6; ++c) dn[c] = 0.0;
            if (lane < 6) mine = 0.0;
            if constexpr (ND == 14) {                             // m of the first node, lm of the last node
                const int c = (i == 0) ? 6 : 13;
#pragma unroll
                for (int k = 6; k < ND; ++k) dn[k] = (k == c) ? 0.0 : dn[k];
                if (lane == c) mine = 0.0;
            }
        }
        bad |= !(fabs(mine) <= 1.79e308);
        double* out = update + (traj * (long long)N + i) * ND;
        if (NU == ND) { if (lane < ND) out[lane] = mine; }
        else if (lane < ND) {                                      // the kept columns only (:169-178)
            const int c0 = (i == N - 1) ? G::C0L : G::C0;
            const double lam = __shfl_sync((1u << ND) - 1u, mine, lane >= c0 ? lane - c0 : lane);
            out[lane] = (lane < c0 || lane >= c0 + NU) ? 0.0 : lam;
        }
    }
    const bool anybad = __any_sync(full, bad && lane < NU);
    if (status && lane == 0) status[traj] = anybad ? LTO_ST_NAN : 0;
}

template <int NU>
__global__ void __launch_bounds__(32 * WARPS) k_indirect_newton(const double* __restrict__ phi, const double* __restrict__ defect,
                                                                 double* __restrict__ W, double* __restrict__ V, double* __restrict__ update,
                                                                 int32_t* __restrict__ status, long long n_traj, int n_nodes) {
    using G = Geo<NU>;
    constexpr int ND = G::ND, NP = G::NP, NR = G::NR, WROW = G::WROW, VROW = G::VROW, NREF = G::NREF;
    __shared__ __align__(16) double vbuf[WARPS][2 * G::VBUF];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long traj = (long long)blockIdx.x * WARPS + wid;
    if (traj >= n_traj) return;
    constexpr int NCOL = 2 * NU + 1;
    const int N = n_nodes;
    const double* phi_t = phi + traj * (long long)(N - 1) * ND * ND;
    const double* d_t = defect + traj * (long long)(N - 1) * ND;
    double* W_t = W + traj * (long long)N * ND * WROW;
    double* V_t = V ? V + traj * (long long)N * NREF * VROW : nullptr;
    double* vb = vbuf[wid];
    const unsigned full = 0xffffffffu;
    // the pin row of the last node that lane c carries (full mode): r, v -> rows 0..5, lm (14-dim) -> row 6; -1 if c is free
    const int pin_last = (lane < 6) ? lane : ((ND == 14 && lane == ND - 1) ? 6 : -1);

    // ---------------- forward sweep
    double a[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) a[r] = 0.0;
    if (NU == ND && lane < NP) {
#pragma unroll
        for (int r = 0; r < NP; ++r) a[r] = (r == lane) ? 1.0 : 0.0;      // [I 0] delta_1 = 0  (:141)
    }
    double nx[ND];
    load_rows<NU>(nx, lane, N > 1, N == 2, phi_t, d_t);
#pragma unroll 1
    for (int i = 0; i < N; ++i) {
        if (i < N - 1) {
#pragma unroll
            for (int r = 0; r < ND; ++r) a[NP + r] = nx[r];
        } else {
#pragma unroll
            for (int r = 0; r < ND; ++r) a[NP + r] = 0.0;
            if (NU == ND && pin_last >= 0) {
#pragma unroll
                for (int r = 0; r < NP; ++r) a[NP + r] = (r == pin_last) ? 1.0 : 0.0;   // pin rows: delta_N = 0 on the pinned components (:142)
            }
        }
        // prefetch the next node's block while this one is factorised
        load_rows<NU>(nx, lane, i + 1 < N - 1, i + 2 == N - 1, phi_t + (long long)(i + 1) * ND * ND, d_t + (long long)(i + 1) * ND);
        double* vs = V_t ? V_t + (long long)i * NREF * VROW : nullptr;
        sweep<NU, 0>(a, lane, vb, vs);
        if constexpr (NU < ND) compress<NU, 0>(a, lane, vb, vs);
        if (lane < NCOL) {
            double* w = W_t + (long long)i * ND * WROW + lane;
#pragma unroll
            for (int r = 0; r < NU; ++r) w[r * WROW] = a[r];
        }
        // carry: rows NU..NU+NP-1 of the next node's columns (+ rhs) become rows 0..NP-1 of the next panel
#pragma unroll
        for (int r = 0; r < NP; ++r) {
            const double up = __shfl_sync(full, a[NU + r], (lane + NU) & 31);
            a[r] = (lane < NU) ? up : ((lane == 2 * NU) ? a[NU + r] : 0.0);
        }
    }
    __syncwarp();
    __threadfence_block();
    back_substitute<NU>(W_t, update, status, traj, N, lane);
}

// Second solve with the SAME matrix (the second-order correction, multiShoot_CRTBP_indirect.jl:207): the stored reflections
// are replayed on the new right-hand side -- every lane carries the whole NR-row rhs column and does the identical arithmetic,
// so a reflection is a 4-chain dot product and one FMA sweep with no exchange between lanes -- then the same back substitution.
template <int NU>
__global__ void __launch_bounds__(32 * WARPS) k_indirect_newton_resolve(const double* __restrict__ defect, double* __restrict__ W,
                                                                         const double* __restrict__ V, double* __restrict__ update,
                                                                         int32_t* __restrict__ status, long long n_traj, int n_nodes) {
    using G = Geo<NU>;
    constexpr int ND = G::ND, NP = G::NP, NR = G::NR, WROW = G::WROW, VROW = G::VROW, NREF = G::NREF;
    constexpr int NV2 = NREF * VROW / 2;                                // double2 per node of stored reflections (120 / 154)
    __shared__ __align__(16) double2 vsm[WARPS][2][NV2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long traj = (long long)blockIdx.x * WARPS + wid;
    if (traj >= n_traj) return;
    const int N = n_nodes;
    const double* d_t = defect + traj * (long long)(N - 1) * ND;
    double* W_t = W + traj * (long long)N * ND * WROW;
    const double2* V_t = reinterpret_cast<const double2*>(V + traj * (long long)N * NREF * VROW);
    // a node's reflections come from HBM: fetched one node ahead into shared memory (all lanes then read them as broadcasts)
    auto fetch = [&](int node, int buf) {
        const double2* src = V_t + (long long)node * NV2;
        const unsigned dst = cwc::smem_u32(&vsm[wid][buf][0]);
        for (int q = lane; q < NV2; q += 32)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (unsigned)(q * sizeof(double2))), "l"(src + q) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto load_d = [&](int node, double (&dd)[ND]) {
        if (node < N - 1) {
            const double2* dp = reinterpret_cast<const double2*>(d_t + (long long)node * ND);
#pragma unroll
            for (int r = 0; r < ND; r += 2) { const double2 v = __ldg(dp + r / 2); dd[r] = -v.x; dd[r + 1] = -v.y; }
        } else {
#pragma unroll
            for (int r = 0; r < ND; ++r) dd[r] = 0.0;
        }
    };
    double y[NR], dnext[ND];
#pragma unroll
    for (int r = 0; r < NR; ++r) y[r] = 0.0;
    fetch(0, 0);
    load_d(0, dnext);
#pragma unroll 1
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int r = 0; r < ND; ++r) y[NP + r] = dnext[r];
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();                                                    // every lane's part of node i's reflections has landed
        if (i + 1 < N) { fetch(i + 1, (i + 1) & 1); load_d(i + 1, dnext); }
        const double2* vp = &vsm[wid][i & 1][0];
#pragma unroll
        for (int k = 0; k < NREF; ++k) {
            double v[VROW];
#pragma unroll
            for (int q = k / 2; q < VROW / 2; ++q) { const double2 t = vp[k * (VROW / 2) + q]; v[2 * q] = t.x; v[2 * q + 1] = t.y; }
            double d[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int r = k; r < NR; ++r) d[(r - k) & 3] = fma(v[r], y[r], d[(r - k) & 3]);
            const double t = ((d[0] + d[1]) + (d[2] + d[3])) * v[NR];
#pragma unroll
            for (int r = k; r < NR; ++r) y[r] = fma(v[r], t, y[r]);
        }
        // the rhs column of the stored factor rows, then the carry
        double mine = 0.0;
#pragma unroll
        for (int r = 0; r < NU; ++r) mine = (lane == r) ? y[r] : mine;
        if (lane < NU) W_t[((long long)i * ND + lane) * WROW + 2 * NU] = mine;
#pragma unroll
        for (int r = 0; r < NP; ++r) y[r] = y[NU + r];
        __syncwarp();                                                    // all lanes are done with this buffer before it is refilled (node i + 2)
    }
    __syncwarp();
    __threadfence_block();
    back_substitute<NU>(W_t, update, status, traj, N, lane);
}

}  // namespace nwt

// the factor rows of every node, then the stored reflections of every node
size_t indirect_newton_workspace_bytes(long long n_traj, int n_nodes, int ndim) {
    return (size_t)n_traj * (size_t)n_nodes * (nwt::wbytes_per_node(ndim) + nwt::vbytes_per_node(ndim));
}
static double* reflections_of(double* work, long long n_traj, int n_nodes, int ndim) {
    return work + (size_t)n_traj * (size_t)n_nodes * (nwt::wbytes_per_node(ndim) / sizeof(double));
}

cudaError_t launch_indirect_newton(const double* phi, const double* defect, double* work, double* update, int32_t* status,
                                   long long n_traj, int n_nodes, int ndim, bool adjoints_only, cudaStream_t st) {
    if (n_traj <= 0 || n_nodes < 2 || (ndim != 12 && ndim != 14)) return cudaErrorInvalidValue;
    const long long blocks = (n_traj + nwt::WARPS - 1) / nwt::WARPS;
    if (blocks > 0x7fffffffll) return cudaErrorInvalidValue;
    double* V = reflections_of(work, n_traj, n_nodes, ndim);
    const dim3 g((unsigned)blocks), b(32 * nwt::WARPS);
    if (ndim == 12) {
        if (adjoints_only) nwt::k_indirect_newton<6><<<g, b, 0, st>>>(phi, defect, work, V, update, status, n_traj, n_nodes);
        else nwt::k_indirect_newton<12><<<g, b, 0, st>>>(phi, defect, work, V, update, status, n_traj, n_nodes);
    } else {
        if (adjoints_only) nwt::k_indirect_newton<7><<<g, b, 0, st>>>(phi, defect, work, V, update, status, n_traj, n_nodes);
        else nwt::k_indirect_newton<14><<<g, b, 0, st>>>(phi, defect, work, V, update, status, n_traj, n_nodes);
    }
    return cudaGetLastError();
}

// same matrix, new right-hand side: needs the workspace of the preceding launch_indirect_newton with the same shape, dimension and mode
cudaError_t launch_indirect_newton_resolve(const double* defect, double* work, double* update, int32_t* status, long long n_traj, int n_nodes,
                                           int ndim, bool adjoints_only, cudaStream_t st) {
    if (n_traj <= 0 || n_nodes < 2 || (ndim != 12 && ndim != 14)) return cudaErrorInvalidValue;
    const long long blocks = (n_traj + nwt::WARPS - 1) / nwt::WARPS;
    if (blocks > 0x7fffffffll) return cudaErrorInvalidValue;
    const double* V = reflections_of(work, n_traj, n_nodes, ndim);
    const dim3 g((unsigned)blocks), b(32 * nwt::WARPS);
    if (ndim == 12) {
        if (adjoints_only) nwt::k_indirect_newton_resolve<6><<<g, b, 0, st>>>(defect, work, V, update, status, n_traj, n_nodes);
        else nwt::k_indirect_newton_resolve<12><<<g, b, 0, st>>>(defect, work, V, update, status, n_traj, n_nodes);
    } else {
        if (adjoints_only) nwt::k_indirect_newton_resolve<7><<<g, b, 0, st>>>(defect, work, V, update, status, n_traj, n_nodes);
        else nwt::k_indirect_newton_resolve<14><<<g, b, 0, st>>>(defect, work, V, update, status, n_traj, n_nodes);
    }
    return cudaGetLastError();
}

}  // namespace lto
