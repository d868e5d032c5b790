// lto_guess.cu -- C ABI of the batched trajectory-stacking initial guess (include/lto_b200.h, lto_stack_guess_batch): the demos'
// two-ballistic-arc guess (CRTBP_Multishoot_direct_demo.jl:117-157, solvers.trajectory_stack_guess) for n_traj transfers in one
// call, every stage on the device:
//   state_0 = spline(X0)(tau1) -> arc 1 from t_TU[0] to its nodes and t_split -> tau2_0 = find_τ(Xf, arc-1 end)
//   -> arc 2 from t_split, starting at spline(Xf)(tau2_0), to the remaining nodes and t_TU[end] -> tau2 = find_τ(Xf, arc-2 end)
//   -> state_f = spline(Xf)(tau2) -> XC_all.
// The arcs are pairs-form segment tables (one segment per node, all starting at the arc's start) propagated by lto_indirect_dev with
// the caller's parameters and no STM -- the kernels the host path's GpuBackend.propagate reaches -- so a transfer's arcs are those of
// the host path whenever its start states are.  The orbit lookups are lto_orbit.h.  Inputs go in with one copy, results come back
// with one synchronise.
#include "lto_internal.h"
#include "lto_handle.h"
#include "lto_orbit.h"
#include <cmath>
#include <cstring>
#include <vector>

namespace lto {
namespace gss {

// out[j*6 + k] = spline(coef)(wrap(tau[j]))[k]
__global__ void k_orbit_eval(const double* __restrict__ coef, int n, const double* __restrict__ tau, double* __restrict__ out, long long T) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T * 6) return;
    out[i] = orbit_eval(coef, n, orbit_wrap(tau[i / 6]), (int)(i % 6));
}

// table[c*6 + k] = spline(coef)(tau_c)[k] for find_τ's 1001 candidates
__global__ void k_orbit_table(const double* __restrict__ coef, int n, double* __restrict__ table) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= LTO_ORBIT_NTAU * 6) return;
    table[i] = orbit_eval(coef, n, orbit_tau_candidate(i / 6), i % 6);
}

// Pairs-form segment table of one arc, thread (j, i) for i = 0 .. N.  Trajectory j's arc 1 has k1[j] + 1 segments from t_TU[j][0]:
// to the nodes with t_TU < t_split and to t_split; its arc 2 has N - k1[j] + 1 from t_split: to the remaining nodes and to
// t_TU[j][N-1].  Every segment starts at [start[j]; 0^6].
__global__ void k_arc_table(const double* __restrict__ start, const double* __restrict__ t_TU, const double* __restrict__ t_split,
                            const int* __restrict__ k1, const long long* __restrict__ off, int arc, double* __restrict__ x0,
                            double* __restrict__ t0, double* __restrict__ t1, long long T, int N) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= T * (N + 1)) return;
    const long long j = g / (N + 1);
    const int i = (int)(g - j * (N + 1)), k = k1[j];
    const double* t = t_TU + j * N;
    const int n_nodes = arc == 0 ? k : N - k;                            // nodes of this arc; segment n_nodes goes to the arc's end
    if (i > n_nodes) return;
    const long long s = off[j] + i;
    t0[s] = arc == 0 ? t[0] : t_split[j];
    t1[s] = i < n_nodes ? t[arc == 0 ? i : k + i] : (arc == 0 ? t_split[j] : t[N - 1]);
    for (int c = 0; c < 6; ++c) { x0[s * 12 + c] = start[j * 6 + c]; x0[s * 12 + 6 + c] = 0.0; }
}

// find_τ (HelperFunctions.jl:38-48), one warp per trajectory: the first of the 1001 candidates closest to the arc's end state
// x(t_end) = row off[j] + n_end[j] of the arc's output (arc 1: n_end = k1; arc 2: N - k1)
__global__ void __launch_bounds__(256) k_find_tau(const double* __restrict__ table, const double* __restrict__ arc_out,
                                                  const long long* __restrict__ off, const int* __restrict__ k1, int arc, int N,
                                                  double* __restrict__ tau, long long T) {
    const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (j >= T) return;
    const double* x = arc_out + (off[j] + (arc == 0 ? k1[j] : N - k1[j])) * 12;
    double best = 0.0; int kb = -1;
    for (int c = lane; c < LTO_ORBIT_NTAU; c += 32) {
        const double d = orbit_distance(table + c * 6, x);
        if (kb < 0 || orbit_before(d, c, best, kb)) { best = d; kb = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double d = __shfl_xor_sync(0xffffffffu, best, o);
        const int c = __shfl_xor_sync(0xffffffffu, kb, o);
        if (orbit_before(d, c, best, kb)) { best = d; kb = c; }
    }
    if (lane == 0) tau[j] = orbit_tau_candidate(kb);
}

// XC_all (12 x N per trajectory) from the arcs' node values, thread (j, i): node i < k1 from arc 1, the others from arc 2; node 0 is
// [state_0; 0], node N-1 [state_f; 0].  Thread (j, 0) also writes the trajectory's status: the worst of its arc segments'.
__global__ void k_assemble(const double* __restrict__ out1, const double* __restrict__ out2, const int32_t* __restrict__ st1,
                           const int32_t* __restrict__ st2, const long long* __restrict__ off1, const long long* __restrict__ off2,
                           const int* __restrict__ k1, const double* __restrict__ state_0, const double* __restrict__ state_f,
                           double* __restrict__ XC, int32_t* __restrict__ status, long long T, int N) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= T * N) return;
    const long long j = g / N;
    const int i = (int)(g - j * N), k = k1[j];
    double* dst = XC + g * 12;
    if (i == 0 || i == N - 1) {
        const double* s = (i == 0 ? state_0 : state_f) + j * 6;
        for (int c = 0; c < 6; ++c) { dst[c] = s[c]; dst[6 + c] = 0.0; }
    } else {
        const double* src = i < k ? out1 + (off1[j] + i) * 12 : out2 + (off2[j] + i - k) * 12;
        for (int c = 0; c < 12; ++c) dst[c] = src[c];
    }
    if (i == 0) {
        int w = 0;
        for (int s = 0; s <= k; ++s) w = max(w, (int)st1[off1[j] + s]);
        for (int s = 0; s <= N - k; ++s) w = max(w, (int)st2[off2[j] + s]);
        status[j] = w;
    }
}

static inline unsigned nblk(long long n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace gss
}  // namespace lto

using namespace lto;

extern "C" {

int lto_stack_guess_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, const double* X0_states, int n0,
                          const double* Xf_states, int nf, const double* tau1, const double* t_TU, const double* t_split, double* XC_all,
                          double* tau2, double* state_0, double* state_f, int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2 (got %d)", n_nodes);
    if (n0 < 3 || nf < 3) return fail(h, LTO_ERR_ARG, "orbit tables need >= 3 points (got n0 = %d, nf = %d)", n0, nf);
    if (n_traj == 0) return LTO_SUCCESS;
    if (!X0_states || !Xf_states || !tau1 || !t_TU || !t_split || !XC_all || !tau2 || !state_0 || !state_f)
        return fail(h, LTO_ERR_ARG, "null array argument");
    if (n_traj > 0x7fffffffll) return fail(h, LTO_ERR_ARG, "too many trajectories");
    for (long long i = 0; i < 6ll * n0; ++i)
        if (!std::isfinite(X0_states[i])) return fail(h, LTO_ERR_ARG, "X0_states has a non-finite entry (node %lld)", i / 6);
    for (long long i = 0; i < 6ll * nf; ++i)
        if (!std::isfinite(Xf_states[i])) return fail(h, LTO_ERR_ARG, "Xf_states has a non-finite entry (node %lld)", i / 6);
    const long long T = n_traj, N = n_nodes;
    for (long long j = 0; j < T; ++j) {
        const double* t = t_TU + j * N;
        for (int i = 0; i < N; ++i) {
            if (!std::isfinite(t[i])) return fail(h, LTO_ERR_ARG, "trajectory %lld: t_TU[%d] is not finite", j, i);
            if (i > 0 && !(t[i] > t[i - 1])) return fail(h, LTO_ERR_ARG, "trajectory %lld: t_TU is not strictly increasing at node %d", j, i);
        }
        if (!(t_split[j] > t[0] && t_split[j] <= t[N - 1]))
            return fail(h, LTO_ERR_ARG, "trajectory %lld: t_split = %.17g is outside (t_TU[0], t_TU[end]] = (%.17g, %.17g]", j, t_split[j], t[0], t[N - 1]);
        if (!std::isfinite(tau1[j]) || std::fabs(tau1[j]) > 1e3)
            return fail(h, LTO_ERR_ARG, "trajectory %lld: tau1 = %.17g must be finite with |tau1| <= 1e3", j, tau1[j]);
    }
    if (h->n_child > 0) {
        return split_trajectories(h, T, [&](lto_handle* c, long long u0, long long nu) {
            return lto_stack_guess_batch(c, p, nu, n_nodes, X0_states, n0, Xf_states, nf, tau1 + u0, t_TU + u0 * N, t_split + u0,
                                         XC_all + u0 * N * 12, tau2 + u0, state_0 + u0 * 6, state_f + u0 * 6, status ? status + u0 : nullptr);
        });
    }
    CK(h, cudaSetDevice(h->device));
    cudaStream_t st = h->s_compute;
    // host: the splines and the arcs' segment offsets (k1[j] nodes before t_split; arc 1 has k1 + 1 segments, arc 2 N - k1 + 1)
    std::vector<int> k1((size_t)T);
    std::vector<long long> off1((size_t)T), off2((size_t)T);
    long long S1 = 0, S2 = 0;
    for (long long j = 0; j < T; ++j) {
        const double* t = t_TU + j * N;
        int k = 0;
        while (k < N && t[k] < t_split[j]) ++k;                           // t_TU < tof1 (strict): a node at t_split starts arc 2
        k1[j] = k; off1[j] = S1; off2[j] = S2;
        S1 += k + 1; S2 += N - k + 1;
    }
    const size_t bC0 = al((size_t)(n0 - 1) * 24 * 8), bCf = al((size_t)(nf - 1) * 24 * 8), bV = al(T * 8), bTT = al(T * N * 8),
                 bK = al(T * 4), bO = al(T * 8);
    const size_t in_bytes = bC0 + bCf + bV * 2 + bTT + bK + bO * 2;
    std::vector<char> stage(in_bytes);
    {
        std::vector<double> work(4 * (size_t)std::max(n0, nf));
        char* q = stage.data();
        orbit_fit(X0_states, n0, (double*)q, work.data()); q += bC0;
        orbit_fit(Xf_states, nf, (double*)q, work.data()); q += bCf;
        memcpy(q, tau1, T * 8); q += bV;
        memcpy(q, t_split, T * 8); q += bV;
        memcpy(q, t_TU, T * N * 8); q += bTT;
        memcpy(q, k1.data(), T * 4); q += bK;
        memcpy(q, off1.data(), T * 8); q += bO;
        memcpy(q, off2.data(), T * 8);
    }
    const size_t bS6 = al(T * 6 * 8), bTab = al(LTO_ORBIT_NTAU * 6 * 8), bXC = al(T * N * 12 * 8), bSt = al(T * 4);
    const size_t bX1 = al(S1 * 12 * 8), bT1 = al(S1 * 8), bI1 = al(S1 * 4), bX2 = al(S2 * 12 * 8), bT2 = al(S2 * 8), bI2 = al(S2 * 4);
    const size_t need = in_bytes + bS6 * 3 + bV * 2 + bTab + bXC + bSt + bX1 * 2 + bT1 * 2 + bI1 + bX2 * 2 + bT2 * 2 + bI2;
    int rc = ensure(h, &h->d_slv, &h->d_slv_cap, need); if (rc) return rc;
    char* q = (char*)h->d_slv;
    auto take = [&](size_t b) { char* r = q; q += b; return r; };
    char* dIn = q;
    const double* dC0 = (const double*)take(bC0); const double* dCf = (const double*)take(bCf);
    const double* dTau1 = (const double*)take(bV); const double* dTs = (const double*)take(bV); const double* dT = (const double*)take(bTT);
    const int* dK1 = (const int*)take(bK); const long long* dOff1 = (const long long*)take(bO); const long long* dOff2 = (const long long*)take(bO);
    double* dS0 = (double*)take(bS6); double* dSf0 = (double*)take(bS6); double* dSf = (double*)take(bS6);
    double* dTau20 = (double*)take(bV); double* dTau2 = (double*)take(bV);
    double* dTab = (double*)take(bTab); double* dXC = (double*)take(bXC); int32_t* dSt = (int32_t*)take(bSt);
    double* dX1 = (double*)take(bX1); double* dA1 = (double*)take(bT1); double* dB1 = (double*)take(bT1); double* dO1 = (double*)take(bX1);
    int32_t* dSt1 = (int32_t*)take(bI1);
    double* dX2 = (double*)take(bX2); double* dA2 = (double*)take(bT2); double* dB2 = (double*)take(bT2); double* dO2 = (double*)take(bX2);
    int32_t* dSt2 = (int32_t*)take(bI2);
    CK(h, cudaMemcpyAsync(dIn, stage.data(), in_bytes, cudaMemcpyHostToDevice, st));
    CK(h, cudaEventRecord(h->ev_t0, st));
    const long long TA = T * (N + 1);
    gss::k_orbit_table<<<gss::nblk(LTO_ORBIT_NTAU * 6, 256), 256, 0, st>>>(dCf, nf, dTab);
    gss::k_orbit_eval<<<gss::nblk(T * 6, 256), 256, 0, st>>>(dC0, n0, dTau1, dS0, T);                        // state_0
    gss::k_arc_table<<<gss::nblk(TA, 256), 256, 0, st>>>(dS0, dT, dTs, dK1, dOff1, 0, dX1, dA1, dB1, T, n_nodes);
    h->launches += 3;
    CK(h, cudaGetLastError());
    rc = lto_indirect_dev(h, p, S1, 0, 12, dX1, dA1, dB1, nullptr, nullptr, nullptr, dO1, dSt1, nullptr, nullptr); if (rc) return rc;
    gss::k_find_tau<<<gss::nblk(T * 32, 256), 256, 0, st>>>(dTab, dO1, dOff1, dK1, 0, n_nodes, dTau20, T);       // tau2_0
    gss::k_orbit_eval<<<gss::nblk(T * 6, 256), 256, 0, st>>>(dCf, nf, dTau20, dSf0, T);                     // state_f0
    gss::k_arc_table<<<gss::nblk(TA, 256), 256, 0, st>>>(dSf0, dT, dTs, dK1, dOff2, 1, dX2, dA2, dB2, T, n_nodes);
    h->launches += 3;
    CK(h, cudaGetLastError());
    rc = lto_indirect_dev(h, p, S2, 0, 12, dX2, dA2, dB2, nullptr, nullptr, nullptr, dO2, dSt2, nullptr, nullptr); if (rc) return rc;
    gss::k_find_tau<<<gss::nblk(T * 32, 256), 256, 0, st>>>(dTab, dO2, dOff2, dK1, 1, n_nodes, dTau2, T);        // tau2
    gss::k_orbit_eval<<<gss::nblk(T * 6, 256), 256, 0, st>>>(dCf, nf, dTau2, dSf, T);                       // state_f
    gss::k_assemble<<<gss::nblk(T * N, 256), 256, 0, st>>>(dO1, dO2, dSt1, dSt2, dOff1, dOff2, dK1, dS0, dSf, dXC, dSt, T, n_nodes);
    h->launches += 3;
    CK(h, cudaGetLastError());
    CK(h, cudaEventRecord(h->ev_t1, st));
    CK(h, cudaMemcpyAsync(XC_all, dXC, T * N * 12 * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(tau2, dTau2, T * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(state_0, dS0, T * 6 * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(state_f, dSf, T * 6 * 8, cudaMemcpyDeviceToHost, st));
    if (status) CK(h, cudaMemcpyAsync(status, dSt, T * 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));                                     // (also keeps `stage` alive until its copy is done)
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

}  // extern "C"
