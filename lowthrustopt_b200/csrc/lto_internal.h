// lto_internal.h -- argument blocks shared by the C ABI layer and the kernel launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "lto_prop_generic.cuh"

namespace lto {

// Device-pointer view of one direct-method call (multiShoot_CRTBP_direct.jl:66-143).
// npt == 0: pairs form, segment s reads row s of Xa/Xb/ua/ub/ta/tb.
// npt  > 0: trajectory form with npt nodes per trajectory; segment s = (j, i) reads nodes
//           j*npt+i (a) and j*npt+i+1 (b) of X_all/u_all/t_TU passed in Xa/ua/ta.
struct DirectArgs {
    const double *Xa, *Xb, *ua, *ub, *ta, *tb;
    double *defect, *errors, *jac;
    int32_t* status;
    long long n_seg;
    int npt;
    DirectCfg cfg;
    EPConst c;
};

struct IndirectArgs {
    const double *x0, *t0, *t1, *x_target;
    const double *thrustLimit_arr, *rho_arr;   // per segment (pairs) or per trajectory (npt > 0), or NULL
    double *defect, *phi;
    int32_t *status, *nsteps_out;
    unsigned long long* counter;               // device work-queue counter (throughput kernel)
    double* scratch;                           // indirect_cw_scratch_bytes(n_sm) of device memory (throughput kernel)
    unsigned long long* prof;                  // optional per-warp cycle counters [grid][8 warps][4] (diagnostics), or NULL
    long long n_seg;
    int npt;
    IndirectCfg cfg;
    SCConst c;
    double* quad;                              // K4 cost pass only (launch_indirect_cost): per segment (int |a_u| dt, int |a_u|^2 dt)
    // K4 switch pass only (launch_indirect_switch): per segment the first max_switch (time, direction) switches of |lv| - 1 on its steps,
    // their count, and the on (1) / off (0) side of |lv| - 1 at its start (bit 0) and at its propagated end (bit 1)
    double* sw_t;
    int32_t *sw_dir, *sw_count, *sw_side;
    int max_switch;
};

__host__ __device__ inline long long lto_node_a(long long s, int npt) { return npt > 0 ? s + s / (npt - 1) : s; }
__host__ __device__ inline long long lto_traj_of(long long s, int npt) { return npt > 0 ? s / (npt - 1) : s; }

// launchers (each returns the launch error and the number of kernels it enqueued)
cudaError_t launch_direct_generic(const DirectArgs& a, int nstate, cudaStream_t st, int* n_launch);
cudaError_t launch_indirect_generic(const IndirectArgs& a, int ndim, cudaStream_t st, int* n_launch);
// throughput kernels; return cudaErrorNotSupported when the configuration is not covered
cudaError_t launch_direct_fast(const DirectArgs& a, int nstate, cudaStream_t st, int* n_launch);
cudaError_t launch_indirect_fast(const IndirectArgs& a, int ndim, cudaStream_t st, int* n_launch);
size_t indirect_cw_scratch_bytes(int n_sm);
// K4 with the control-cost quadrature (a.quad) and the per-trajectory sums of lto_indirect_cost_batch: dv[j] = dv_scale * sum of the
// trajectory's int |a_u| dt, energy[j] = e_scale * sum of its int |a_u|^2 dt, status_traj[j] = the worst segment status (a.status)
cudaError_t launch_indirect_cost(const IndirectArgs& a, long long n_traj, double dv_scale, double e_scale, double* dv, double* energy,
                                 int32_t* status_traj, cudaStream_t st, int* n_launch);
// K4 with the switch scan (a.sw_*) and the per-trajectory assembly of lto_indirect_switch_batch: t_node (n_traj x npt) are the node times
// of the node rule; per trajectory the first max_switch (t_switch, direction) and n_switch (-1 where status_traj is not LTO_ST_OK),
// on_start and the worst segment status
cudaError_t launch_indirect_switch(const IndirectArgs& a, long long n_traj, const double* t_node, double* t_switch, int32_t* direction,
                                   int32_t* n_switch, int32_t* on_start, int32_t* status_traj, cudaStream_t st, int* n_launch);
cudaError_t launch_sumsq_rows(const double* v, long long n_rows, long long len, double* out, cudaStream_t st);
cudaError_t launch_fp64_probe(int iters, double* d_sink, int n_sm, cudaStream_t st, long long* n_threads, int* chains);

}  // namespace lto
