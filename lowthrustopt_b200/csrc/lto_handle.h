// lto_handle.h -- the library handle and the error helpers shared by the C ABI translation units
// (lto_capi.cu: propagation entry points; lto_solve.cu: Newton update / batched solver entry points; lto_guess.cu: the batched
// trajectory-stacking guess).
#pragma once
#include "../../include/lto_b200.h"
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stddef.h>
#include <stdint.h>
#include <thread>
#include <vector>

static const size_t LTO_PROF_WORDS = 16384;
#define LTO_MAX_DEVICES 16

struct lto_handle {
    int device;
    int n_sm;
    cudaStream_t s_compute, s_copy, s_h2d;          // kernels; device->host (and peer pushes); host->device
    cudaEvent_t ev_in, ev_t0, ev_t1;
    cudaEvent_t ev_chunk[8], ev_h2d[8];
    void* d_in; size_t d_in_cap;
    void* d_out; size_t d_out_cap;
    void* h_stage; size_t h_stage_cap;          // pinned staging of PAGEABLE caller inputs (direct host calls), grow-only
    unsigned long long* d_ctr;
    void* d_scr; size_t d_scr_cap;
    unsigned long long* d_prof;                 // LTO_ICW_PROF=1: per-warp cycle counters of the last indirect throughput launch
    void* d_nwt; size_t d_nwt_cap;              // factor workspace of the Newton update (lto_newton.cu)
    long long nwt_traj; int nwt_nodes, nwt_adj;  // shape / mode of the factorisation it holds (0 trajectories: none)
    int nwt_ndim;                               // and its system dimension (12 or 14)
    void* d_slv; size_t d_slv_cap;              // arrays of the batched solver (lto_solve.cu)
    int64_t launches;
    double last_ms;
    char err[512];
    int n_child;                                // > 0: a multi-device handle (lto_init_devices); the work is done by the children
    lto_handle* child[LTO_MAX_DEVICES];
};

// NVTX range around every C-ABI entry point that does device work (SURVEY section 5, tracing): shows up as a named span on the
// calling thread's timeline in Nsight Systems / ncu --nvtx; header-only NVTX3, a no-op when no tool is attached.
struct LtoNvtxRange {
    explicit LtoNvtxRange(const char* name) { nvtxRangePushA(name); }
    ~LtoNvtxRange() { nvtxRangePop(); }
};
#define LTO_NVTX() LtoNvtxRange lto_nvtx_range__(__func__)

int lto_fail(lto_handle* h, int code, const char* fmt, ...);
int lto_ensure(lto_handle* h, void** p, size_t* cap, size_t need);      // grow-only device buffer
#define fail lto_fail
#define ensure lto_ensure
#define CK(h, call)                                                                                   \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return fail(h, LTO_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
    } while (0)

static inline size_t al(size_t x) { return (x + 255) & ~(size_t)255; }

// Multi-device handles (lto_init_devices): whole trajectories in equal contiguous ranges, one host worker thread per device;
// every device copies its slab of the results straight into the caller's arrays.
template <class F>
static inline int split_trajectories(lto_handle* h, long long n_traj, F&& call) {
    const int nc = h->n_child;
    std::vector<int> rcs(nc, 0);
    std::vector<std::thread> th;
    for (int i = 0; i < nc; ++i) {
        const long long u0 = n_traj * i / nc, u1 = n_traj * (i + 1) / nc;
        if (u1 <= u0) continue;
        th.emplace_back([&, i, u0, u1] { rcs[i] = call(h->child[i], u0, u1 - u0); });
    }
    for (auto& t : th) t.join();
    for (int i = 0; i < nc; ++i)
        if (rcs[i]) return fail(h, rcs[i], "device %d: %s", h->child[i]->device, h->child[i]->err);
    return LTO_SUCCESS;
}
