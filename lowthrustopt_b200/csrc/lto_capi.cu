// lto_capi.cu -- the C ABI of liblto_b200.so (include/lto_b200.h): handle, device
// scratch, host<->device pipelining and kernel dispatch.  No torch, no C++ types
// across the boundary, no exceptions, no CPU fallback.
#include "../../include/lto_b200.h"
#include "lto_internal.h"
#include "lto_handle.h"
#include <cstdio>
#include <cstring>
#include <cstdarg>
#include <algorithm>
#include <cstdlib>
#include <cmath>
#include <thread>
#include <vector>

using namespace lto;

static char g_err[512] = "";

int lto_fail(lto_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    snprintf(g_err, sizeof g_err, "%s", buf);
    if (h) snprintf(h->err, sizeof h->err, "%s", buf);
    return code;
}

int lto_ensure(lto_handle* h, void** p, size_t* cap, size_t need) {
    if (need <= *cap) return 0;
    if (*p) { cudaError_t e = cudaFree(*p); *p = nullptr; *cap = 0; if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "cudaFree: %s", cudaGetErrorString(e)); }
    size_t want = need + need / 4 + 4096;
    cudaError_t e = cudaMalloc(p, want);
    if (e != cudaSuccess) { *p = nullptr; return fail(h, LTO_ERR_NOMEM, "cudaMalloc(%zu): %s", want, cudaGetErrorString(e)); }
    *cap = want;
    return 0;
}

extern "C" {

int lto_version(void) { return LTO_B200_VERSION; }

void lto_direct_params_default(lto_direct_params* p) {
    memset(p, 0, sizeof *p);
    p->MU = 0.012150585609624037; p->DU = 384747.96285603708; p->TU = 375699.81732246041;   // LowThrustOpt.jl:24-26
    p->Isp = 2000.0; p->g0 = 9.81; p->default_mass = 1000.0; p->tol = 1e-13;
    p->mode = LTO_FIXED; p->err_norm = LTO_NORM_STATE; p->max_attempts = 0; p->kernel = LTO_KERNEL_AUTO;
}
void lto_indirect_params_default(lto_indirect_params* p) {
    memset(p, 0, sizeof *p);
    p->MU = 0.012150585609624037; p->DU = 384747.96285603708; p->TU = 375699.81732246041;
    p->thrustLimit = 0.05; p->mass = 1000.0; p->time_direction = 1.0; p->p = 1.0; p->rho = 1.0;
    p->Isp = 2000.0; p->g0 = 9.81; p->reltol = 1e-13; p->abstol = 1e-13;                      // multiShoot_CRTBP_indirect.jl:79
    p->controller = LTO_CTRL_RMS; p->err_norm = LTO_NORM_STATE_SENS; p->max_attempts = 0; p->kernel = LTO_KERNEL_AUTO;
}

int lto_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int lto_init(int device, lto_handle** out) {
    LTO_NVTX();
    if (!out) return fail(nullptr, LTO_ERR_ARG, "lto_init: null handle pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(nullptr, LTO_ERR_NODEVICE, "lto_init: no CUDA device (%s); liblto_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    }
    if (device < 0 || device >= n) return fail(nullptr, LTO_ERR_ARG, "lto_init: device %d out of range [0,%d)", device, n);
    cudaDeviceProp prop;
    CK(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, LTO_ERR_NODEVICE, "lto_init: device %d is sm_%d%d; this library carries sm_100a code only", device,
                    prop.major, prop.minor);
    CK(nullptr, cudaSetDevice(device));
    lto_handle* h = (lto_handle*)calloc(1, sizeof(lto_handle));
    if (!h) return fail(nullptr, LTO_ERR_NOMEM, "lto_init: out of host memory");
    h->device = device; h->n_sm = prop.multiProcessorCount;
    auto setup = [&]() -> int {
        CK(h, cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
        CK(h, cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
        CK(h, cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
        CK(h, cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
        CK(h, cudaEventCreate(&h->ev_t0));
        CK(h, cudaEventCreate(&h->ev_t1));
        for (int i = 0; i < 8; ++i) CK(h, cudaEventCreateWithFlags(&h->ev_chunk[i], cudaEventDisableTiming));
        for (int i = 0; i < 8; ++i) CK(h, cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
        CK(h, cudaMalloc((void**)&h->d_ctr, 256));                         // work-queue counter of the throughput kernels
        if (getenv("LTO_ICW_PROF")) { CK(h, cudaMalloc((void**)&h->d_prof, LTO_PROF_WORDS * 8)); CK(h, cudaMemset(h->d_prof, 0, LTO_PROF_WORDS * 8)); }
        return LTO_SUCCESS;
    };
    const int rc = setup();
    if (rc) {                                                              // no handle leaves this function: the message moves to the global slot
        char msg[sizeof h->err];
        memcpy(msg, h->err, sizeof msg); msg[sizeof msg - 1] = 0;
        lto_destroy(h);
        cudaGetLastError();
        return fail(nullptr, rc, "lto_init: %s", msg);
    }
    *out = h;
    return LTO_SUCCESS;
}

int lto_init_devices(int n_devices, const int* devices, lto_handle** out) {
    LTO_NVTX();
    if (!out) return fail(nullptr, LTO_ERR_ARG, "lto_init_devices: null handle pointer");
    *out = nullptr;
    if (n_devices < 1 || n_devices > LTO_MAX_DEVICES || !devices)
        return fail(nullptr, LTO_ERR_ARG, "lto_init_devices: n_devices must be 1..%d", LTO_MAX_DEVICES);
    if (n_devices == 1) return lto_init(devices[0], out);
    for (int i = 0; i < n_devices; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return fail(nullptr, LTO_ERR_ARG, "lto_init_devices: device %d listed twice", devices[i]);
    lto_handle* h = (lto_handle*)calloc(1, sizeof(lto_handle));
    if (!h) return fail(nullptr, LTO_ERR_NOMEM, "lto_init_devices: out of host memory");
    h->device = -1;
    for (int i = 0; i < n_devices; ++i) {
        int rc = lto_init(devices[i], &h->child[i]);
        if (rc) { for (int j = 0; j < i; ++j) lto_destroy(h->child[j]); free(h); return rc; }
        h->n_child = i + 1;
    }
    h->n_sm = h->child[0]->n_sm;
    *out = h;
    return LTO_SUCCESS;
}

void lto_destroy(lto_handle* h) {
    if (!h) return;
    if (h->n_child > 0) { for (int i = 0; i < h->n_child; ++i) lto_destroy(h->child[i]); free(h); return; }
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->s_compute); cudaStreamSynchronize(h->s_copy); cudaStreamSynchronize(h->s_h2d);
    if (h->d_in) cudaFree(h->d_in);
    if (h->d_out) cudaFree(h->d_out);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->d_ctr) cudaFree(h->d_ctr);
    if (h->d_scr) cudaFree(h->d_scr);
    if (h->d_prof) cudaFree(h->d_prof);
    if (h->d_nwt) cudaFree(h->d_nwt);
    if (h->d_slv) cudaFree(h->d_slv);
    for (int i = 0; i < 8; ++i) { cudaEventDestroy(h->ev_chunk[i]); cudaEventDestroy(h->ev_h2d[i]); }
    cudaEventDestroy(h->ev_in); cudaEventDestroy(h->ev_t0); cudaEventDestroy(h->ev_t1);
    cudaStreamDestroy(h->s_compute); cudaStreamDestroy(h->s_copy); cudaStreamDestroy(h->s_h2d);
    free(h);
}

const char* lto_last_error(const lto_handle* h) { return h ? h->err : g_err; }

void* lto_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void lto_host_free(void* p) { if (p) cudaFreeHost(p); }
int64_t lto_kernel_launches(const lto_handle* h) {
    if (!h) return 0;
    int64_t n = h->launches;
    for (int i = 0; i < h->n_child; ++i) n += h->child[i]->launches;
    return n;
}
double lto_last_kernel_ms(const lto_handle* h) {
    if (!h) return 0.0;
    double ms = h->last_ms;
    for (int i = 0; i < h->n_child; ++i) ms = std::max(ms, h->child[i]->last_ms);
    return ms;
}
int lto_n_devices(const lto_handle* h) { return h ? (h->n_child > 0 ? h->n_child : 1) : 0; }
void* lto_stream(lto_handle* h) { return (h && h->n_child == 0) ? (void*)h->s_compute : nullptr; }
int lto_sync(lto_handle* h) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    for (int i = 0; i < h->n_child; ++i) { int rc = lto_sync(h->child[i]); if (rc) return fail(h, rc, "%s", h->child[i]->err); }
    if (h->n_child > 0) return LTO_SUCCESS;
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaStreamSynchronize(h->s_compute));
    return LTO_SUCCESS;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// parameter translation
// ---------------------------------------------------------------------------
static int make_direct(lto_handle* h, const lto_direct_params* p, int nstate, int nsteps, DirectArgs* a) {
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (nstate != 6 && nstate != 7) return fail(h, LTO_ERR_ARG, "nstate must be 6 or 7 (got %d)", nstate);
    if (p->mode != LTO_FIXED && p->mode != LTO_ADAPTIVE) return fail(h, LTO_ERR_ARG, "bad mode %d", p->mode);
    if (p->mode == LTO_FIXED && nsteps < 2) return fail(h, LTO_ERR_ARG, "nsteps must be >= 2 (got %d)", nsteps);
    const double g0 = p->g0 > 0 ? p->g0 : 9.81;
    a->c.mu = p->MU; a->c.m1 = 1.0 - p->MU;
    a->c.kthr = p->TU * p->TU / p->DU / 1e3;
    a->c.cmdot = p->TU / (p->Isp * g0);
    a->c.default_mass = p->default_mass > 0 ? p->default_mass : 1000.0;
    a->cfg.mode = p->mode; a->cfg.nsteps = nsteps; a->cfg.tol = p->tol > 0 ? p->tol : 1e-13;
    a->cfg.err_norm = p->err_norm; a->cfg.max_attempts = p->max_attempts > 0 ? p->max_attempts : 100000;
    return 0;
}
static int make_indirect(lto_handle* h, const lto_indirect_params* p, int ndim, bool sens, IndirectArgs* a) {
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (ndim != 12 && ndim != 14) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
    if (!(p->p == 0.0 || p->p >= 1.0)) return fail(h, LTO_ERR_ARG, "Invalid value of p!");   // CRTBP_stateCostate_deriv.jl:52
    const double g0 = p->g0 > 0 ? p->g0 : 9.81;
    a->c.mu = p->MU; a->c.m1 = 1.0 - p->MU;
    a->c.kthr = p->TU * p->TU / p->DU / 1e3;
    a->c.thrustLimit = p->thrustLimit; a->c.mass = p->mass; a->c.omega = p->time_direction;
    a->c.p = p->p; a->c.rho = p->rho;
    a->c.cm = p->TU / (a->c.kthr * (p->Isp > 0 ? p->Isp : 2000.0) * g0);
    a->cfg.atol = p->abstol > 0 ? p->abstol : 1e-13; a->cfg.rtol = p->reltol > 0 ? p->reltol : 1e-13;
    a->cfg.controller = p->controller; a->cfg.err_norm = sens ? p->err_norm : 0;
    a->cfg.max_attempts = p->max_attempts > 0 ? p->max_attempts : 100000;
    return 0;
}

static int dispatch_direct(lto_handle* h, const DirectArgs& a, int nstate, int kernel) {
    int nl = 0;
    cudaError_t e = cudaErrorNotSupported;
    if (kernel != LTO_KERNEL_GENERIC) e = launch_direct_fast(a, nstate, h->s_compute, &nl);
    if (e == cudaErrorNotSupported) {
        if (kernel == LTO_KERNEL_FAST) return fail(h, LTO_ERR_ARG, "LTO_KERNEL_FAST does not cover this configuration");
        e = launch_direct_generic(a, nstate, h->s_compute, &nl);
    }
    h->launches += nl;
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "direct kernel launch: %s", cudaGetErrorString(e));
    return 0;
}
static int dispatch_indirect(lto_handle* h, const IndirectArgs& a, int ndim, int kernel, cudaStream_t st = nullptr) {
    int nl = 0;
    if (!st) st = h->s_compute;
    cudaError_t e = cudaErrorNotSupported;
    if (kernel != LTO_KERNEL_GENERIC) e = launch_indirect_fast(a, ndim, st, &nl);
    if (e == cudaErrorNotSupported) {
        if (kernel == LTO_KERNEL_FAST) return fail(h, LTO_ERR_ARG, "LTO_KERNEL_FAST does not cover this configuration");
        e = launch_indirect_generic(a, ndim, st, &nl);
    }
    h->launches += nl;
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "indirect kernel launch: %s", cudaGetErrorString(e));
    return 0;
}

// Chunk schedule (segments per launch) of the H2D -> kernel -> D2H pipeline of the host entry points.
// Cost model, measured on a B200 behind PCIe 5 x16 (DESIGN.md section 6): the device->host copy engine moves
// out_bytes_per_seg at ~50 GB/s (d ns per segment), a launch over c segments takes a_ns + c * r_ns (a_ns: launch + the
// tail of the adaptive kernels' work queue, 0.25 ms for K3), and the call ends when the last chunk's copy does.
//   * copy-bound with cheap launches (K1: r = 10 ns, d = 24 ns per segment): a geometric ramp. The first chunk is one
//     wave of the persistent grid, so the copy engine starts after ~60 us, and every later chunk is as large as it can be
//     while its kernel still finishes inside the previous chunk's copy -- the copy engine never waits again.
//   * otherwise (K3 / K3-14: r ~ d, expensive tail): k equal chunks, k = sqrt(n * d / a) minimises k * a + n * d / k
//     (the launch tails paid k times + the last chunk's exposed copy).
// `quantum` keeps chunks on wave / whole-trajectory boundaries.
static void plan_chunks(std::vector<long long>& plan, long long n_seg, size_t out_bytes_per_seg, double r_ns, double a_ns,
                        long long wave, long long unit) {
    plan.clear();
    if (n_seg <= 0) return;
    if (n_seg * (long long)out_bytes_per_seg <= (8ll << 20)) { plan.push_back(n_seg); return; }      // small: one shot
    const double d_ns = (double)out_bytes_per_seg / 50.0;
    auto up = [](long long x, long long q) { return (x + q - 1) / q * q; };
    const long long q_wave = up(std::max(wave, unit), unit);
    const double next_of_wave = ((double)q_wave * d_ns - a_ns) / r_ns;
    if (next_of_wave >= (double)q_wave) {
        // tk: when the kernels enqueued so far finish; tc: when the copies enqueued so far finish.  The next chunk is the largest
        // number of waves whose kernel ends before the copy engine runs dry (slack carries over from chunk to chunk).
        long long c = q_wave, left = n_seg;
        double tk = 0.0, tc = 0.0;
        while (left > 0) {
            const long long take = (left - c < q_wave) ? left : c;      // no sliver at the end
            plan.push_back(take); left -= take;
            tk += a_ns + (double)take * r_ns;
            tc = std::max(tc, tk) + (double)take * d_ns;
            c = std::max(q_wave, (long long)((tc - tk - a_ns) / r_ns) / q_wave * q_wave);
        }
        return;
    }
    long long k = (long long)std::llround(std::sqrt((double)n_seg * d_ns / std::max(a_ns, 1.0)));
    k = std::min<long long>(std::max<long long>(k, 1), 256);
    const long long q = up(std::max<long long>(2048, unit), unit);
    const long long c = up((n_seg + k - 1) / k, q);
    for (long long left = n_seg; left > 0; left -= std::min(c, left)) plan.push_back(std::min(c, left));
}

// Per-kernel constants of the model (B200, 1965 MHz).  Direct: K1 0.68 ms per 65,536 segments of 2 x 9 steps (one wave of
// n_sm x 32 segments: 49 us), K2 (ode78 controller) 0.50 ms + a tail of retried legs, K4 (defect only) 0.082 ms.
static void plan_direct(std::vector<long long>& plan, int n_sm, long long n_seg, int npt, int nstate, int nsteps, int mode, bool want_jac) {
    const size_t NS = (size_t)nstate, NV = 2 * (NS + 3);
    const size_t per_seg = NS * 8 + 8 + 4 + (want_jac ? NS * NV * 8 : 0);
    const bool fixed = mode == LTO_FIXED;
    const double r_ns = !want_jac ? 1.3 : fixed ? (nstate == 7 ? 10.4 : 11.0) * (double)std::max(nsteps - 1, 1) / 9.0 : 7.7;
    const double a_ns = (want_jac && !fixed) ? 60e3 : 10e3;
    plan_chunks(plan, n_seg, per_seg, r_ns, a_ns, (long long)n_sm * 32, npt > 0 ? npt - 1 : 1);
}
// Indirect: K3 17.5 ns per segment + 0.25 ms per launch (the work queue's tail: about one segment lifetime at 64 slots per SM),
// K3-14 26 ns + 0.33 ms, K4 (defect only) 2.5 ns + 50 us.
static void plan_indirect(std::vector<long long>& plan, int n_sm, long long n_seg, int npt, int ndim, bool want_jac) {
    const size_t ND = (size_t)ndim;
    const size_t per_seg = ND * 8 + 12 + (want_jac ? ND * ND * 8 : 0);
    const double r_ns = !want_jac ? 2.5 : ndim == 14 ? 26.0 : 17.5;
    const double a_ns = !want_jac ? 50e3 : ndim == 14 ? 330e3 : 250e3;
    plan_chunks(plan, n_seg, per_seg, r_ns, a_ns, (long long)n_sm * 64, npt > 0 ? npt - 1 : 1);
}

// ---------------------------------------------------------------------------
// Pageable caller memory (what a Julia / numpy caller holds; bench.py e2e.pageable, config 3).
//   * pageable RESULT arrays: 27 % of the all-pinned rate (the 78 MB of Jacobian blocks are staged by the driver, the copy/compute overlap is
//     gone).  What pays is pinned result arrays: lto_host_alloc; the Python and Julia bindings allocate theirs from a pool of such blocks
//     (capi.PinnedPool, julia/lto_b200.jl pinned_array; INTEGRATION.md).
//   * pageable INPUTS: a cudaMemcpyAsync from pageable memory blocks the enqueueing thread, so nothing of a chunk is enqueued before its inputs
//     have crossed -- with K1's ramped schedule (last chunk = half the batch) the call ended one half-batch kernel + copy after the last input
//     byte: 73 % of the all-pinned rate.  Direct calls therefore detect pageable inputs (cudaPointerGetAttributes), copy each chunk's rows into
//     a pinned block of the handle themselves (so every CUDA call stays asynchronous) and use a schedule of EQUAL two-wave chunks: the staging of
//     chunk k+1 overlaps the kernel and the copy-out of chunk k and only one small chunk is exposed at the end: 32.9 M segments/s = 84 % of
//     the all-pinned rate (nstate 6: 92 %); what is left is one core's memcpy of the 11.5 MB.  (Measured and not kept: the same staging with
//     the ramped schedule -- calling thread 26.3 M, worker threads 28.2 M: the schedule was the problem; two helper threads staging ahead of
//     the enqueueing thread with the equal schedule -- 29.3 M: thread start-up and hand-over cost more than they hide on these hosts.)
//     The indirect calls already run equal chunks and lose 4 % with pageable inputs.
static bool is_pageable(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}
static int ensure_host(lto_handle* h, void** p, size_t* cap, size_t need) {
    if (*cap >= need) return 0;
    if (*p) { cudaFreeHost(*p); *p = nullptr; *cap = 0; }
    const size_t want = need + need / 4;
    if (cudaHostAlloc(p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); *p = nullptr; return 1; }   // caller falls back to the driver's staging
    *cap = want;
    return 0;
}
// ---------------------------------------------------------------------------

// ---------------------------------------------------------------------------
// multi-device handles: contiguous, equal unit ranges (segments, or whole trajectories in the
// trajectory forms) per device, one host worker thread per device; every device copies its
// slab of the outputs straight into the caller's arrays, so no collective is needed.
// ---------------------------------------------------------------------------
template <class F>
static int run_children(lto_handle* h, long long n_units, F&& call) {
    const int nc = h->n_child;
    std::vector<int> rcs(nc, 0);
    std::vector<std::thread> th;
    for (int i = 0; i < nc; ++i) {
        const long long u0 = n_units * i / nc, u1 = n_units * (i + 1) / nc;
        if (u1 <= u0) continue;
        th.emplace_back([&, i, u0, u1] { rcs[i] = call(h->child[i], u0, u1 - u0); });
    }
    for (auto& t : th) t.join();
    for (int i = 0; i < nc; ++i)
        if (rcs[i]) return fail(h, rcs[i], "device %d: %s", h->child[i]->device, h->child[i]->err);
    return LTO_SUCCESS;
}

static int direct_host(lto_handle* h, const lto_direct_params* p, long long n_seg, int npt, long long n_nodes_total,
                       int nstate, int nsteps, const double* Xa, const double* Xb, const double* ua, const double* ub,
                       const double* ta, const double* tb, double* defect, double* errors, int32_t* status, double* jac,
                       bool want_jac);
static int direct_host_multi(lto_handle* h, const lto_direct_params* p, long long n_seg, int npt, int nstate, int nsteps,
                             const double* Xa, const double* Xb, const double* ua, const double* ub, const double* ta,
                             const double* tb, double* defect, double* errors, int32_t* status, double* jac, bool want_jac) {
    if (nstate != 6 && nstate != 7) return fail(h, LTO_ERR_ARG, "nstate must be 6 or 7 (got %d)", nstate);
    const long long spu = npt > 0 ? npt - 1 : 1, rpu = npt > 0 ? npt : 1;      // segments / input rows per unit
    const long long NS = nstate, NV = 2 * (NS + 3);
    return run_children(h, n_seg / spu, [&](lto_handle* c, long long u0, long long nu) {
        const long long r0 = u0 * rpu, s0 = u0 * spu;
        return direct_host(c, p, nu * spu, npt, nu * rpu, nstate, nsteps, Xa + r0 * NS, Xb ? Xb + r0 * NS : nullptr, ua + r0 * 3,
                           ub ? ub + r0 * 3 : nullptr, ta + r0, tb ? tb + r0 : nullptr, defect + s0 * NS, errors ? errors + s0 : nullptr,
                           status ? status + s0 : nullptr, jac ? jac + s0 * NS * NV : nullptr, want_jac);
    });
}

// ---------------------------------------------------------------------------
// host-buffer direct call
// ---------------------------------------------------------------------------
static int direct_host(lto_handle* h, const lto_direct_params* p, long long n_seg, int npt, long long n_nodes_total,
                       int nstate, int nsteps, const double* Xa, const double* Xb, const double* ua, const double* ub,
                       const double* ta, const double* tb, double* defect, double* errors, int32_t* status, double* jac,
                       bool want_jac) {
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (n_seg < 0) return fail(h, LTO_ERR_ARG, "negative segment count");
    if (h->n_child > 0) {
        if (n_seg > 0 && (!Xa || !ua || !ta || !defect || (npt == 0 && (!Xb || !ub || !tb)) || (want_jac && !jac)))
            return fail(h, LTO_ERR_ARG, "null array argument");
        return direct_host_multi(h, p, n_seg, npt, nstate, nsteps, Xa, Xb, ua, ub, ta, tb, defect, errors, status, jac, want_jac);
    }
    DirectArgs a; memset(&a, 0, sizeof a);
    int rc = make_direct(h, p, nstate, nsteps, &a);
    if (rc) return rc;
    if (n_seg == 0) return LTO_SUCCESS;
    if (!Xa || !ua || !ta || !defect || (npt == 0 && (!Xb || !ub || !tb)) || (want_jac && !jac))
        return fail(h, LTO_ERR_ARG, "null array argument");
    CK(h, cudaSetDevice(h->device));
    const int NS = nstate, NV = 2 * (NS + 3);
    const long long rows = npt > 0 ? n_nodes_total : n_seg;       // rows of each input array
    // ---- device input block
    const size_t bX = al(rows * NS * 8), bU = al(rows * 3 * 8), bT = al(rows * 8);
    const size_t in_bytes = (npt > 0 ? 1 : 2) * (bX + bU + bT);
    rc = ensure(h, &h->d_in, &h->d_in_cap, in_bytes); if (rc) return rc;
    char* di = (char*)h->d_in;
    double* dXa = (double*)di; di += bX; double* dua = (double*)di; di += bU; double* dta = (double*)di; di += bT;
    double *dXb, *dub, *dtb;
    if (npt > 0) { dXb = dXa + NS; dub = dua + 3; dtb = dta + 1; }
    else { dXb = (double*)di; di += bX; dub = (double*)di; di += bU; dtb = (double*)di; di += bT; }
    // ---- device output block
    const size_t bD = al(n_seg * NS * 8), bE = al(n_seg * 8), bS = al(n_seg * 4), bJ = want_jac ? al(n_seg * NS * NV * 8) : 0;
    rc = ensure(h, &h->d_out, &h->d_out_cap, bD + bE + bS + bJ); if (rc) return rc;
    char* dq = (char*)h->d_out;
    double* dD = (double*)dq; dq += bD; double* dE = (double*)dq; dq += bE; int32_t* dS = (int32_t*)dq; dq += bS;
    double* dJ = want_jac ? (double*)dq : nullptr;
    // ---- H2D goes chunk by chunk on its own stream (below): the first kernel starts after the first chunk's inputs have
    // arrived, and host->device and device->host transfers run on different copy engines
    CK(h, cudaEventRecord(h->ev_t0, h->s_compute));
    // ---- chunked compute + D2H pipeline
    std::vector<long long> plan;
    plan_direct(plan, h->n_sm, n_seg, npt, nstate, nsteps, p->mode, want_jac);
    // pageable inputs (see above): own pinned staging in CHUNK-major order (one host->device copy per chunk), equal two-wave chunks
    char* hs = nullptr;
    if (plan.size() > 1 && is_pageable(Xa) && ensure_host(h, &h->h_stage, &h->h_stage_cap, in_bytes) == 0) {
        hs = (char*)h->h_stage;
        const long long unit = npt > 0 ? npt - 1 : 1;
        const long long c = std::max<long long>(unit, (2ll * h->n_sm * 32 + unit - 1) / unit * unit);
        plan.clear();
        for (long long left = n_seg; left > 0;) { const long long take = (left < c + c / 2) ? left : c; plan.push_back(take); left -= take; }
    }
    static const bool tl = getenv("LTO_DEBUG_TIMELINE") != nullptr;
    cudaEvent_t tl_k[16], tl_c0[16], tl_c1[16];
    long long s0 = 0;
    size_t stage_off = 0;
    for (int ci = 0; ci < (int)plan.size(); s0 += plan[ci], ++ci) {
        const long long ns = plan[ci];
        const long long r0 = lto_node_a(s0, npt);
        // this chunk's input rows (trajectory form: whole trajectories, n_nodes rows each)
        const long long nr = npt > 0 ? ns / (npt - 1) * npt : ns;
        if (hs) {
            // [Xa | ua | ta ( | Xb | ub | tb )] of this chunk, contiguous in the pinned block and, at the same offset, in the device block
            char* st = hs + stage_off;
            double* dv = (double*)((char*)h->d_in + stage_off);
            size_t o = 0;
            auto add = [&](const double* src, size_t bytes) { memcpy(st + o, src, bytes); o += bytes; };
            add(Xa + r0 * NS, nr * NS * 8); add(ua + r0 * 3, nr * 3 * 8); add(ta + r0, nr * 8);
            a.Xa = dv; a.ua = a.Xa + nr * NS; a.ta = a.ua + nr * 3;
            if (npt == 0) {
                add(Xb + r0 * NS, nr * NS * 8); add(ub + r0 * 3, nr * 3 * 8); add(tb + r0, nr * 8);
                a.Xb = a.ta + nr; a.ub = a.Xb + nr * NS; a.tb = a.ub + nr * 3;
            } else { a.Xb = a.Xa + NS; a.ub = a.ua + 3; a.tb = a.ta + 1; }
            CK(h, cudaMemcpyAsync(dv, st, o, cudaMemcpyHostToDevice, h->s_h2d));
            stage_off += o;
        } else {
            CK(h, cudaMemcpyAsync(dXa + r0 * NS, Xa + r0 * NS, nr * NS * 8, cudaMemcpyHostToDevice, h->s_h2d));
            CK(h, cudaMemcpyAsync(dua + r0 * 3, ua + r0 * 3, nr * 3 * 8, cudaMemcpyHostToDevice, h->s_h2d));
            CK(h, cudaMemcpyAsync(dta + r0, ta + r0, nr * 8, cudaMemcpyHostToDevice, h->s_h2d));
            if (npt == 0) {
                CK(h, cudaMemcpyAsync(dXb + r0 * NS, Xb + r0 * NS, nr * NS * 8, cudaMemcpyHostToDevice, h->s_h2d));
                CK(h, cudaMemcpyAsync(dub + r0 * 3, ub + r0 * 3, nr * 3 * 8, cudaMemcpyHostToDevice, h->s_h2d));
                CK(h, cudaMemcpyAsync(dtb + r0, tb + r0, nr * 8, cudaMemcpyHostToDevice, h->s_h2d));
            }
            a.Xa = dXa + r0 * NS; a.Xb = dXb + r0 * NS; a.ua = dua + r0 * 3; a.ub = dub + r0 * 3; a.ta = dta + r0; a.tb = dtb + r0;
        }
        CK(h, cudaEventRecord(h->ev_h2d[ci & 7], h->s_h2d));
        CK(h, cudaStreamWaitEvent(h->s_compute, h->ev_h2d[ci & 7], 0));
        a.defect = dD + s0 * NS; a.errors = dE + s0; a.status = dS + s0; a.jac = want_jac ? dJ + s0 * NS * NV : nullptr;
        a.n_seg = ns; a.npt = npt;
        rc = dispatch_direct(h, a, nstate, p->kernel); if (rc) return rc;
        cudaEvent_t ev = h->ev_chunk[ci & 7];
        CK(h, cudaEventRecord(ev, h->s_compute));
        CK(h, cudaStreamWaitEvent(h->s_copy, ev, 0));
        if (tl && ci < 16) { cudaEventCreate(&tl_k[ci]); cudaEventRecord(tl_k[ci], h->s_compute); cudaEventCreate(&tl_c0[ci]); cudaEventRecord(tl_c0[ci], h->s_copy); }
        CK(h, cudaMemcpyAsync(defect + s0 * NS, dD + s0 * NS, ns * NS * 8, cudaMemcpyDeviceToHost, h->s_copy));
        if (errors) CK(h, cudaMemcpyAsync(errors + s0, dE + s0, ns * 8, cudaMemcpyDeviceToHost, h->s_copy));
        if (status) CK(h, cudaMemcpyAsync(status + s0, dS + s0, ns * 4, cudaMemcpyDeviceToHost, h->s_copy));
        if (want_jac) CK(h, cudaMemcpyAsync(jac + s0 * NS * NV, dJ + s0 * NS * NV, ns * NS * NV * 8, cudaMemcpyDeviceToHost, h->s_copy));
        if (tl && ci < 16) { cudaEventCreate(&tl_c1[ci]); cudaEventRecord(tl_c1[ci], h->s_copy); }
    }
    CK(h, cudaEventRecord(h->ev_t1, h->s_compute));
    CK(h, cudaStreamSynchronize(h->s_copy));
    CK(h, cudaStreamSynchronize(h->s_compute));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    if (tl) {   // LTO_DEBUG_TIMELINE=1: when each chunk's kernel ended and when its copy-out started / ended, ms after the call's first enqueue
        for (int ci = 0; ci < (int)plan.size() && ci < 16; ++ci) {
            float a0 = 0, a1 = 0, a2 = 0;
            cudaEventElapsedTime(&a0, h->ev_t0, tl_k[ci]); cudaEventElapsedTime(&a1, h->ev_t0, tl_c0[ci]); cudaEventElapsedTime(&a2, h->ev_t0, tl_c1[ci]);
            fprintf(stderr, "[lto timeline] chunk %d: %lld segments, kernel done %.3f, copy-out %.3f .. %.3f ms\n", ci, plan[ci], a0, a1, a2);
            cudaEventDestroy(tl_k[ci]); cudaEventDestroy(tl_c0[ci]); cudaEventDestroy(tl_c1[ci]);
        }
    }
    return LTO_SUCCESS;
}

// stream memory operations (driver API through the runtime's entry-point query): completion flags / counters on streams
typedef int (*lto_cu_stream_val_fn)(void* stream, unsigned long long addr, unsigned long long value, unsigned int flags);
static lto_cu_stream_val_fn g_cu_write64 = nullptr, g_cu_wait64 = nullptr;
static int resolve_stream_memops(lto_handle* h) {
    if (g_cu_write64 && g_cu_wait64) return 0;
    void* fw = nullptr; void* fq = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue64", &fw, cudaEnableDefault, &qr) != cudaSuccess || !fw ||
        cudaGetDriverEntryPoint("cuStreamWaitValue64", &fq, cudaEnableDefault, &qr) != cudaSuccess || !fq) {
        cudaGetLastError();
        return fail(h, LTO_ERR_CUDA, "stream memory operations (cuStreamWriteValue64 / cuStreamWaitValue64) are not available");
    }
    g_cu_write64 = (lto_cu_stream_val_fn)fw; g_cu_wait64 = (lto_cu_stream_val_fn)fq;
    return 0;
}
static int indirect_host(lto_handle* h, const lto_indirect_params* p, long long n_seg, int npt, long long n_nodes_total,
                         long long n_traj, int ndim, const double* x0, const double* t0, const double* t1,
                         const double* x_target, const double* tl_arr, const double* rho_arr, double* defect,
                         int32_t* status, int32_t* nsteps_out, double* phi, bool want_jac) {
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (n_seg < 0) return fail(h, LTO_ERR_ARG, "negative segment count");
    if (h->n_child > 0) {
        if (ndim != 12 && ndim != 14) return fail(h, LTO_ERR_ARG, "ndim must be 12 or 14 (got %d)", ndim);
        if (n_seg > 0 && (!x0 || !t0 || !defect || (npt == 0 && !t1) || (want_jac && !phi))) return fail(h, LTO_ERR_ARG, "null array argument");
        const long long spu = npt > 0 ? npt - 1 : 1, rpu = npt > 0 ? npt : 1, ND = ndim;
        return run_children(h, n_seg / spu, [&](lto_handle* c, long long u0, long long nu) {
            const long long r0 = u0 * rpu, s0 = u0 * spu;
            return indirect_host(c, p, nu * spu, npt, nu * rpu, nu, ndim, x0 + r0 * ND, t0 + r0, t1 ? t1 + r0 : nullptr,
                                 x_target ? x_target + r0 * ND : nullptr, tl_arr ? tl_arr + u0 : nullptr, rho_arr ? rho_arr + u0 : nullptr,
                                 defect + s0 * ND, status ? status + s0 : nullptr, nsteps_out ? nsteps_out + 2 * s0 : nullptr,
                                 phi ? phi + s0 * ND * ND : nullptr, want_jac);
        });
    }
    IndirectArgs a; memset(&a, 0, sizeof a);
    int rc = make_indirect(h, p, ndim, want_jac, &a);
    if (rc) return rc;
    if (n_seg == 0) return LTO_SUCCESS;
    if (!x0 || !t0 || !defect || (npt == 0 && !t1) || (want_jac && !phi)) return fail(h, LTO_ERR_ARG, "null array argument");
    // Reversed spans (t1 < t0): the reference's solve(ODEProblem(.., (t0, t1))) would integrate backwards; the kernels step forwards
    // only and would hand back x0 and Phi = I.  A wrong answer with status OK is worse than a refused call (ADVICE r1): reject.
    for (long long sgm = 0; sgm < n_seg; ++sgm) {
        const long long ia = lto_node_a(sgm, npt);
        const double ta = t0[ia], tb = npt > 0 ? t0[ia + 1] : t1[ia];
        if (tb < ta) return fail(h, LTO_ERR_ARG, "segment %lld has t1 < t0 (%.17g < %.17g): reversed spans are not supported", sgm, tb, ta);
    }
    CK(h, cudaSetDevice(h->device));
    const int ND = ndim;
    const long long rows = npt > 0 ? n_nodes_total : n_seg;
    const long long prow = npt > 0 ? n_traj : n_seg;              // rows of the per-segment/per-trajectory parameter arrays
    const bool sep_target = (npt == 0 && x_target != nullptr);
    const size_t bX = al(rows * ND * 8), bT = al(rows * 8), bP = al(prow * 8);
    const size_t in_bytes = bX + bT + (npt == 0 ? bT : 0) + (sep_target ? bX : 0) + (tl_arr ? bP : 0) + (rho_arr ? bP : 0);
    rc = ensure(h, &h->d_in, &h->d_in_cap, in_bytes); if (rc) return rc;
    char* di = (char*)h->d_in;
    double* dX = (double*)di; di += bX; double* dT0 = (double*)di; di += bT;
    double* dT1; if (npt > 0) dT1 = dT0 + 1; else { dT1 = (double*)di; di += bT; }
    double* dXT = nullptr; if (npt > 0) dXT = dX + ND; else if (sep_target) { dXT = (double*)di; di += bX; }
    double* dTL = nullptr; if (tl_arr) { dTL = (double*)di; di += bP; }
    double* dRH = nullptr; if (rho_arr) { dRH = (double*)di; di += bP; }
    const size_t bD = al(n_seg * ND * 8), bS = al(n_seg * 4), bN = al(n_seg * 8), bJ = want_jac ? al(n_seg * ND * ND * 8) : 0;
    rc = ensure(h, &h->d_out, &h->d_out_cap, bD + bS + bN + bJ); if (rc) return rc;
    char* dq = (char*)h->d_out;
    double* dD = (double*)dq; dq += bD; int32_t* dS = (int32_t*)dq; dq += bS; int32_t* dN = (int32_t*)dq; dq += bN;
    double* dJ = want_jac ? (double*)dq : nullptr;
    const size_t scr_bytes = want_jac ? al(indirect_cw_scratch_bytes(h->n_sm)) : 0;
    if (want_jac) { rc = ensure(h, &h->d_scr, &h->d_scr_cap, scr_bytes); if (rc) return rc; }
    // per-trajectory / per-segment parameter arrays are small: up front; the node data goes chunk by chunk (below)
    if (tl_arr) CK(h, cudaMemcpyAsync(dTL, tl_arr, prow * 8, cudaMemcpyHostToDevice, h->s_h2d));
    if (rho_arr) CK(h, cudaMemcpyAsync(dRH, rho_arr, prow * 8, cudaMemcpyHostToDevice, h->s_h2d));
    CK(h, cudaEventRecord(h->ev_t0, h->s_compute));
    std::vector<long long> plan;
    plan_indirect(plan, h->n_sm, n_seg, npt, ndim, want_jac);
    long long s0 = 0;
    for (int ci = 0; ci < (int)plan.size(); s0 += plan[ci], ++ci) {
        const long long ns = plan[ci];
        const long long r0 = lto_node_a(s0, npt);
        const long long p0 = lto_traj_of(s0, npt);
        const long long nr = npt > 0 ? ns / (npt - 1) * npt : ns;
        CK(h, cudaMemcpyAsync(dX + r0 * ND, x0 + r0 * ND, nr * ND * 8, cudaMemcpyHostToDevice, h->s_h2d));
        CK(h, cudaMemcpyAsync(dT0 + r0, t0 + r0, nr * 8, cudaMemcpyHostToDevice, h->s_h2d));
        if (npt == 0) CK(h, cudaMemcpyAsync(dT1 + r0, t1 + r0, nr * 8, cudaMemcpyHostToDevice, h->s_h2d));
        if (sep_target) CK(h, cudaMemcpyAsync(dXT + r0 * ND, x_target + r0 * ND, nr * ND * 8, cudaMemcpyHostToDevice, h->s_h2d));
        CK(h, cudaEventRecord(h->ev_h2d[ci & 7], h->s_h2d));
        CK(h, cudaStreamWaitEvent(h->s_compute, h->ev_h2d[ci & 7], 0));
        a.x0 = dX + r0 * ND; a.t0 = dT0 + r0; a.t1 = dT1 + r0; a.x_target = dXT ? dXT + r0 * ND : nullptr;
        a.thrustLimit_arr = dTL ? dTL + p0 : nullptr; a.rho_arr = dRH ? dRH + p0 : nullptr;
        a.defect = dD + s0 * ND; a.status = dS + s0; a.nsteps_out = dN + 2 * s0; a.phi = want_jac ? dJ + s0 * ND * ND : nullptr;
        a.n_seg = ns; a.npt = npt; a.counter = h->d_ctr; a.scratch = (double*)h->d_scr; a.prof = h->d_prof;
        rc = dispatch_indirect(h, a, ndim, p->kernel); if (rc) return rc;
        cudaEvent_t ev = h->ev_chunk[ci & 7];
        CK(h, cudaEventRecord(ev, h->s_compute));
        CK(h, cudaStreamWaitEvent(h->s_copy, ev, 0));
        CK(h, cudaMemcpyAsync(defect + s0 * ND, dD + s0 * ND, ns * ND * 8, cudaMemcpyDeviceToHost, h->s_copy));
        if (status) CK(h, cudaMemcpyAsync(status + s0, dS + s0, ns * 4, cudaMemcpyDeviceToHost, h->s_copy));
        if (nsteps_out) CK(h, cudaMemcpyAsync(nsteps_out + 2 * s0, dN + 2 * s0, ns * 8, cudaMemcpyDeviceToHost, h->s_copy));
        if (want_jac) CK(h, cudaMemcpyAsync(phi + s0 * ND * ND, dJ + s0 * ND * ND, ns * ND * ND * 8, cudaMemcpyDeviceToHost, h->s_copy));
    }
    CK(h, cudaEventRecord(h->ev_t1, h->s_compute));
    CK(h, cudaStreamSynchronize(h->s_copy));
    CK(h, cudaStreamSynchronize(h->s_compute));
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

extern "C" {

int lto_host_chunk_plan(int method, int n_sm, int64_t n_seg, int n_nodes, int nvar, int nsteps, int mode, int want_jac,
                        int64_t* chunks, int cap) {
    if (n_sm <= 0 || n_seg < 0 || n_nodes == 1 || n_nodes < 0 || cap < 0 || (cap > 0 && !chunks)) return LTO_ERR_ARG;
    if (n_nodes > 0 && n_seg % (n_nodes - 1) != 0) return LTO_ERR_ARG;
    std::vector<long long> plan;
    if (method == 0) {
        if (nvar != 6 && nvar != 7) return LTO_ERR_ARG;
        plan_direct(plan, n_sm, n_seg, n_nodes, nvar, nsteps, mode, want_jac != 0);
    } else if (method == 1) {
        if (nvar != 12 && nvar != 14) return LTO_ERR_ARG;
        plan_indirect(plan, n_sm, n_seg, n_nodes, nvar, want_jac != 0);
    } else return LTO_ERR_ARG;
    for (int i = 0; i < (int)plan.size() && i < cap; ++i) chunks[i] = plan[i];
    return (int)plan.size();
}

int lto_direct_defect(lto_handle* h, const lto_direct_params* p, int64_t n_seg, int nstate, int nsteps, const double* Xa,
                      const double* Xb, const double* ua, const double* ub, const double* ta, const double* tb,
                      double* defect, double* errors, int32_t* status) {
    LTO_NVTX();
    return direct_host(h, p, n_seg, 0, 0, nstate, nsteps, Xa, Xb, ua, ub, ta, tb, defect, errors, status, nullptr, false);
}
int lto_direct_defect_jac(lto_handle* h, const lto_direct_params* p, int64_t n_seg, int nstate, int nsteps,
                          const double* Xa, const double* Xb, const double* ua, const double* ub, const double* ta,
                          const double* tb, double* defect, double* errors, int32_t* status, double* jac) {
    LTO_NVTX();
    return direct_host(h, p, n_seg, 0, 0, nstate, nsteps, Xa, Xb, ua, ub, ta, tb, defect, errors, status, jac, true);
}
int lto_direct_defect_traj(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nstate, int nsteps,
                           const double* X_all, const double* u_all, const double* t_TU, double* defect, double* errors,
                           int32_t* status) {
    LTO_NVTX();
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    return direct_host(h, p, n_traj * (n_nodes - 1), n_nodes, n_traj * n_nodes, nstate, nsteps, X_all, nullptr, u_all, nullptr,
                       t_TU, nullptr, defect, errors, status, nullptr, false);
}
int lto_direct_defect_jac_traj(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nstate,
                               int nsteps, const double* X_all, const double* u_all, const double* t_TU, double* defect,
                               double* errors, int32_t* status, double* jac) {
    LTO_NVTX();
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    return direct_host(h, p, n_traj * (n_nodes - 1), n_nodes, n_traj * n_nodes, nstate, nsteps, X_all, nullptr, u_all, nullptr,
                       t_TU, nullptr, defect, errors, status, jac, true);
}

int lto_indirect_defect(lto_handle* h, const lto_indirect_params* p, int64_t n_seg, int ndim, const double* x0,
                        const double* t0, const double* t1, const double* x_target, const double* thrustLimit_seg,
                        const double* rho_seg, double* defect, int32_t* status, int32_t* nsteps_out) {
    LTO_NVTX();
    return indirect_host(h, p, n_seg, 0, 0, 0, ndim, x0, t0, t1, x_target, thrustLimit_seg, rho_seg, defect, status, nsteps_out,
                         nullptr, false);
}
int lto_indirect_defect_jac(lto_handle* h, const lto_indirect_params* p, int64_t n_seg, int ndim, const double* x0,
                            const double* t0, const double* t1, const double* x_target, const double* thrustLimit_seg,
                            const double* rho_seg, double* defect, int32_t* status, int32_t* nsteps_out, double* phi) {
    LTO_NVTX();
    return indirect_host(h, p, n_seg, 0, 0, 0, ndim, x0, t0, t1, x_target, thrustLimit_seg, rho_seg, defect, status, nsteps_out,
                         phi, true);
}
int lto_indirect_defect_traj(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, int ndim,
                             const double* XC_all, const double* t_TU, const double* thrustLimit_traj, const double* rho_traj,
                             double* defect, int32_t* status, int32_t* nsteps_out) {
    LTO_NVTX();
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    return indirect_host(h, p, n_traj * (n_nodes - 1), n_nodes, n_traj * n_nodes, n_traj, ndim, XC_all, t_TU, nullptr, nullptr,
                         thrustLimit_traj, rho_traj, defect, status, nsteps_out, nullptr, false);
}
int lto_indirect_defect_jac_traj(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, int ndim,
                                 const double* XC_all, const double* t_TU, const double* thrustLimit_traj,
                                 const double* rho_traj, double* defect, int32_t* status, int32_t* nsteps_out, double* phi) {
    LTO_NVTX();
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2");
    return indirect_host(h, p, n_traj * (n_nodes - 1), n_nodes, n_traj * n_nodes, n_traj, ndim, XC_all, t_TU, nullptr, nullptr,
                         thrustLimit_traj, rho_traj, defect, status, nsteps_out, phi, true);
}

int lto_direct_dev(lto_handle* h, const lto_direct_params* p, int64_t n_seg, int n_nodes, int nstate, int nsteps,
                   const double* Xa, const double* Xb, const double* ua, const double* ub, const double* ta, const double* tb,
                   double* defect, double* errors, int32_t* status, double* jac) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) return fail(h, LTO_ERR_ARG, "device-pointer entry points need a single-device handle (lto_init)");
    DirectArgs a; memset(&a, 0, sizeof a);
    int rc = make_direct(h, p, nstate, nsteps, &a); if (rc) return rc;
    if (n_seg <= 0) return n_seg == 0 ? LTO_SUCCESS : fail(h, LTO_ERR_ARG, "negative segment count");
    if (n_nodes == 1 || n_nodes < 0) return fail(h, LTO_ERR_ARG, "n_nodes must be 0 (pairs) or >= 2");
    if (!Xa || !ua || !ta || !defect || (n_nodes == 0 && (!Xb || !ub || !tb))) return fail(h, LTO_ERR_ARG, "null array argument");
    CK(h, cudaSetDevice(h->device));
    a.Xa = Xa; a.ua = ua; a.ta = ta;
    if (n_nodes > 0) { a.Xb = Xa + nstate; a.ub = ua + 3; a.tb = ta + 1; } else { a.Xb = Xb; a.ub = ub; a.tb = tb; }
    a.defect = defect; a.errors = errors; a.status = status; a.jac = jac; a.n_seg = n_seg; a.npt = n_nodes;
    return dispatch_direct(h, a, nstate, p->kernel);
}
int lto_indirect_dev(lto_handle* h, const lto_indirect_params* p, int64_t n_seg, int n_nodes, int ndim, const double* x0,
                     const double* t0, const double* t1, const double* x_target, const double* thrustLimit_arr,
                     const double* rho_arr, double* defect, int32_t* status, int32_t* nsteps_out, double* phi) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) return fail(h, LTO_ERR_ARG, "device-pointer entry points need a single-device handle (lto_init)");
    IndirectArgs a; memset(&a, 0, sizeof a);
    int rc = make_indirect(h, p, ndim, phi != nullptr, &a); if (rc) return rc;
    if (n_seg <= 0) return n_seg == 0 ? LTO_SUCCESS : fail(h, LTO_ERR_ARG, "negative segment count");
    if (n_nodes == 1 || n_nodes < 0) return fail(h, LTO_ERR_ARG, "n_nodes must be 0 (pairs) or >= 2");
    if (!x0 || !t0 || !defect || (n_nodes == 0 && !t1)) return fail(h, LTO_ERR_ARG, "null array argument");
    CK(h, cudaSetDevice(h->device));
    a.x0 = x0; a.t0 = t0;
    if (n_nodes > 0) { a.t1 = t0 + 1; a.x_target = x0 + ndim; } else { a.t1 = t1; a.x_target = x_target; }
    a.thrustLimit_arr = thrustLimit_arr; a.rho_arr = rho_arr;
    if (phi) { rc = ensure(h, &h->d_scr, &h->d_scr_cap, indirect_cw_scratch_bytes(h->n_sm)); if (rc) return rc; }
    a.defect = defect; a.status = status; a.nsteps_out = nsteps_out; a.phi = phi; a.n_seg = n_seg; a.npt = n_nodes; a.counter = h->d_ctr;
    a.scratch = (double*)h->d_scr; a.prof = h->d_prof;
    return dispatch_indirect(h, a, ndim, p->kernel);
}

int lto_indirect_cost_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, const double* XC_all,
                            const double* t_TU, const double* thrustLimit_traj, const double* rho_traj, double* dv, double* energy,
                            double* defect, int32_t* status) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (!p) return fail(h, LTO_ERR_ARG, "null params");
    if (n_traj < 0) return fail(h, LTO_ERR_ARG, "negative trajectory count");
    if (n_nodes < 2) return fail(h, LTO_ERR_ARG, "n_nodes must be >= 2 (got %d)", n_nodes);
    if (p->controller != LTO_CTRL_RMS)
        return fail(h, LTO_ERR_ARG, "the cost quadrature runs in the defect-only kernel K4: controller must be LTO_CTRL_RMS (got %d)", p->controller);
    if (p->kernel == LTO_KERNEL_GENERIC) return fail(h, LTO_ERR_ARG, "the generic kernel has no cost quadrature (kernel must be AUTO or FAST)");
    IndirectArgs a; memset(&a, 0, sizeof a);
    int rc = make_indirect(h, p, 12, false, &a); if (rc) return rc;
    if (n_traj == 0) return LTO_SUCCESS;
    if (!XC_all || !t_TU || !dv || !energy) return fail(h, LTO_ERR_ARG, "null array argument");
    const long long T = n_traj, N = n_nodes, n_seg = T * (N - 1);
    if (n_seg > 0x7fffffffll) return fail(h, LTO_ERR_ARG, "too many segments (%lld)", n_seg);
    for (long long j = 0; j < T; ++j) {
        const double* t = t_TU + j * N;
        for (int i = 0; i < N; ++i) {
            if (!std::isfinite(t[i])) return fail(h, LTO_ERR_ARG, "trajectory %lld: t_TU[%d] is not finite", j, i);
            if (i > 0 && t[i] < t[i - 1])
                return fail(h, LTO_ERR_ARG, "trajectory %lld: t_TU[%d] < t_TU[%d] (%.17g < %.17g): reversed spans are not supported", j, i, i - 1,
                            t[i], t[i - 1]);
        }
    }
    if (h->n_child > 0) {
        return split_trajectories(h, T, [&](lto_handle* c, long long u0, long long nu) {
            return lto_indirect_cost_batch(c, p, nu, n_nodes, XC_all + u0 * N * 12, t_TU + u0 * N, thrustLimit_traj ? thrustLimit_traj + u0 : nullptr,
                                           rho_traj ? rho_traj + u0 : nullptr, dv + u0, energy + u0, defect ? defect + u0 * (N - 1) * 12 : nullptr,
                                           status ? status + u0 : nullptr);
        });
    }
    CK(h, cudaSetDevice(h->device));
    cudaStream_t st = h->s_compute;
    // inputs: one staged copy
    const size_t bX = al(T * N * 12 * 8), bT = al(T * N * 8), bP = al(T * 8);
    const size_t in_bytes = bX + bT + (thrustLimit_traj ? bP : 0) + (rho_traj ? bP : 0);
    std::vector<char> stage(in_bytes);
    {
        char* q = stage.data();
        memcpy(q, XC_all, T * N * 12 * 8); q += bX;
        memcpy(q, t_TU, T * N * 8); q += bT;
        if (thrustLimit_traj) { memcpy(q, thrustLimit_traj, T * 8); q += bP; }
        if (rho_traj) memcpy(q, rho_traj, T * 8);
    }
    rc = ensure(h, &h->d_in, &h->d_in_cap, in_bytes); if (rc) return rc;
    const size_t bD = al(n_seg * 12 * 8), bS = al(n_seg * 4), bQ = al(n_seg * 2 * 8), bV = al(T * 8), bST = al(T * 4);
    rc = ensure(h, &h->d_out, &h->d_out_cap, bD + bS + bQ + 2 * bV + bST); if (rc) return rc;
    char* di = (char*)h->d_in;
    double* dX = (double*)di; di += bX;
    double* dT = (double*)di; di += bT;
    double* dTL = nullptr; if (thrustLimit_traj) { dTL = (double*)di; di += bP; }
    double* dRH = nullptr; if (rho_traj) dRH = (double*)di;
    char* dq = (char*)h->d_out;
    double* dD = (double*)dq; dq += bD; int32_t* dS = (int32_t*)dq; dq += bS; double* dQ = (double*)dq; dq += bQ;
    double* dDV = (double*)dq; dq += bV; double* dE = (double*)dq; dq += bV; int32_t* dST = (int32_t*)dq;
    CK(h, cudaMemcpyAsync(h->d_in, stage.data(), in_bytes, cudaMemcpyHostToDevice, st));
    a.x0 = dX; a.t0 = dT; a.t1 = dT + 1; a.x_target = dX + 12; a.thrustLimit_arr = dTL; a.rho_arr = dRH;
    a.defect = dD; a.status = dS; a.quad = dQ; a.n_seg = n_seg; a.npt = n_nodes; a.counter = h->d_ctr;
    // dv in m/s: int umag dt * DU 1e3 / TU;  energy in N^2 TU: int (umag * mass * DU 1e3 / TU^2)^2 dt (solvers._quad_cost's units)
    const double dv_scale = p->DU * 1e3 / p->TU, f_scale = p->mass * p->DU * 1e3 / (p->TU * p->TU);
    CK(h, cudaEventRecord(h->ev_t0, st));
    int nl = 0;
    const cudaError_t e = launch_indirect_cost(a, T, dv_scale, f_scale * f_scale, dDV, dE, dST, st, &nl);
    h->launches += nl;
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "indirect cost launch: %s", cudaGetErrorString(e));
    CK(h, cudaEventRecord(h->ev_t1, st));
    CK(h, cudaMemcpyAsync(dv, dDV, T * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(energy, dE, T * 8, cudaMemcpyDeviceToHost, st));
    if (status) CK(h, cudaMemcpyAsync(status, dST, T * 4, cudaMemcpyDeviceToHost, st));
    if (defect) CK(h, cudaMemcpyAsync(defect, dD, n_seg * 12 * 8, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));                                     // (also keeps `stage` alive until its copy is done)
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1)); h->last_ms = ms;
    return LTO_SUCCESS;
}

int lto_sumsq_dev(lto_handle* h, const double* v, int64_t n_rows, int64_t row_len, double* out) {
    LTO_NVTX();
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) return fail(h, LTO_ERR_ARG, "device-pointer entry points need a single-device handle (lto_init)");
    if (n_rows < 0 || row_len < 0 || (n_rows > 0 && (!v || !out))) return fail(h, LTO_ERR_ARG, "bad argument");
    CK(h, cudaSetDevice(h->device));
    cudaError_t e = launch_sumsq_rows(v, n_rows, row_len, out, h->s_compute);
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "sumsq launch: %s", cudaGetErrorString(e));
    if (n_rows > 0) h->launches += 1;
    return LTO_SUCCESS;
}

// ---- peer memory (multi-process multi-GPU: outputs written straight into the solver rank's HBM over NVLink) ----
void* lto_dev_alloc(lto_handle* h, size_t bytes) {
    if (!h || h->n_child > 0) return nullptr;
    if (cudaSetDevice(h->device) != cudaSuccess) return nullptr;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 256) != cudaSuccess) { cudaGetLastError(); fail(h, LTO_ERR_NOMEM, "cudaMalloc(%zu) failed", bytes); return nullptr; }
    return p;
}
void lto_dev_free(lto_handle* h, void* p) {
    if (!h || !p) return;
    cudaSetDevice(h->device);
    cudaFree(p);
}
int lto_ipc_export(lto_handle* h, void* dev_ptr, void* handle64) {
    if (!h || !dev_ptr || !handle64) return fail(h, LTO_ERR_ARG, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CK(h, cudaSetDevice(h->device));
    cudaIpcMemHandle_t mh;
    CK(h, cudaIpcGetMemHandle(&mh, dev_ptr));
    memcpy(handle64, &mh, 64);
    return LTO_SUCCESS;
}
int lto_ipc_open(lto_handle* h, const void* handle64, void** dev_ptr) {
    if (!h || !handle64 || !dev_ptr) return fail(h, LTO_ERR_ARG, "null argument");
    CK(h, cudaSetDevice(h->device));
    cudaIpcMemHandle_t mh;
    memcpy(&mh, handle64, 64);
    CK(h, cudaIpcOpenMemHandle(dev_ptr, mh, cudaIpcMemLazyEnablePeerAccess));
    return LTO_SUCCESS;
}
int lto_ipc_close(lto_handle* h, void* dev_ptr) {
    if (!h || !dev_ptr) return fail(h, LTO_ERR_ARG, "null argument");
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaIpcCloseMemHandle(dev_ptr));
    return LTO_SUCCESS;
}
// dst/src: device pointers (local or peer-mapped).  Enqueued on the copy stream after everything enqueued so far on the
// compute stream, i.e. a DMA-engine push that overlaps the next kernel.  lto_sync_copies waits for all of them.
int lto_push_async(lto_handle* h, void* dst, const void* src, size_t bytes) {
    LTO_NVTX();
    if (!h || h->n_child > 0) return fail(h, LTO_ERR_ARG, "needs a single-device handle");
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaEventRecord(h->ev_in, h->s_compute));
    CK(h, cudaStreamWaitEvent(h->s_copy, h->ev_in, 0));
    if (bytes) CK(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, h->s_copy));
    return LTO_SUCCESS;
}
int lto_sync_copies(lto_handle* h) {
    LTO_NVTX();
    if (!h || h->n_child > 0) return fail(h, LTO_ERR_ARG, "needs a single-device handle");
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaStreamSynchronize(h->s_copy));
    return LTO_SUCCESS;
}

// Stream-ordered 64-bit flags (driver stream memory operations, resolved at run time so that the library does not
// link libcuda): "my slab is written" signals from every rank into the solver rank's memory, awaited on its stream.
int lto_signal_dev(lto_handle* h, void* flag, uint64_t value) {
    if (!h || h->n_child > 0 || !flag) return fail(h, LTO_ERR_ARG, "needs a single-device handle and a flag address");
    CK(h, cudaSetDevice(h->device));
    int rc = resolve_stream_memops(h); if (rc) return rc;
    int e = g_cu_write64((void*)h->s_compute, (unsigned long long)(uintptr_t)flag, (unsigned long long)value, 0u /* CU_STREAM_WRITE_VALUE_DEFAULT */);
    if (e != 0) return fail(h, LTO_ERR_CUDA, "cuStreamWriteValue64 -> CUresult %d", e);
    return LTO_SUCCESS;
}
int lto_wait_dev(lto_handle* h, void* flag, uint64_t value) {
    if (!h || h->n_child > 0 || !flag) return fail(h, LTO_ERR_ARG, "needs a single-device handle and a flag address");
    CK(h, cudaSetDevice(h->device));
    int rc = resolve_stream_memops(h); if (rc) return rc;
    int e = g_cu_wait64((void*)h->s_compute, (unsigned long long)(uintptr_t)flag, (unsigned long long)value, 0u /* CU_STREAM_WAIT_VALUE_GEQ */);
    if (e != 0) return fail(h, LTO_ERR_CUDA, "cuStreamWaitValue64 -> CUresult %d", e);
    return LTO_SUCCESS;
}

int lto_debug_profile(lto_handle* h, unsigned long long* out, int n_words) {
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) h = h->child[0];
    if (!h->d_prof) return fail(h, LTO_ERR_ARG, "profiling counters are off (set LTO_ICW_PROF=1 before lto_init)");
    CK(h, cudaSetDevice(h->device));
    CK(h, cudaStreamSynchronize(h->s_compute));
    CK(h, cudaMemcpy(out, h->d_prof, std::min<size_t>((size_t)n_words, LTO_PROF_WORDS) * 8, cudaMemcpyDeviceToHost));
    return LTO_SUCCESS;
}

int lto_fp64_peak_probe(lto_handle* h, int iters, double* flops_per_s, double* ms_out) {
    if (!h) return fail(nullptr, LTO_ERR_ARG, "null handle");
    if (h->n_child > 0) h = h->child[0];
    CK(h, cudaSetDevice(h->device));
    int rc = ensure(h, &h->d_out, &h->d_out_cap, 4096); if (rc) return rc;
    long long nthreads = 0; int fmas = 0;
    cudaError_t e = launch_fp64_probe(16, (double*)h->d_out, h->n_sm, h->s_compute, &nthreads, &fmas);   // warm-up
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "probe launch: %s", cudaGetErrorString(e));
    CK(h, cudaEventRecord(h->ev_t0, h->s_compute));
    e = launch_fp64_probe(iters, (double*)h->d_out, h->n_sm, h->s_compute, &nthreads, &fmas);
    if (e != cudaSuccess) return fail(h, LTO_ERR_CUDA, "probe launch: %s", cudaGetErrorString(e));
    CK(h, cudaEventRecord(h->ev_t1, h->s_compute));
    CK(h, cudaStreamSynchronize(h->s_compute));
    h->launches += 2;
    float ms = 0.f; CK(h, cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1));
    if (ms_out) *ms_out = ms;
    if (flops_per_s) *flops_per_s = 2.0 * (double)nthreads * (double)iters * (double)fmas / ((double)ms * 1e-3);
    return LTO_SUCCESS;
}

}  // extern "C"
